"""Stage the UNMODIFIED reference package into the git-ignored `oracle/_ref/` so that it travels to the GPU box.
TEST / BASELINE INFRASTRUCTURE ONLY -- nothing under `hipgp_b200/` may import it.

    python oracle/make_ref.py            # copies <root>/ziggy and run_solve_kn_experiment.py, byte for byte

<root> is the reference checkout: $HIPGP_REFERENCE_ROOT when set, else the `reference_path` that BASELINE.json records.

The reference is not part of this repository.  A copy of the working tree that includes git-ignored paths (like the
built `.so`) carries the staged copy along, so `oracle/_ref/ziggy` is what

  * `tests/test_gpu_dropin.py` imports after `hipgp_b200.install_as_ziggy()`: the reference's OWN model classes
    (`ziggy.hipgp.MeanFieldToeplitzGP`, `BlockToeplitzGP`) and `toeplitz_expanded.gram_solve` callers then run on top of the
    CUDA drop-ins and are compared with the golden vectors;
  * `bench.py --impl reference` times on the box's host cores (the reference's own CPU path under `oracle/ref_shim.py`,
    `cpu_baseline.kind = "reference"`).

Nothing is edited: every staged file is compared with its source by SHA-256 and the digests are written to
`oracle/_ref/MANIFEST.json`.  `oracle/_ref/` is listed in `.gitignore`: reference sources never enter the history.
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def reference_source():
    """The reference checkout: $HIPGP_REFERENCE_ROOT, else BASELINE.json's reference_path (None if neither is given)."""
    if os.environ.get("HIPGP_REFERENCE_ROOT"):
        return os.environ["HIPGP_REFERENCE_ROOT"]
    try:
        with open(os.path.join(HERE, "..", "BASELINE.json")) as f:
            return json.load(f).get("reference_path")
    except (OSError, ValueError):
        return None


SRC = reference_source()
DST = os.path.join(HERE, "_ref")
FILES_EXTRA = ["experiments-hip-gp/run_solve_kn_experiment.py"]


def _sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        h.update(f.read())
    return h.hexdigest()


def stage(verbose=True):
    """Returns the staged root, or None when the reference tree is not available."""
    if not SRC or not os.path.isdir(os.path.join(SRC, "ziggy")):
        return DST if os.path.isdir(os.path.join(DST, "ziggy")) else None
    manifest = {}
    pairs = []
    for root, _dirs, files in os.walk(os.path.join(SRC, "ziggy")):
        for f in files:
            if f.endswith(".py"):
                p = os.path.join(root, f)
                pairs.append((p, os.path.join(DST, os.path.relpath(p, SRC))))
    for rel in FILES_EXTRA:
        pairs.append((os.path.join(SRC, rel), os.path.join(DST, rel)))
    for src, dst in pairs:
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        if not os.path.exists(dst) or _sha(dst) != _sha(src):
            shutil.copyfile(src, dst)
        assert _sha(dst) == _sha(src), dst
        manifest[os.path.relpath(dst, DST)] = _sha(dst)
    with open(os.path.join(DST, "MANIFEST.json"), "w") as f:
        json.dump({"source": SRC, "files": manifest}, f, indent=1, sort_keys=True)
    if verbose:
        print("staged %d reference files into %s" % (len(manifest), DST))
    return DST


def verify():
    """Every staged file still has the digest recorded when it was copied (nothing edited in place)."""
    with open(os.path.join(DST, "MANIFEST.json")) as f:
        man = json.load(f)["files"]
    bad = [rel for rel, h in man.items() if _sha(os.path.join(DST, rel)) != h]
    return bad


if __name__ == "__main__":
    root = stage()
    if root is None:
        print("reference tree not found at %r (HIPGP_REFERENCE_ROOT or BASELINE.json reference_path)" % SRC)
        sys.exit(1)
    assert not verify()
