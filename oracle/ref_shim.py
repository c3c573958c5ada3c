"""Legacy-API shim that lets the UNMODIFIED reference (the `ziggy` package of suyashk12/hipgp, pinned to
torch 1.4) import and run on torch >= 2.x.  TEST INFRASTRUCTURE ONLY.

Used by `tests/golden/make_golden.py` (to generate the committed golden vectors, in the build container), by
`tests/test_oracle_vs_reference.py` / `tests/test_gpu_dropin.py` and by `bench.py --impl reference`.  The reference is
taken from the reference checkout (oracle/make_ref.py: $HIPGP_REFERENCE_ROOT, else BASELINE.json's reference_path) when
that exists and otherwise from the staged, git-ignored, byte-identical copy `oracle/_ref/` written by `oracle/make_ref.py`; tests skip when neither is
there.  Nothing in `hipgp_b200/` may import this module.

What it patches (all removed from torch after 1.7):
  * `torch.fft(x, signal_ndim)` / `torch.ifft(x, signal_ndim)` -- function form, complex numbers as
    a trailing real dimension of size 2 (reference call sites: ziggy/misc/toeplitz_tensor.py:25,79,82;
    ziggy/misc/toeplitz_expanded.py:96,170,184; ziggy/misc/gpt_fft.py:8,12)
  * `Tensor.fft`, `Tensor.ifft`
  * `torch.solve(B, A)` (ziggy/hipgp.py:332)
  * module `pyprind` (ziggy/kernels.py:247) -- progress bar only
"""
import sys
import types

import torch
import torch.fft as _tfft

import os as _os

_STAGED = _os.path.join(_os.path.dirname(_os.path.abspath(__file__)), "_ref")


def reference_root():
    """Directory that holds the unmodified `ziggy` package: the reference checkout, else the staged copy oracle/_ref, else None."""
    from . import make_ref
    for root in (make_ref.SRC, _STAGED):
        if root and _os.path.isdir(_os.path.join(root, "ziggy")):
            return root
    return None


class _CallableFFTModule(types.ModuleType):
    """`torch.fft` stays a module (torch.fft.fftn still works) but is also callable like torch<=1.7."""

    def __init__(self, mod, inverse):
        super().__init__(mod.__name__)
        self.__dict__.update(mod.__dict__)
        self._inverse = inverse

    def __call__(self, x, signal_ndim, normalized=False):
        return _legacy_fft(x, signal_ndim, normalized, self._inverse)


def _legacy_fft(x, signal_ndim, normalized=False, inverse=False):
    assert x.shape[-1] == 2, "legacy complex layout: trailing dim of size 2"
    xc = torch.view_as_complex(x.contiguous())
    dims = tuple(range(xc.dim() - signal_ndim, xc.dim()))
    norm = "ortho" if normalized else "backward"
    yc = _tfft.ifftn(xc, dim=dims, norm=norm) if inverse else _tfft.fftn(xc, dim=dims, norm=norm)
    return torch.view_as_real(yc)


def install():
    if getattr(torch, "_hipgp_legacy_shim", False):
        return
    if "pyprind" not in sys.modules:
        m = types.ModuleType("pyprind")
        m.prog_bar = lambda it, *a, **k: it
        sys.modules["pyprind"] = m
    torch.fft = _CallableFFTModule(_tfft, inverse=False)
    sys.modules["torch.fft"] = torch.fft
    torch.ifft = lambda x, signal_ndim, normalized=False: _legacy_fft(x, signal_ndim, normalized, True)
    torch.Tensor.fft = lambda self, signal_ndim, normalized=False: _legacy_fft(self, signal_ndim, normalized, False)
    torch.Tensor.ifft = lambda self, signal_ndim, normalized=False: _legacy_fft(self, signal_ndim, normalized, True)
    torch.solve = lambda B, A: (torch.linalg.solve(A, B), None)
    torch._hipgp_legacy_shim = True


def import_reference():
    """Returns the unmodified reference package `ziggy` (raises if no reference tree is found)."""
    root = reference_root()
    if root is None:
        raise ImportError("reference tree not present (neither the reference checkout nor oracle/_ref; run oracle/make_ref.py)")
    install()
    if root not in sys.path:
        sys.path.insert(0, root)
    import ziggy  # noqa: F401
    return ziggy
