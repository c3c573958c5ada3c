// fast_inst.cu -- explicit instantiation of the specialised kernel launchers for one (length group, dtype) pair of
// HIPGP_FAST_LIST.  Compiled 10 times (-DHIPGP_INST_GROUP=0..9: group g/2, float for even g, double for odd g) so the
// build parallelises; without the macro it instantiates everything (single-command builds, e.g. the CPU emulation).
#include "fast_launch.cuh"
namespace hipgp {
#define INST(T, LEN)                                                                                            \
    template void launch_rows_fast_len<T, LEN>(hipgp_plan*, bool, RowsParams<T>&, cudaStream_t);                \
    template void launch_cols_fast_len<T, LEN>(hipgp_plan*, ColsParams<T>&, long, long, cudaStream_t);            \
    template bool rows_fast_fits_len<T, LEN>(long);
#ifndef HIPGP_INST_GROUP
#define X(LEN, ...) INST(float, LEN) INST(double, LEN)
HIPGP_FAST_LIST(X)
#undef X
#else
#if HIPGP_INST_GROUP % 2 == 0
#define X(LEN, ...) INST(float, LEN)
#else
#define X(LEN, ...) INST(double, LEN)
#endif
#if HIPGP_INST_GROUP / 2 == 0
HIPGP_FAST_LIST_G0(X)
#elif HIPGP_INST_GROUP / 2 == 1
HIPGP_FAST_LIST_G1(X)
#elif HIPGP_INST_GROUP / 2 == 2
HIPGP_FAST_LIST_G2(X)
#elif HIPGP_INST_GROUP / 2 == 3
HIPGP_FAST_LIST_G3(X)
#else
HIPGP_FAST_LIST_G4(X)
#endif
#undef X
#endif
}  // namespace hipgp
