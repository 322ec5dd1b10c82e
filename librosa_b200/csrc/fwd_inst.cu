// fwd_inst.cu — instantiates fwd_kernel for one transform size (compile with -DB2L_LOG2M=k).
#include "fwd_kernel.cuh"
#include "internal.h"

#ifndef B2L_LOG2M
#error "compile with -DB2L_LOG2M=<2..11>"
#endif

namespace b2l {
namespace {

template <class K>
cudaError_t run_op(K kern, int op, int nt, const FwdArgs* a, int grid, size_t smem, cudaStream_t st, int* result) {
  if (op == OP_SET_SMEM) return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (op == OP_OCCUPANCY) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(result, kern, nt, smem);
  kern<<<grid, nt, smem, st>>>(*a);
  return cudaGetLastError();
}

template <int L, int TPF, int NW, int DUAL, bool TM = false>
cudaError_t by_mode(int op, int mode, const FwdArgs* a, int grid, size_t smem, cudaStream_t st, int* result) {
  switch (mode) {
    case MODE_STFT: return run_op(fwd_kernel<L, TPF, NW, MODE_STFT, DUAL, TM>, op, NW * 32, a, grid, smem, st, result);
    case MODE_MEL: return run_op(fwd_kernel<L, TPF, NW, MODE_MEL, DUAL, TM>, op, NW * 32, a, grid, smem, st, result);
    case MODE_SPEC: return run_op(fwd_kernel<L, TPF, NW, MODE_SPEC, DUAL, TM>, op, NW * 32, a, grid, smem, st, result);
    case MODE_STATS: return run_op(fwd_kernel<L, TPF, NW, MODE_STATS, DUAL, TM>, op, NW * 32, a, grid, smem, st, result);
  }
  return cudaErrorInvalidValue;
}

}  // namespace

#define B2L_CAT2(a, b) a##b
#define B2L_CAT(a, b) B2L_CAT2(a, b)

// `nw` selects the variant: 16 or 8 warps; 116 = 16 warps as two independent 8-warp halves (NSPLIT = 2);
// + 1000 = the same with the window / twiddle tables in Tensor Memory (TM).
template <int L>
cudaError_t fwd_dispatch(int op, int nw, int mode, const FwdArgs* a, int grid, size_t smem, cudaStream_t st,
                         int* result) {
  constexpr int M = 1 << L;
  constexpr int TPF = M >= 32 ? M / 32 : 1;
  if constexpr (L >= 10) {
    if (nw == 16) return by_mode<L, TPF, 16, 1>(op, mode, a, grid, smem, st, result);
    if (nw == 8) return by_mode<L, TPF, 8, 1>(op, mode, a, grid, smem, st, result);
    if (nw == 116) return by_mode<L, TPF, 16, 2>(op, mode, a, grid, smem, st, result);
    if (nw == 1016) return by_mode<L, TPF, 16, 1, true>(op, mode, a, grid, smem, st, result);
    if constexpr (L <= 11) {
      if (nw == 1116) return by_mode<L, TPF, 16, 2, true>(op, mode, a, grid, smem, st, result);
    }
  } else {
    constexpr int NW = TPF > 16 ? 16 : TPF;
    if (nw == NW) return by_mode<L, TPF, NW, 1>(op, mode, a, grid, smem, st, result);
    if constexpr (L == 9) {
      if (nw == 116) return by_mode<L, TPF, 16, 2>(op, mode, a, grid, smem, st, result);
      if (nw == 1116) return by_mode<L, TPF, 16, 2, true>(op, mode, a, grid, smem, st, result);
    }
  }
  return cudaErrorInvalidValue;
}

cudaError_t B2L_CAT(fwd_op_, B2L_LOG2M)(int op, int nw, int mode, const FwdArgs* a, int grid, size_t smem,
                                         cudaStream_t st, int* result) {
  return fwd_dispatch<B2L_LOG2M>(op, nw, mode, a, grid, smem, st, result);
}

}  // namespace b2l
