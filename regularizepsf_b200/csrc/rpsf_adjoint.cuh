// rpsf_adjoint.cuh — the kernels that only the transpose of apply() needs (rpsf_plan_create_adjoint, DESIGN.md section 7).
// The transpose runs the forward kernels on the box of the patch footprints; these three move data in and out of it.
#pragma once
#include <cuda_runtime.h>

namespace rpsf {

// conj of the private kernel layout: complex values stored (re, im), so negate every odd real.  Used for kmain and
// knyq alike (the packed DC / Nyquist column holds plain values of the Hermitian part too).
template <typename T>
__global__ void conj_spectrum(const T* __restrict__ src, T* __restrict__ dst, long long n_reals) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_reals; i += (long long)gridDim.x * blockDim.x)
    dst[i] = (i & 1) ? -src[i] : src[i];
}

// rows x cols pixels of every frame from `src` (any row pitch / frame stride) into the box buffer; grid
// (column blocks, row blocks, frames), rows strided by the grid
template <typename T>
__global__ void adjoint_copy_in(const T* __restrict__ src, long long src_pitch, long long src_stride, int rows, int cols,
                                T* __restrict__ dst, long long dst_pitch, long long dst_stride) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= cols) return;
  const T* s = src + (long long)blockIdx.z * src_stride + x;
  T* d = dst + (long long)blockIdx.z * dst_stride + x;
  for (int y = blockIdx.y; y < rows; y += gridDim.y) d[(long long)y * dst_pitch] = s[(long long)y * src_pitch];
}

// padᵀ: out[y][x] = sum over box rows i of row_idx[row_off[y] .. row_off[y+1]) and box columns j of
// col_idx[col_off[x] .. col_off[x+1]) of box[i][j], in ascending (i, j) order.  The lists are the preimages of the
// np.pad index map (pad_index), so a pixel collects every padded position the forward copied it to; a gather, no
// atomics, bit-stable.  An empty list (the margin of constant mode, or a pixel no patch reads) gives 0.
template <typename T>
__global__ void fold_pad_adjoint(const T* __restrict__ box, long long box_pitch, long long box_stride,
                                 const int* __restrict__ row_off, const int* __restrict__ row_idx,
                                 const int* __restrict__ col_off, const int* __restrict__ col_idx,
                                 T* __restrict__ out, long long out_pitch, long long out_stride, int H, int W) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= W) return;
  const T* frame = box + (long long)blockIdx.z * box_stride;
  T* o = out + (long long)blockIdx.z * out_stride + x;
  const int c0 = col_off[x], c1 = col_off[x + 1];
  for (int y = blockIdx.y; y < H; y += gridDim.y) {
    T acc = T(0);
    for (int i = row_off[y]; i < row_off[y + 1]; ++i) {
      const T* row = frame + (long long)row_idx[i] * box_pitch;
      for (int j = c0; j < c1; ++j) acc += row[col_idx[j]];
    }
    o[(long long)y * out_pitch] = acc;
  }
}

}  // namespace rpsf
