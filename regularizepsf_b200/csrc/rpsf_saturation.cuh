// rpsf_saturation.cuh — the saturation branch of ArrayPSFTransform.apply on the device.
// Included by rpsf_api.cu only (patch-size independent, so not part of the per-size units).
#pragma once
#include "rpsf_kernels.cuh"

namespace rpsf {

// ============================================================================ saturation branch
// transform.py:125-138,171-172.  The reference pads 2P per side, masks `padded > threshold`,
// dilates the mask (scipy binary_dilation, 3x3 cross, `iterations` times), then walks the masked
// pixels IN RASTER ORDER replacing each by the nanmean of padded[i-h:i+h, j-h:j+h] (h = width//2;
// later pixels see earlier fills, masked pixels not yet reached count as NaN), corrects the
// filled frame and finally copies the raw value back into every masked pixel.  The fill runs in
// the padded domain (a mirrored blob is filled in a different order than its original), so the
// padded frame is materialised here — only on this branch — and K1 reads it with PAD_NONE.
struct SatGeom {
  int H, W, pad;            // frame shape, pad = 2P per side
  int Hp, Wp;               // padded shape
  int half;                 // neighbourhood_width // 2
  int row_begin, row_end;   // owned output rows
  long long img_pitch, img_frame_stride, out_pitch, out_frame_stride;
  int out_row0, pad_mode;
};

template <typename T> __device__ __forceinline__ T quiet_nan();
template <> __device__ __forceinline__ float quiet_nan<float>() { return __int_as_float(0x7fc00000); }
template <> __device__ __forceinline__ double quiet_nan<double>() { return __longlong_as_double(0x7ff8000000000000LL); }

// padded frame + initial mask (+ per-frame "any" flag).  grid (col blocks, Hp, frames).  The mask is decided on
// `src`, the caller's pixels before their conversion to T (laid out like `image`, with pitches of its own): the
// reference compares the float64 value, and a float64 or 32/64-bit integer pixel just above the threshold can round
// to it or below in float32.  Where the conversion is exact, src is the image itself.
template <typename T, typename TS>
__global__ void sat_pad_mask(const T* __restrict__ image, const TS* __restrict__ src, long long src_pitch,
                             long long src_frame_stride, T* __restrict__ pf, unsigned char* __restrict__ mask,
                             int* __restrict__ any_flag, double threshold, SatGeom g) {
  const int i = blockIdx.y, f = blockIdx.z;
  const bool direct = g.pad_mode == PAD_NONE;      // a materialised pad: negative indices address the caller's margin
  const int y = pad_index(i - g.pad, g.H, g.pad_mode);
  const bool row_in = y >= 0 || direct;
  const T* row = row_in ? image + (long long)f * g.img_frame_stride + (long long)y * g.img_pitch : nullptr;
  const TS* src_row = row_in ? src + (long long)f * src_frame_stride + (long long)y * src_pitch : nullptr;
  const long long base = ((long long)f * g.Hp + i) * g.Wp;
  bool any = false;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < g.Wp; j += gridDim.x * blockDim.x) {
    const int x = pad_index(j - g.pad, g.W, g.pad_mode);
    const bool in = row && (x >= 0 || direct);
    const T v = in ? row[x] : T(0);
    pf[base + j] = v;
    const bool m = (in ? double(src_row[x]) : 0.0) > threshold;
    mask[base + j] = m ? 1 : 0;
    any |= m;
  }
  if (__any_sync(0xffffffffu, any) && (threadIdx.x & 31) == 0) atomicOr(any_flag + f, 1);
}

// one binary_dilation iteration with the 3x3 cross, border value 0.  iterations < 1 means
// "until nothing changes" in scipy, which for a cross is "everything, if anything": mode_all.
__global__ void sat_dilate(const unsigned char* __restrict__ src, unsigned char* __restrict__ dst,
                           const int* __restrict__ any_flag, int Hp, int Wp, int mode_all) {
  const int i = blockIdx.y, f = blockIdx.z;
  const long long base = ((long long)f * Hp + i) * Wp;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < Wp; j += gridDim.x * blockDim.x) {
    unsigned char m;
    if (mode_all) {
      m = any_flag[f] ? 1 : 0;
    } else {
      m = src[base + j];
      if (!m) {
        if (j > 0) m |= src[base + j - 1];
        if (j + 1 < Wp) m |= src[base + j + 1];
        if (i > 0) m |= src[base + j - Wp];
        if (i + 1 < Hp) m |= src[base + j + Wp];
      }
    }
    dst[base + j] = m;
  }
}

// raster-ordered compaction of the masked pixels: per-row counts, scan, ordered scatter.
__global__ void sat_row_count(const unsigned char* __restrict__ mask, int* __restrict__ row_count, int Hp, int Wp) {
  const int warps = blockDim.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * warps + (threadIdx.x >> 5), f = blockIdx.y;
  if (i >= Hp) return;
  const unsigned char* row = mask + ((long long)f * Hp + i) * Wp;
  int n = 0;
  for (int j0 = 0; j0 < Wp; j0 += 32) {
    const int j = j0 + lane;
    n += __popc(__ballot_sync(0xffffffffu, j < Wp && row[j]));
  }
  if (lane == 0) row_count[(long long)f * (Hp + 1) + i] = n;
}
// exclusive scan of each frame's Hp row counts, in place; entry Hp receives the total.  One CTA per frame.
__global__ void sat_row_scan(int* __restrict__ row_count, int Hp) {
  __shared__ int carry, chunk_sum, part[32];
  int* rc = row_count + (long long)blockIdx.x * (Hp + 1);
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int i0 = 0; i0 < Hp; i0 += blockDim.x) {
    const int i = i0 + threadIdx.x;
    const int v = i < Hp ? rc[i] : 0;
    int incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += t; }
    if (lane == 31) part[w] = incl;
    __syncthreads();
    if (w == 0) {
      int pv = lane < (blockDim.x >> 5) ? part[lane] : 0, pi = pv;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, pi, d); if (lane >= d) pi += t; }
      part[lane] = pi - pv;                       // exclusive offset of each warp
      if (lane == 31) chunk_sum = pi;
    }
    __syncthreads();
    const int chunk_total = chunk_sum;
    if (i < Hp) rc[i] = carry + part[w] + incl - v;
    __syncthreads();
    if (threadIdx.x == 0) carry += chunk_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) rc[Hp] = carry;
}
__global__ void sat_row_scatter(const unsigned char* __restrict__ mask, const int* __restrict__ row_offset,
                                int* __restrict__ list, int Hp, int Wp) {
  const int warps = blockDim.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * warps + (threadIdx.x >> 5), f = blockIdx.y;
  if (i >= Hp) return;
  const unsigned char* row = mask + ((long long)f * Hp + i) * Wp;
  int* out = list + (long long)f * Hp * Wp;
  int at = row_offset[(long long)f * (Hp + 1) + i];
  for (int j0 = 0; j0 < Wp; j0 += 32) {
    const int j = j0 + lane;
    const bool m = j < Wp && row[j];
    const unsigned b = __ballot_sync(0xffffffffu, m);
    if (m) out[at + __popc(b & ((1u << lane) - 1u))] = i * Wp + j;
    at += __popc(b);
  }
}

// The ordered fill.  state: 0 = not masked, 1 = masked, not filled yet, 2 = filled.  A pixel is
// ready once no masked pixel of its window that precedes it in raster order is still pending;
// then its window holds exactly what the sequential reference loop would see (pending pixels
// after it are NaN there too).  CTAs claim 256-pixel chunks of the raster-ordered list by ticket,
// so every dependency lives in the same or an already-claimed chunk and polling cannot deadlock.
template <typename T>
__global__ void sat_fill(T* __restrict__ pf_all, unsigned char* __restrict__ state_all, const int* __restrict__ list_all,
                         const int* __restrict__ row_offset, int* __restrict__ tickets, SatGeom g) {
  const int f = blockIdx.y;
  T* pf = pf_all + (long long)f * g.Hp * g.Wp;
  volatile unsigned char* state = state_all + (long long)f * g.Hp * g.Wp;
  const int* list = list_all + (long long)f * g.Hp * g.Wp;
  const int total = row_offset[(long long)f * (g.Hp + 1) + g.Hp];
  __shared__ int s_ticket;
  const int h = g.half;
  for (;;) {
    if (threadIdx.x == 0) s_ticket = atomicAdd(tickets + f, 1);
    __syncthreads();
    const long long base = (long long)s_ticket * blockDim.x;
    __syncthreads();
    if (base >= total) break;
    const long long idx = base + threadIdx.x;
    bool done = idx >= total;
    int i = 0, j = 0;
    if (!done) { const int lin = list[idx]; i = lin / g.Wp; j = lin - i * g.Wp; }
    // numpy slices padded[i-h:i+h, j-h:j+h]: a negative start wraps around and the slice is empty
    const bool empty = h <= 0 || i < h || j < h;
    const int i1 = min(i + h, g.Hp), j1 = min(j + h, g.Wp);
    while (!done) {
      bool ready = true;
      if (!empty) {
        for (int ii = i - h; ii <= i && ready; ++ii) {
          const int jend = ii < i ? j1 : j;
          for (int jj = j - h; jj < jend; ++jj)
            if (state[(long long)ii * g.Wp + jj] == 1) { ready = false; break; }
        }
      }
      if (ready) {
        __threadfence();
        T sum = T(0);
        int cnt = 0;
        if (!empty) {
          for (int ii = i - h; ii < i1; ++ii)
            for (int jj = j - h; jj < j1; ++jj) {
              const long long at = (long long)ii * g.Wp + jj;
              // a masked pixel at or after (i, j) in raster order is still NaN when the reference
              // reaches (i, j) — even if it is already filled here (the window is asymmetric, so
              // a later pixel in column j-h does not depend on this one and may finish first)
              const bool later = ii > i || (ii == i && jj >= j);
              if (later ? state[at] != 0 : state[at] == 1) continue;
              const T v = *(volatile T*)(pf + at);
              if (v == v) { sum += v; ++cnt; }
            }
        }
        *(volatile T*)(pf + (long long)i * g.Wp + j) = cnt ? sum / T(cnt) : quiet_nan<T>();
        __threadfence();
        state[(long long)i * g.Wp + j] = 2;
        done = true;
      }
    }
    __syncthreads();
  }
}

// canvas[mask] = raw[mask] (transform.py:171-172), restricted to the cropped, owned rows.
template <typename T>
__global__ void sat_restore(const T* __restrict__ image, T* __restrict__ out, const int* __restrict__ list_all,
                            const int* __restrict__ row_offset, SatGeom g) {
  const int f = blockIdx.y;
  const int* list = list_all + (long long)f * g.Hp * g.Wp;
  const int total = row_offset[(long long)f * (g.Hp + 1) + g.Hp];
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < total; k += gridDim.x * blockDim.x) {
    const int lin = list[k];
    const int i = lin / g.Wp, j = lin - i * g.Wp;
    const int y = i - g.pad, x = j - g.pad;
    if (y < g.row_begin || y >= g.row_end || x < 0 || x >= g.W) continue;
    out[(long long)f * g.out_frame_stride + (long long)(y - g.out_row0) * g.out_pitch + x] =
        image[(long long)f * g.img_frame_stride + (long long)y * g.img_pitch + x];
  }
}

// ============================================================================ caller-given mask
// apply(mask=M): the padded frame's pixels marked by pad(M) are filled like saturated ones.  With an infinite threshold
// the map is linear in the image; its transpose runs the fill backwards (sat_fill_count, sat_fill_adjoint, mask_gather).

// state[i][j] |= M[pad_index(i - pad)][pad_index(j - pad)]: the caller's mask padded with the frame's index map (the margin
// of constant mode is unmasked).  mask_frame_stride 0 shares one mask across the frames.  grid (col blocks, Hp, frames).
__global__ void mask_ingest(const unsigned char* __restrict__ mask, long long mask_pitch, long long mask_frame_stride,
                            unsigned char* __restrict__ state, SatGeom g) {
  const int i = blockIdx.y, f = blockIdx.z;
  const int y = pad_index(i - g.pad, g.H, g.pad_mode);
  if (y < 0) return;
  const unsigned char* row = mask + (long long)f * mask_frame_stride + (long long)y * mask_pitch;
  const long long base = ((long long)f * g.Hp + i) * g.Wp;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < g.Wp; j += gridDim.x * blockDim.x) {
    const int x = pad_index(j - g.pad, g.W, g.pad_mode);
    if (x >= 0 && row[x]) state[base + j] = 1;
  }
}

// The contributor count n of every masked pixel when the unmasked pixels are finite: the `cnt` sat_fill reaches, decided
// by the mask alone.  The same raster-ordered chunks, tickets and readiness rule as sat_fill.  state: 1 (pending) ->
// 2 (n > 0) or 3 (n = 0: the fill is NaN, a structural NaN that later windows skip).
__global__ void sat_fill_count(unsigned char* __restrict__ state_all, const int* __restrict__ list_all,
                               const int* __restrict__ row_offset, int* __restrict__ tickets, int* __restrict__ count_all,
                               SatGeom g) {
  const int f = blockIdx.y;
  volatile unsigned char* state = state_all + (long long)f * g.Hp * g.Wp;
  const int* list = list_all + (long long)f * g.Hp * g.Wp;
  int* count = count_all + (long long)f * g.Hp * g.Wp;
  const int total = row_offset[(long long)f * (g.Hp + 1) + g.Hp];
  __shared__ int s_ticket;
  const int h = g.half;
  for (;;) {
    if (threadIdx.x == 0) s_ticket = atomicAdd(tickets + f, 1);
    __syncthreads();
    const long long base = (long long)s_ticket * blockDim.x;
    __syncthreads();
    if (base >= total) break;
    const long long idx = base + threadIdx.x;
    bool done = idx >= total;
    int i = 0, j = 0;
    if (!done) { const int lin = list[idx]; i = lin / g.Wp; j = lin - i * g.Wp; }
    const bool empty = h <= 0 || i < h || j < h;
    const int i1 = min(i + h, g.Hp), j1 = min(j + h, g.Wp);
    while (!done) {
      bool ready = true;
      if (!empty) {
        for (int ii = i - h; ii <= i && ready; ++ii) {
          const int jend = ii < i ? j1 : j;
          for (int jj = j - h; jj < jend; ++jj)
            if (state[(long long)ii * g.Wp + jj] == 1) { ready = false; break; }
        }
      }
      if (ready) {
        __threadfence();
        int cnt = 0;
        if (!empty) {
          for (int ii = i - h; ii < i1; ++ii)
            for (int jj = j - h; jj < j1; ++jj) {
              const unsigned char st = state[(long long)ii * g.Wp + jj];
              const bool later = ii > i || (ii == i && jj >= j);
              cnt += st == 0 || (!later && st == 2);
            }
        }
        count[(long long)i * g.Wp + j] = cnt;
        __threadfence();
        state[(long long)i * g.Wp + j] = cnt ? 2 : 3;
        done = true;
      }
    }
    __syncthreads();
  }
}

// The later masked pixels m' = (ii, jj) whose window holds (i, j): ii in (i - h, i + h], jj in (j - h, j + h], with a
// non-empty window (ii >= h, jj >= h).  `from_later`: only those after (i, j) in raster order.
struct FillReach { int i0, i1, j0, j1; };
__device__ __forceinline__ FillReach fill_reach(int i, int j, int h, int Hp, int Wp) {
  return {max(i - h + 1, h), min(i + h, Hp - 1), max(j - h + 1, h), min(j + h, Wp - 1)};
}

// The transposed fill, for the masked pixels, in gather form: u holds v on entry; on exit u[m] = (v[m] + sum of u[m']
// over the later masked m' with n > 0 whose window holds m) / n[m], the share m passes to each pixel of its window (0
// for a structural NaN).  CTAs claim 256-pixel chunks from the END of the raster-ordered list by ticket: every m' a
// pixel waits for comes later in the list, so it lives in the same or an already-claimed chunk and polling cannot
// deadlock (sat_fill's argument, reversed).  No atomics on values, a fixed summation order: bit-stable.
// state: 2 (n > 0, pending) -> 4 (done); 3 stays.
template <typename T>
__global__ void sat_fill_adjoint(T* __restrict__ u_all, unsigned char* __restrict__ state_all,
                                 const int* __restrict__ list_all, const int* __restrict__ row_offset,
                                 int* __restrict__ tickets, const int* __restrict__ count_all, SatGeom g) {
  const int f = blockIdx.y;
  T* u = u_all + (long long)f * g.Hp * g.Wp;
  volatile unsigned char* state = state_all + (long long)f * g.Hp * g.Wp;
  const int* list = list_all + (long long)f * g.Hp * g.Wp;
  const int* count = count_all + (long long)f * g.Hp * g.Wp;
  const int total = row_offset[(long long)f * (g.Hp + 1) + g.Hp];
  __shared__ int s_ticket;
  const int h = g.half;
  for (;;) {
    if (threadIdx.x == 0) s_ticket = atomicAdd(tickets + f, 1);
    __syncthreads();
    const long long end = (long long)total - (long long)s_ticket * blockDim.x;
    __syncthreads();
    if (end <= 0) break;
    const long long idx = end - blockDim.x + threadIdx.x;
    int i = 0, j = 0;
    bool done = idx < 0;
    if (!done) { const int lin = list[idx]; i = lin / g.Wp; j = lin - i * g.Wp; }
    const long long at0 = (long long)i * g.Wp + j;
    if (!done && state[at0] == 3) { u[at0] = T(0); done = true; }
    const FillReach r = fill_reach(i, j, h, g.Hp, g.Wp);
    while (!done) {
      bool ready = true;
      for (int ii = max(r.i0, i); ii <= r.i1 && ready; ++ii)
        for (int jj = ii == i ? max(r.j0, j + 1) : r.j0; jj <= r.j1; ++jj)
          if (state[(long long)ii * g.Wp + jj] == 2) { ready = false; break; }
      if (ready) {
        __threadfence();
        T acc = u[at0];
        for (int ii = max(r.i0, i); ii <= r.i1; ++ii)
          for (int jj = ii == i ? max(r.j0, j + 1) : r.j0; jj <= r.j1; ++jj) {
            const long long at = (long long)ii * g.Wp + jj;
            if (state[at] == 4) acc += *(volatile T*)(u + at);
          }
        *(volatile T*)(u + at0) = acc / T(count[at0]);
        __threadfence();
        state[at0] = 4;
        done = true;
      }
    }
    __syncthreads();
  }
}

// Fᵀ for the unmasked pixels and the combine, unordered: o[k] = v[k] + the shares of the masked m' (state 4) whose window
// holds k for an unmasked k; grad at a masked pixel of the frame, 0 at one in the margin (there the forward restores a
// raw pixel of the margin, which no output reads).  grid (col blocks, Hp, frames).
template <typename T>
__global__ void mask_gather_adjoint(const T* __restrict__ u_all, const unsigned char* __restrict__ state_all,
                                    const T* __restrict__ grad, long long grad_pitch, long long grad_frame_stride,
                                    T* __restrict__ o_all, SatGeom g) {
  const int i = blockIdx.y, f = blockIdx.z;
  const long long frame = (long long)f * g.Hp * g.Wp;
  const T* u = u_all + frame;
  const unsigned char* state = state_all + frame;
  const int y = i - g.pad;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < g.Wp; j += gridDim.x * blockDim.x) {
    const long long at0 = (long long)i * g.Wp + j;
    T acc;
    if (state[at0] != 0) {
      const int x = j - g.pad;
      acc = (y >= 0 && y < g.H && x >= 0 && x < g.W)
                ? grad[(long long)f * grad_frame_stride + (long long)y * grad_pitch + x] : T(0);
    } else {
      acc = u[at0];
      const FillReach r = fill_reach(i, j, g.half, g.Hp, g.Wp);
      for (int ii = r.i0; ii <= r.i1; ++ii)
        for (int jj = r.j0; jj <= r.j1; ++jj) {
          const long long at = (long long)ii * g.Wp + jj;
          if (state[at] == 4) acc += u[at];
        }
    }
    o_all[frame + at0] = acc;
  }
}

// (1 - M) * src into the box of an adjoint plan (adjoint_copy_in with the caller's mask; rows x cols pixels from frame
// position (r0, c0)).  grid (column blocks, row blocks, frames).
template <typename T>
__global__ void mask_copy_in(const T* __restrict__ src, long long src_pitch, long long src_stride,
                             const unsigned char* __restrict__ mask, long long mask_pitch, long long mask_stride,
                             int rows, int cols, T* __restrict__ dst, long long dst_pitch, long long dst_stride) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= cols) return;
  const T* s = src + (long long)blockIdx.z * src_stride + x;
  const unsigned char* m = mask + (long long)blockIdx.z * mask_stride + x;
  T* d = dst + (long long)blockIdx.z * dst_stride + x;
  for (int y = blockIdx.y; y < rows; y += gridDim.y)
    d[(long long)y * dst_pitch] = m[(long long)y * mask_pitch] ? T(0) : s[(long long)y * src_pitch];
}

// the box of an adjoint plan (frame rows [by0, by0 + bh), columns [bx0, bx0 + bw)) onto the padded frame, 0 outside it.
// grid (col blocks, Hp, frames).
template <typename T>
__global__ void box_to_padded(const T* __restrict__ box, long long box_pitch, long long box_stride, int by0, int bx0,
                              int bh, int bw, T* __restrict__ u_all, SatGeom g) {
  const int i = blockIdx.y, f = blockIdx.z;
  const int r = i - g.pad - by0;
  const bool row_in = r >= 0 && r < bh;
  const T* row = box + (long long)f * box_stride + (long long)r * box_pitch;
  T* dst = u_all + ((long long)f * g.Hp + i) * g.Wp;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < g.Wp; j += gridDim.x * blockDim.x) {
    const int c = j - g.pad - bx0;
    dst[j] = (row_in && c >= 0 && c < bw) ? row[c] : T(0);
  }
}

}  // namespace rpsf
