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

}  // namespace rpsf
