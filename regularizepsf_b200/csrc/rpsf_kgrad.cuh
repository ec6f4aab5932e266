// rpsf_kgrad.cuh — gradient of ArrayPSFTransform.apply with respect to the transfer kernel (DESIGN.md section 6).
//
// Without saturation apply is linear in the kernel.  For patch p and one frame
//   X_p = FFT2(w ⊙ S_p pad(x))              K1 of the forward plan (row spectra in its workspace)
//   G_p = FFT2(w ⊙ S_p zero_extend(g))      K1 of the adjoint plan, on its zero-bordered box
//   ∂<apply(x), g>/∂K_p = conj(X_p) ⊙ G_p / P²   summed over the frames of the batch
// in PyTorch's convention (∂L/∂Re + i ∂L/∂Im).  x and g are real, so the result is Hermitian and the column bins
// [0, P/2] determine it; the rest is written as their conjugate mirror.
//
// A CTA owns SLOTS (active patch, tile of C column bins) like the column pass K2.  Per frame, in order, it column-FFTs
// the X tile (coop_fft_forward), parks the spectrum in its own shared-memory slots, column-FFTs the G tile and adds
// conj(X) G to accumulators held per thread; the batch is summed in frame order, no atomics, so results are bit-stable.
// Column 0 of tile 0 packs the DC and Nyquist columns (z = a + i b, both real over rows): after the column FFT
// A = (Z + conj Z(-k)) / 2 and B = (Z - conj Z(-k)) / (2i).
#pragma once
#include "rpsf_kernels.cuh"

namespace rpsf {

template <int P, typename T> struct GradTile {
  using TL = Tile<P>;
  static constexpr int N1 = TL::N1, N2 = TL::N2, HALF = TL::HALF;
  // one 128-byte line per tile row (a narrower tile than K2's in double keeps P = 512 within shared memory)
  static constexpr int LINE = 128 / (int)sizeof(cplx<T>);
  static constexpr int C = HALF < LINE ? HALF : LINE;
  static constexpr int NTILE = HALF / C;
  static constexpr int SLOT_THREADS = C * N1;
  static constexpr size_t TILE_BYTES = sizeof(cplx<T>) * P * C;
  static constexpr int SLOTS_BY_THREADS = SLOT_THREADS >= 256 ? 1 : 256 / SLOT_THREADS;
  static constexpr int SLOTS_BY_SMEM = TILE_BYTES >= 65536 ? 1 : (int)(65536 / TILE_BYTES);
  static constexpr int SLOTS = SLOTS_BY_THREADS < SLOTS_BY_SMEM ? SLOTS_BY_THREADS : SLOTS_BY_SMEM;
  static constexpr int THREADS = SLOTS * SLOT_THREADS;
  // accumulators in registers up to 64 of them per thread; beyond (P = 512 in double) in the thread's own shared slots
  static constexpr bool ACC_REG = sizeof(cplx<T>) * N2 <= 256;
  // twiddles | FFT exchange | X of the frame | (accumulators) | per slot: X and accumulator of the Nyquist column
  static constexpr size_t SMEM =
      sizeof(cplx<T>) * (P + (size_t)SLOTS * ((ACC_REG ? 2 : 3) * (size_t)P * C + 2 * (size_t)P));
  static_assert(SMEM <= 227 * 1024, "kgrad tile does not fit shared memory");
};

// xspec / gspec: the band buffers of the forward and adjoint plans after K1 (rpsf_bands.cuh), each read through its own
// plan's bands and scaled by the row window on load (same active patches, same order).
// out: (n, P, P) complex, reference layout; the slot of active patch a is active[a].  Slots of patches that are not
// active are not touched (the caller zeroes them).
template <int P, typename T>
__global__ void __launch_bounds__(GradTile<P, T>::THREADS)
kgrad(const cplx<T>* __restrict__ xspec, const RowBands xb, const cplx<T>* __restrict__ gspec, const RowBands gb,
      cplx<T>* __restrict__ out, const int* __restrict__ active, const cplx<T>* __restrict__ tw_g,
      const T* __restrict__ win_g, int n_active, int batch) {
  using GT = GradTile<P, T>;
  constexpr int N1 = GT::N1, N2 = GT::N2, HALF = GT::HALF, C = GT::C, NTILE = GT::NTILE, SLOTS = GT::SLOTS;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  cplx<T>* xbuf = tw + P;                                   // FFT exchange, SLOTS * P * C
  cplx<T>* xs = xbuf + SLOTS * P * C;                       // X of the current frame, SLOTS * P * C
  cplx<T>* accs = xs + SLOTS * P * C;                       // !ACC_REG: accumulators, SLOTS * P * C
  cplx<T>* nyq = accs + (GT::ACC_REG ? 0 : SLOTS * P * C);  // SLOTS * 2P
  for (int i = threadIdx.x; i < P; i += blockDim.x) tw[i] = tw_g[i];

  const int c = threadIdx.x % C;
  const int n1 = (threadIdx.x / C) % N1;
  const int slot = threadIdx.x / (C * N1);
  const long long first = (long long)blockIdx.x * SLOTS;
  const long long sitem = first + slot;
  const long long total = (long long)n_active * NTILE;
  const bool valid = sitem < total;
  const int a = valid ? int(sitem / NTILE) : 0;
  const int tile = valid ? int(sitem % NTILE) : 1;          // never 0 when invalid
  bool any_tile0 = false;                                   // CTA-uniform
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) any_tile0 |= (first + s < total) && ((first + s) % NTILE == 0);
  const bool special = valid && tile == 0 && c == 0;

  // exchange / ownership index: element k2 of thread n1 of column c in this slot (each thread reads back only its own)
  auto ex = [=](int k2, int nn) { return ((slot * N2 + k2) * N1 + nn) * C + c; };
  auto sync = []() { __syncthreads(); };
  cplx<T>* nyq_x = nyq + slot * 2 * P;                      // X of the Nyquist column, this frame
  cplx<T>* nyq_acc = nyq_x + P;                             // its accumulated product

  cplx<T> acc[GT::ACC_REG ? N2 : 1];
  static_for<0, N2>([&](auto ee) {
    constexpr int e = decltype(ee)::value;
    if constexpr (GT::ACC_REG) acc[e] = mk<T>(T(0), T(0));
    else accs[ex(e, n1)] = mk<T>(T(0), T(0));
    if (special) nyq_acc[e * N1 + n1] = mk<T>(T(0), T(0));
  });
  __syncthreads();                                          // twiddle table visible

  const long long column = tile * C + c;
  // the column spectrum of one frame's tile in v (for the packed column: the DC column).  The Nyquist column of the
  // packed column goes to nyq_x (X), or is multiplied by conj(nyq_x) into nyq_acc (G).
  auto column_fft = [&](const cplx<T>* __restrict__ spec, const RowBands& rb, int f, cplx<T>(&v)[N2], bool is_g) {
    const cplx<T>* base = spec + ((long long)f * rb.frame_rows + (valid ? rb.patch_row[a] : 0)) * HALF + column;
    static_for<0, N2>([&](auto jj) {
      constexpr int j = decltype(jj)::value;
      const int r = n1 + N1 * j;
      v[j] = valid ? cscale_rn(base[(long long)r * HALF], T(0.5) * __ldg(win_g + r)) : mk<T>(T(0), T(0));
    });
    coop_fft_forward<P, T>(v, n1, xbuf, tw, ex, sync);
    if (any_tile0) {
      cplx<T>* zs = xbuf + slot * P;                        // natural order, one column per slot
      if (special) {
        static_for<0, N2>([&](auto ee) {
          constexpr int e = decltype(ee)::value;
          constexpr int m = e / N1, k1 = e % N1;
          zs[(n1 + N1 * m) + N2 * k1] = v[e];
        });
      }
      __syncthreads();
      if (special) {
        static_for<0, N2>([&](auto ee) {
          constexpr int e = decltype(ee)::value;
          constexpr int m = e / N1, k1 = e % N1;
          const int k = (n1 + N1 * m) + N2 * k1;
          const cplx<T> zr = zs[(P - k) & (P - 1)];
          const cplx<T> d = mk<T>(v[e].x - zr.x, v[e].y + zr.y);                 // Z - conj Z(-k)
          v[e] = mk<T>(T(0.5) * (v[e].x + zr.x), T(0.5) * (v[e].y - zr.y));     // A = (Z + conj Z(-k)) / 2
          const cplx<T> b = mk<T>(T(0.5) * d.y, T(-0.5) * d.x);                // B = (Z - conj Z(-k)) / (2i)
          if (is_g) nyq_acc[e * N1 + n1] = cadd(nyq_acc[e * N1 + n1], cmulc(b, nyq_x[e * N1 + n1]));
          else nyq_x[e * N1 + n1] = b;
        });
      }
      __syncthreads();
    }
  };

  for (int f = 0; f < batch; ++f) {
    cplx<T> v[N2];
    column_fft(xspec, xb, f, v, false);
    static_for<0, N2>([&](auto ee) { xs[ex(decltype(ee)::value, n1)] = v[decltype(ee)::value]; });
    column_fft(gspec, gb, f, v, true);
    static_for<0, N2>([&](auto ee) {
      constexpr int e = decltype(ee)::value;
      const cplx<T> prod = cmulc(v[e], xs[ex(e, n1)]);                         // G conj(X)
      if constexpr (GT::ACC_REG) acc[e] = cadd(acc[e], prod);
      else accs[ex(e, n1)] = cadd(accs[ex(e, n1)], prod);
    });
  }

  if (!valid) return;
  const T scale = T(1) / (T(P) * T(P));                     // a power of two: exact
  cplx<T>* o = out + (long long)active[a] * P * P;
  const int col = tile * C + c;
  static_for<0, N2>([&](auto ee) {
    constexpr int e = decltype(ee)::value;
    constexpr int m = e / N1, k1 = e % N1;
    const int k = (n1 + N1 * m) + N2 * k1;
    cplx<T> val;
    if constexpr (GT::ACC_REG) val = acc[e];
    else val = accs[ex(e, n1)];
    val = cscale(val, scale);
    if (special) {
      o[(long long)k * P] = val;
      o[(long long)k * P + HALF] = cscale(nyq_acc[e * N1 + n1], scale);
    } else {
      o[(long long)k * P + col] = val;
      o[(long long)((P - k) & (P - 1)) * P + (P - col)] = mk<T>(val.x, -val.y);
    }
  });
}

}  // namespace rpsf
