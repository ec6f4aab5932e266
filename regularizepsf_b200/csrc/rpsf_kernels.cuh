// rpsf_kernels.cuh — sm_100a kernels for ArrayPSFTransform.apply and its setup.
//
// Reference path: regularizepsf/transform.py:116-177 (apply), :78-82 (construct),
// regularizepsf/psf.py:216-219 (PSF FFT cube).  Design notes in DESIGN.md.
//
// Data layout in HBM
//   image      [frame][row][col] real T, row pitch in elements (resident rows may be a slab)
//   spectrum   workspace S[frame][active patch][row r][P/2 bins] complex T.  Each row holds the
//              Hermitian half of that row's spectrum; bin 0 packs (DC.re, Nyquist.re), which
//              are both real for a real row, so a row is exactly P/2 complex = the size of
//              the real row it came from.
//   kernel     private, built once per transform from the (N,P,P) reference-layout cube:
//              Hermitian-symmetrised (only that part survives np.real(ifft2(.)),
//              transform.py:164), scaled by 1/P^2, and permuted into the register order of
//              the column-FFT kernel so every load is a coalesced 8/16-byte vector.
#pragma once
#include <cstdint>
#include "rpsf_fft.cuh"
#include "rpsf_bands.cuh"

// Programmatic dependent launch (sm_90+).  K1 -> K2 -> K3 -> next K1 are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization (rpsf_inst.cu: launch_chain): a kernel's CTAs may become resident
// while the kernel before it in the stream drains, run their prologue (tables, mbarrier init, the transfer-kernel
// tile) and then wait here for the predecessor to complete and flush.  Every kernel waits BEFORE it releases its own
// dependents, so "my CTAs run" implies "everything before my predecessor is complete": plan constants written by an
// earlier kernel of the stream are safe to read in the prologue.  Both are no-ops in a launch without the attribute.
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

namespace rpsf {

// PAD_NONE: the frame pointer addresses a materialised padded frame (saturation branch), every
// index a patch can produce is in bounds and is used as is (it may be negative).
enum PadMode : int { PAD_SYMMETRIC = 0, PAD_REFLECT = 1, PAD_EDGE = 2, PAD_WRAP = 3, PAD_CONSTANT = 4, PAD_NONE = 5 };

// np.pad index maps (transform.py:119-123 pads 2P per side; only the part a patch touches is
// ever read, so the pad is never materialised).  Returns -1 for "constant" outside the frame.
__host__ __device__ __forceinline__ int pad_index(int i, int n, int mode) {
  if ((i >= 0 && i < n) || mode == PAD_NONE) return i;
  switch (mode) {
    case PAD_SYMMETRIC: {
      if (i < 0 && i >= -n) return -i - 1;                  // first reflection: no division
      if (i >= n && i < 2 * n) return 2 * n - 1 - i;
      const int period = 2 * n;
      int m = i % period; if (m < 0) m += period;
      return m < n ? m : period - 1 - m;
    }
    case PAD_REFLECT: {
      if (n == 1) return 0;
      if (i < 0 && i > -n) return -i;
      if (i >= n && i < 2 * n - 1) return 2 * n - 2 - i;
      const int period = 2 * n - 2;
      int m = i % period; if (m < 0) m += period;
      return m < n ? m : period - m;
    }
    case PAD_EDGE: return i < 0 ? 0 : n - 1;
    case PAD_WRAP: { int m = i % n; if (m < 0) m += n; return m; }
    default: return -1;
  }
}

struct ApplyGeom {
  int H, W;                 // full frame shape
  int img_row0, img_rows;   // resident image rows [img_row0, img_row0 + img_rows)
  long long img_pitch;      // elements
  long long img_frame_stride;
  int out_row0;             // global row of out[.][0][.]
  int row_begin, row_end;   // owned output rows (global), clipped to [0, H)
  long long out_pitch, out_frame_stride;
  int n_active;             // patches this plan computes
  int pad_mode;
  // Patch sizes without a native FFT length run embedded in the next power of two M >= 2 P - 1 (see
  // embed_transfer_kernel): the FFT length is M, the window and every contribution end at win_len = P.  Equal to the
  // FFT length otherwise.  Only the plain K1 and the colour-phase K3 honour it (the planner selects them).
  int win_len;
};

template <int P> struct Tile {
  static constexpr int N1 = Split<P>::N1, N2 = Split<P>::N2;
  static constexpr int HALF = P / 2;
  static constexpr int C = HALF < 16 ? HALF : 16;           // columns per column-FFT tile (16 = a full 128-byte line per row)
  static constexpr int NTILE = HALF / C;
  static constexpr int SLOT_THREADS = C * N1;
  static constexpr int CTA_THREADS = 256;                   // per column-FFT CTA: tiles are packed into slots up to this size
  static constexpr int SLOTS = SLOT_THREADS >= CTA_THREADS ? 1 : CTA_THREADS / SLOT_THREADS;
  static constexpr int K2_THREADS = SLOTS * SLOT_THREADS;
  // row kernels: teams of N1 threads inside a warp
  static constexpr int TEAMS = 256 / N1;
  static constexpr int ROW_THREADS = 256;
  static constexpr int EX_STRIDE = N1 + 1;                  // padded exchange row (bank spread)
  static constexpr int EX_SIZE = N2 * EX_STRIDE;
  static constexpr int SCR = EX_SIZE > P ? EX_SIZE : P;     // per-team scratch, complex elements
};

__device__ __forceinline__ unsigned team_mask(int n1) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned base = lane & ~unsigned(n1 - 1);
  return (n1 >= 32 ? 0xffffffffu : ((1u << n1) - 1u)) << base;
}

// ============================================================================ K1
// gather + apodize + row FFT.  transform.py:141-163 (slice, stack, window, first FFT axis).
// One team per pair of band rows (rpsf_bands.cuh): z = (row_a + i*row_b) * w_col, complex FFT-P, split into the
// two Hermitian half-spectra, stored packed without the row window.
template <int P, typename T>
__global__ void __launch_bounds__(Tile<P>::ROW_THREADS)
k1_gather_window_rowfft(const T* __restrict__ image, cplx<T>* __restrict__ spec, const RowBands rb,
                        const cplx<T>* __restrict__ tw_g, const T* __restrict__ win_g, ApplyGeom g) {
  using TL = Tile<P>;
  constexpr int N1 = TL::N1, N2 = TL::N2, HALF = TL::HALF, PAIRS = band_quantum<P>() / 2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  T* win = reinterpret_cast<T*>(tw + P);
  cplx<T>* scratch_all = reinterpret_cast<cplx<T>*>(win + P);
  for (int i = threadIdx.x; i < P; i += blockDim.x) { tw[i] = tw_g[i]; win[i] = win_g[i]; }
  __syncthreads();

  const int team = threadIdx.x / N1, t = threadIdx.x % N1;
  cplx<T>* scr = scratch_all + team * TL::SCR;
  const long long item = (long long)blockIdx.x * TL::TEAMS + team;   // (band item, row pair)
  const int bi = int(item / PAIRS), pair = int(item % PAIRS);
  if (bi >= rb.n_items) return;
  const unsigned mask = team_mask(N1);
  auto ex = [](int k2, int n1) { return k2 * TL::EX_STRIDE + n1; };
  auto sync = [mask]() { __syncwarp(mask); };

  const BandItem it = rb.items[bi];
  const int ra = 2 * pair, rb_ = ra + 1;
  const bool live_a = (it.live >> ra) & 1u, live_b = (it.live >> rb_) & 1u;
  // neither row is in a patch window: nobody reads this pair — the whole team leaves
  if (!live_a && !live_b) return;
  const int ya = pad_index(it.row + ra, g.H, g.pad_mode);
  const int yb = pad_index(it.row + rb_, g.H, g.pad_mode);
  const T* img = image + (long long)blockIdx.y * g.img_frame_stride;
  const bool direct = g.pad_mode == PAD_NONE;
  // zero rows of the band and columns past the window (embedded patch sizes) are exact zeros, not 0 * pixel: a NaN
  // outside the patch must not leak in
  const T* rowa = ((ya < 0 && !direct) || !live_a) ? nullptr : img + (long long)(ya - g.img_row0) * g.img_pitch;
  const T* rowb = ((yb < 0 && !direct) || !live_b) ? nullptr : img + (long long)(yb - g.img_row0) * g.img_pitch;

  cplx<T> v[N2];
  const bool interior = (direct || (it.cx >= 0 && it.cx + P <= g.W)) && g.win_len >= P;
  if (interior && rowa && rowb) {
    static_for<0, N2>([&](auto jj) {
      constexpr int j = decltype(jj)::value;
      const int n = t + N1 * j;
      v[j] = cscale(mk<T>(rowa[it.cx + n], rowb[it.cx + n]), win[n]);
    });
  } else {
    static_for<0, N2>([&](auto jj) {
      constexpr int j = decltype(jj)::value;
      const int n = t + N1 * j;
      const int x = pad_index(it.cx + n, g.W, g.pad_mode);
      const bool inside = (x >= 0 || direct) && n < g.win_len;
      const T pa = (rowa && inside) ? rowa[x] : T(0);
      const T pb = (rowb && inside) ? rowb[x] : T(0);
      v[j] = cscale(mk<T>(pa, pb), win[n]);
    });
  }

  coop_fft_forward<P, T>(v, t, scr, tw, ex, sync);

  // natural-order staging: Z[k], k = (t + N1*m) + N2*k1
  static_for<0, N2>([&](auto ee) {
    constexpr int e = decltype(ee)::value;
    constexpr int m = e / N1, k1 = e % N1;
    scr[(t + N1 * m) + N2 * k1] = v[e];
  });
  sync();
  // A[k] = Z[k] + conj Z[P-k],  B[k] = -i (Z[k] - conj Z[P-k]): twice the half-spectra; the reader applies 1/2 and the
  // row window
  cplx<T>* outa = spec + ((long long)blockIdx.y * rb.frame_rows + it.buf_row + ra) * HALF;
  cplx<T>* outb = outa + HALF;
#pragma unroll
  for (int i = 0; i < HALF / N1; ++i) {
    const int k = t + N1 * i;
    const cplx<T> z1 = scr[k];
    const cplx<T> z2 = scr[(P - k) & (P - 1)];
    const cplx<T> D = padd(z1, mk<T>(-z2.x, z2.y));                 // z1 - conj z2
    cplx<T> A = padd(z1, mk<T>(z2.x, -z2.y));                       // z1 + conj z2
    cplx<T> B = mk<T>(D.y, -D.x);                                   // -i (z1 - conj z2)
    if (k == 0) {                       // pack (DC, Nyquist): both real
      const cplx<T> zn = scr[HALF];
      A = mk<T>(T(2) * z1.x, T(2) * zn.x);
      B = mk<T>(T(2) * z1.y, T(2) * zn.y);
    }
    outa[k] = A;
    outb[k] = B;
  }
}

// ============================================================================ K2
// column FFT x transfer kernel x column IFFT: from a patch's rows of the band buffer (rpsf_bands.cuh), scaled by the
// row window on load, to the patch's slot of the spectrum workspace.
// transform.py:163-164 (second FFT axis, `patches * kernel`, first IFFT axis).
// A CTA owns SLOTS tiles of [P rows] x [C bins]; thread (c, n1) of a slot owns P/N1 = N2
// elements of column c.  c is the fastest thread index, so every global access is a
// C*8-byte run and every shared access is conflict-free without padding.
// PRUNED (embedded patch sizes, win_len < P): rows past the window hold no data — the gather kernel skips them — so
// they are taken as zeros without being loaded, and results are only stored for the rows the overlap-add reads
// (win_len rounded up to a whole row pair): the pass moves win_len / P of the bytes.
template <int P, typename T, bool PRUNED = false>
__global__ void __launch_bounds__(Tile<P>::K2_THREADS, (Tile<P>::N2 * sizeof(T) <= 64) ? 3 : (Tile<P>::N2 * sizeof(T) <= 128) ? 2 : 1)
k2_colfft_mul_colifft(const cplx<T>* __restrict__ bands, const RowBands rb, cplx<T>* __restrict__ spec,
                      const cplx<T>* __restrict__ kmain, const cplx<T>* __restrict__ knyq, const int* __restrict__ active,
                      const cplx<T>* __restrict__ tw_g, const T* __restrict__ win_g, int batch, int frames_per_cta,
                      ApplyGeom g) {
  using TL = Tile<P>;
  constexpr int N1 = TL::N1, N2 = TL::N2, HALF = TL::HALF, C = TL::C, NTILE = TL::NTILE;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  cplx<T>* xbuf = tw + P;                                   // SLOTS * P * C complex
  T* wy = reinterpret_cast<T*>(xbuf + TL::SLOTS * P * C);   // row window as the row pass applied it: 0.5 * win
  for (int i = threadIdx.x; i < P; i += blockDim.x) { tw[i] = tw_g[i]; wy[i] = T(0.5) * win_g[i]; }
  __syncthreads();

  const int c = threadIdx.x % C;
  const int n1 = (threadIdx.x / C) % N1;
  const int slot = threadIdx.x / (C * N1);
  const long long first = (long long)blockIdx.x * TL::SLOTS;
  const long long sitem = first + slot;
  const long long total = (long long)g.n_active * NTILE;
  const bool valid = sitem < total;
  const int a = valid ? int(sitem / NTILE) : 0;
  const int tile = valid ? int(sitem % NTILE) : 1;              // never 0 when invalid
  // does any slot of this CTA hold tile 0 (the packed DC/Nyquist column)?  CTA-uniform.
  bool any_tile0 = false;
#pragma unroll
  for (int s = 0; s < TL::SLOTS; ++s) any_tile0 |= (first + s < total) && ((first + s) % NTILE == 0);
  const bool special = valid && tile == 0 && c == 0;

  // The transfer-kernel tile is loaded once and reused for every frame of the batch this CTA
  // walks: registers when it fits (<= 32 extra 32-bit registers), else re-read (L1/L2 hits).
  constexpr bool PREFETCH = sizeof(cplx<T>) * N2 <= 128;
  cplx<T> kv[PREFETCH ? N2 : 1];
  const int gp = valid ? active[a] : 0;
  const cplx<T>* kp = kmain + (((long long)gp * NTILE + (valid ? tile : 0)) * N2) * (N1 * C) + n1 * C + c;
  if constexpr (PREFETCH) {
    static_for<0, N2>([&](auto ee) {
      constexpr int e = decltype(ee)::value;
      kv[e] = valid ? kp[(long long)e * (N1 * C)] : mk<T>(T(0), T(0));
    });
  }
  auto kval = [&](auto ee) -> cplx<T> {
    constexpr int e = decltype(ee)::value;
    if constexpr (PREFETCH) return kv[e];
    else return valid ? kp[(long long)e * (N1 * C)] : mk<T>(T(0), T(0));
  };
  auto ex = [=](int k2, int nn) { return ((slot * N2 + k2) * N1 + nn) * C + c; };
  auto sync = []() { __syncthreads(); };

  const int f_begin = blockIdx.y * frames_per_cta;
  const int f_end = min(batch, f_begin + frames_per_cta);
  const int live_rows = (g.win_len + 1) & ~1;               // the overlap-add reads whole row pairs
  const int prow = valid ? rb.patch_row[a] : 0;
  for (int f = f_begin; f < f_end; ++f) {
    cplx<T>* base = spec + (((long long)f * g.n_active + a) * P) * HALF + tile * C + c;
    const cplx<T>* src = bands + ((long long)f * rb.frame_rows + prow) * HALF + tile * C + c;
    cplx<T> v[N2];
    static_for<0, N2>([&](auto jj) {
      constexpr int j = decltype(jj)::value;
      const int r = n1 + N1 * j;
      const bool live = !PRUNED || r < live_rows;
      v[j] = (valid && live) ? cscale_rn(src[(long long)r * HALF], wy[r]) : mk<T>(T(0), T(0));
    });
    __syncthreads();                                        // the previous frame's exchange reads are done

    coop_fft_forward<P, T>(v, n1, xbuf, tw, ex, sync);

    if (any_tile0) {
      // Packed column: z = a + i*b with a = DC column, b = Nyquist column (both real sequences
      // over rows).  Z'[k] = A[k] K0[k] + i B[k] KN[k] = ((Z+Zm) K0 + (Z-Zm) KN) / 2, Zm = conj Z[-k].
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
        const cplx<T>* kn = knyq + (long long)gp * P + n1;
        static_for<0, N2>([&](auto ee) {
          constexpr int e = decltype(ee)::value;
          constexpr int m = e / N1, k1 = e % N1;
          const int k = (n1 + N1 * m) + N2 * k1;
          const cplx<T> zr = zs[(P - k) & (P - 1)];
          const cplx<T> zm = mk<T>(zr.x, -zr.y);
          const cplx<T> sum = mk<T>(T(0.5) * (v[e].x + zm.x), T(0.5) * (v[e].y + zm.y));
          const cplx<T> dif = mk<T>(T(0.5) * (v[e].x - zm.x), T(0.5) * (v[e].y - zm.y));
          v[e] = cadd(cmul(sum, kval(ee)), cmul(dif, kn[e * N1]));
        });
      }
      __syncthreads();
    }
    if (!special) {
      static_for<0, N2>([&](auto ee) { v[decltype(ee)::value] = cmul(v[decltype(ee)::value], kval(ee)); });
    }

    coop_fft_inverse<P, T>(v, n1, xbuf, tw, ex, sync);
    if (valid) {
      static_for<0, N2>([&](auto jj) {
        constexpr int j = decltype(jj)::value;
        if (!PRUNED || n1 + N1 * j < live_rows) base[(long long)(n1 + N1 * j) * HALF] = v[j];
      });
    }
  }
}

// ---------------------------------------------------------------------------- K2, pipelined
// Same arithmetic as k2_colfft_mul_colifft, restructured so a CTA never waits on HBM: while the
// tile of frame f is being transformed, the tile of frame f+1 streams into the other of two
// shared-memory stages with cp.async (16-byte LDGSTS, no register staging).  A stage doubles as
// the FFT exchange buffer of its tile — thread (c, n1) writes its pass-A outputs exactly over
// the inputs it just read — so two stages plus the twiddle table are all the shared memory
// there is, and results go straight from registers to HBM.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait_pending() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// shared-memory tile stages per CTA: tiles f+1 .. f+K2_STAGES-1 are in flight while tile f is transformed.  Three
// stages were measured slower than two (32.4 vs 31.2 us per frame at B=8): the tile always lands in time.
constexpr int K2_STAGES = 2;

// The frame loop of one CTA.  TILE0: some slot of this CTA holds tile 0, whose column 0 packs the DC
// and Nyquist columns (z = a + i*b, both real sequences over rows):
//   Z'[k] = A[k] K0[k] + i B[k] KN[k] = ((Z + Zm) K0 + (Z - Zm) KN) / 2,  Zm = conj Z[-k].
// Every thread of such a CTA runs that formula — ordinary columns with Zm := Z and KN := 0, which
// reduces it to Z K0 — so neither instantiation has a divergent definition of the spectrum
// registers (a join there costs a register-pair move per element on the common path).
// TPC > 1 (one slot per CTA only): the CTA walks TPC adjacent tiles of its patch, tile-major, so that with one or two
// frames per call the stage ring still has a next tile to prefetch and the transfer-kernel tile of the next unit is
// loaded while the inverse transform of this one runs (a single-frame call otherwise exposes a full memory latency
// per CTA).
template <int P, typename T, bool TILE0, int TPC = 1, bool PRUNED = false>
__device__ __forceinline__ void k2_frames(const cplx<T>* __restrict__ bands, const RowBands& rb, cplx<T>* __restrict__ spec,
                                          const cplx<T>* __restrict__ kp, const cplx<T>* __restrict__ kn, const cplx<T>* tw,
                                          const T* wy, cplx<T>* stage0, bool valid_in, bool special_in, int a, int tile,
                                          int c, int n1, int slot, int lt, int f_begin, int f_end, const ApplyGeom& g) {
  using TL = Tile<P>;
  static_assert(TPC == 1 || TL::SLOTS == 1, "several tiles per CTA need one slot per CTA");
  const bool valid = TL::SLOTS == 1 ? true : valid_in;      // one slot per CTA: the grid is exact
  constexpr int N1 = TL::N1, N2 = TL::N2, HALF = TL::HALF, C = TL::C;
  constexpr int STAGE = TL::SLOTS * P * C;                  // complex elements per stage
  constexpr int CH = 16 / (int)sizeof(cplx<T>);             // complex elements per 16-byte chunk
  constexpr int ROW_CHUNKS = C / CH;
  constexpr int PER_THREAD = (P * ROW_CHUNKS) / TL::SLOT_THREADS;
  constexpr int ROWS_PER_PASS = TL::SLOT_THREADS / ROW_CHUNKS;
  static_assert(C % CH == 0 && (P * ROW_CHUNKS) % TL::SLOT_THREADS == 0, "tile does not split into 16-byte chunks");
  constexpr bool PREFETCH = sizeof(cplx<T>) * N2 <= 128;

  // the transfer-kernel tile is loaded once and reused for every frame this CTA walks
  cplx<T> kv[PREFETCH ? N2 : 1];
  if constexpr (PREFETCH) {
    static_for<0, N2>([&](auto ee) {
      constexpr int e = decltype(ee)::value;
      kv[e] = valid ? kp[(long long)e * (N1 * C)] : mk<T>(T(0), T(0));
    });
  }
  const cplx<T>* kpu = kp;                                  // the transfer-kernel tile of the current unit
  auto kval = [&](auto ee) -> cplx<T> {
    constexpr int e = decltype(ee)::value;
    if constexpr (PREFETCH) return kv[e];
    else return valid ? kpu[(long long)e * (N1 * C)] : mk<T>(T(0), T(0));
  };
  auto sync = []() { __syncthreads(); };
  auto nosync = []() {};

  // cp.async addressing, hoisted: chunk i of this thread is row (lt / ROW_CHUNKS) + i*ROWS_PER_PASS
  const long long frame_stride = (long long)g.n_active * P * HALF;
  const long long band_frame_stride = (long long)rb.frame_rows * HALF;
  cplx<T>* tile_base0 = spec + ((long long)a * P) * HALF + tile * C;            // frame 0, first tile of this CTA
  const int row0 = lt / ROW_CHUNKS, part = lt % ROW_CHUNKS;
  const int live_rows = (g.win_len + 1) & ~1;               // PRUNED: rows the overlap-add reads
  const cplx<T>* src0 =
      bands + ((long long)(valid ? rb.patch_row[a] : 0) + row0) * HALF + tile * C + part * CH;   // the patch's band rows
  const int dst0 = slot * (P * C) + row0 * C + part * CH;
  const int nf = f_end - f_begin;
  const int n_it = TPC * nf;                                // iteration it = unit (it / nf), frame f_begin + it % nf
  auto issue = [&](int it, cplx<T>* stage) {
    if (valid) {
      const int u = TPC == 1 ? 0 : it / nf;
      const int f = f_begin + (TPC == 1 ? it : it - u * nf);
      const cplx<T>* src = src0 + u * C + f * band_frame_stride;
#pragma unroll
      for (int i = 0; i < PER_THREAD; ++i) {
        if (!PRUNED || row0 + i * ROWS_PER_PASS < live_rows)
          cp_async16(stage + dst0 + i * (ROWS_PER_PASS * C), src + (long long)i * (ROWS_PER_PASS * HALF));
        else      // a row past the window: zeros, straight into the stage (visible after the barrier that follows the wait)
          *reinterpret_cast<int4*>(stage + dst0 + i * (ROWS_PER_PASS * C)) = make_int4(0, 0, 0, 0);
      }
    }
    cp_async_commit();
  };
  auto ex = [=](int k2, int nn) { return ((slot * N2 + k2) * N1 + nn) * C + c; };

  // One commit group per tile slot, empty past the end, so "at most NS-2 groups pending" always
  // means "tile f has landed".
  constexpr int NS = K2_STAGES;
  static_assert(NS >= 2 && NS <= 4, "2..4 tile stages");
  int cur = 0;
  grid_dependency_wait();         // the transfer-kernel tile above is already in flight; the spectrum is K1's
  grid_launch_dependents();
#pragma unroll
  for (int s = 0; s < NS - 1; ++s) {
    if (s < n_it) issue(s, stage0 + s * STAGE);
    else cp_async_commit();
  }
  for (int it = 0; it < n_it; ++it, cur = (cur + 1 == NS ? 0 : cur + 1)) {
    const int u = TPC == 1 ? 0 : it / nf;
    const int f = f_begin + (TPC == 1 ? it : it - u * nf);
    const bool special = special_in && (TPC == 1 || u == 0);
    cplx<T>* tile_base = tile_base0 + u * C;
    cplx<T>* xbuf = stage0 + cur * STAGE;
    cp_async_wait_pending<NS - 2>();
    __syncthreads();          // tile `it` landed for everyone; everyone is done with the stage refilled next
    {
      const int nxt = cur + NS - 1 >= NS ? cur - 1 : cur + NS - 1;
      if (it + NS - 1 < n_it) issue(it + NS - 1, stage0 + nxt * STAGE);
      else cp_async_commit();
    }
    cplx<T> v[N2];
    static_for<0, N2>([&](auto jj) {
      constexpr int j = decltype(jj)::value;
      // row n1 + N1*j, column c (the slot pass A writes back to), times the row window
      v[j] = cscale_rn(xbuf[ex(j, n1)], wy[n1 + N1 * j]);
    });

    // The exchange slots a thread reads in the forward pass B are exactly the ones it writes in the
    // inverse pass B, so no barrier is needed between the two unless the buffer is reused in
    // between (the DC/Nyquist column of tile 0 does that).
    if constexpr (TILE0) coop_fft_forward<P, T>(v, n1, xbuf, tw, ex, sync);
    else coop_fft_forward<P, T>(v, n1, xbuf, tw, ex, sync, nosync);

    if constexpr (TILE0) {
      cplx<T>* zs = xbuf + slot * P;                        // natural order, one column per slot
      if (special) {
        static_for<0, N2>([&](auto ee) {
          constexpr int e = decltype(ee)::value;
          constexpr int m = e / N1, k1 = e % N1;
          zs[(n1 + N1 * m) + N2 * k1] = v[e];
        });
      }
      __syncthreads();
      static_for<0, N2>([&](auto ee) {
        constexpr int e = decltype(ee)::value;
        constexpr int m = e / N1, k1 = e % N1;
        const int k = (n1 + N1 * m) + N2 * k1;
        cplx<T> zm = v[e], kny = mk<T>(T(0), T(0));
        if (special) {
          const cplx<T> zr = zs[(P - k) & (P - 1)];
          zm = mk<T>(zr.x, -zr.y);
          kny = kn[e * N1];
        }
        const cplx<T> sum = mk<T>(T(0.5) * (v[e].x + zm.x), T(0.5) * (v[e].y + zm.y));
        const cplx<T> dif = mk<T>(T(0.5) * (v[e].x - zm.x), T(0.5) * (v[e].y - zm.y));
        v[e] = cadd(cmul(sum, kval(ee)), cmul(dif, kny));
      });
      __syncthreads();
    } else {
      static_for<0, N2>([&](auto ee) { v[decltype(ee)::value] = cmul(v[decltype(ee)::value], kval(ee)); });
    }

    if constexpr (TPC > 1) {
      // last frame of this unit: the next unit's transfer-kernel tile travels while the inverse transform runs
      if (f + 1 == f_end && u + 1 < TPC) {
        kpu += (long long)N2 * (N1 * C);
        if constexpr (PREFETCH) {
          static_for<0, N2>([&](auto ee) {
            constexpr int e = decltype(ee)::value;
            kv[e] = valid ? kpu[(long long)e * (N1 * C)] : mk<T>(T(0), T(0));
          });
        }
      }
    }
    // no trailing barrier: the next iteration's top barrier orders these exchange reads
    // before anything is copied into this stage again
    coop_fft_inverse<P, T>(v, n1, xbuf, tw, ex, sync, nosync);
    if (valid) {
      cplx<T>* base = tile_base + f * frame_stride + c;
      static_for<0, N2>([&](auto jj) {
        constexpr int j = decltype(jj)::value;
        if (!PRUNED || n1 + N1 * j < live_rows) base[(long long)(n1 + N1 * j) * HALF] = v[j];
      });
    }
  }
}

// Two CTAs per SM keep the transfer-kernel tile in registers; three (78 registers, the tile re-read from L2) were
// measured slower (35.3 vs 32.2 us per frame).
template <int P, typename T, int TPC = 1, bool PRUNED = false>
__global__ void __launch_bounds__(Tile<P>::K2_THREADS, 2)
k2_pipelined(const cplx<T>* __restrict__ bands, const RowBands rb, cplx<T>* __restrict__ spec,
             const cplx<T>* __restrict__ kmain, const cplx<T>* __restrict__ knyq, const int* __restrict__ active,
             const cplx<T>* __restrict__ tw_g, const T* __restrict__ win_g, int batch, int frames_per_cta, ApplyGeom g) {
  using TL = Tile<P>;
  constexpr int N1 = TL::N1, N2 = TL::N2, C = TL::C, NTILE = TL::NTILE;
  static_assert(TPC == 1 || (TL::SLOTS == 1 && NTILE % TPC == 0), "tiles per CTA must divide the tiles of a patch");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  T* wy = reinterpret_cast<T*>(tw + P);                     // row window as the row pass applied it: 0.5 * win
  cplx<T>* stage0 = reinterpret_cast<cplx<T>*>(wy + P);
  for (int i = threadIdx.x; i < P; i += blockDim.x) { tw[i] = tw_g[i]; wy[i] = T(0.5) * win_g[i]; }

  const int c = threadIdx.x % C;
  const int n1 = (threadIdx.x / C) % N1;
  const int slot = threadIdx.x / (C * N1);
  const int lt = threadIdx.x % TL::SLOT_THREADS;
  const long long first = (long long)blockIdx.x * TL::SLOTS * TPC;
  const long long sitem = first + slot;
  const long long total = (long long)g.n_active * NTILE;
  const bool valid = sitem < total;                          // with one slot per CTA the grid is exact: always true
  const int a = valid ? int(sitem / NTILE) : 0;
  const int tile = valid ? int(sitem % NTILE) : 1;
  bool any_tile0 = false;
#pragma unroll
  for (int s = 0; s < TL::SLOTS; ++s) any_tile0 |= (first + s < total) && ((first + s) % NTILE == 0);
  if constexpr (TL::SLOTS == 1) { if (!valid) return; }
  const bool special = valid && tile == 0 && c == 0;
  const int gp = valid ? active[a] : 0;
  const cplx<T>* kp = kmain + (((long long)gp * NTILE + (valid ? tile : 0)) * N2) * (N1 * C) + n1 * C + c;
  const cplx<T>* kn = knyq + (long long)gp * P + n1;
  const int f_begin = blockIdx.y * frames_per_cta;
  const int f_end = min(batch, f_begin + frames_per_cta);
  if (any_tile0)
    k2_frames<P, T, true, TPC, PRUNED>(bands, rb, spec, kp, kn, tw, wy, stage0, valid, special, a, tile, c, n1, slot, lt,
                                       f_begin, f_end, g);
  else
    k2_frames<P, T, false, TPC, PRUNED>(bands, rb, spec, kp, kn, tw, wy, stage0, valid, special, a, tile, c, n1, slot, lt,
                                        f_begin, f_end, g);
}

// ---------------------------------------------------------------------------- K2 of a transform stack
// k2_pipelined's frame loop for M transfer kernels: per frame, the tile streams in through the same cp.async stage
// ring and the forward column FFT runs once; then, per kernel m, the multiply by kernel m's tile and the inverse FFT,
// stored to spectrum slot (m, f) at spec + m * kspec_stride.  The forward spectrum stays in registers (vf, and for the
// tile-0 instantiation zm, the conjugate mirror of the packed DC/Nyquist column) across the M inverse transforms.
// Kernel m's tile is re-read from L2 per frame (M tiles do not fit the registers).  The arithmetic of every element is
// k2_frames' (same device functions, same operand order), so each slot equals what k2_pipelined writes for kernel m.
template <int P, typename T, bool TILE0>
__device__ __forceinline__ void k2_stack_frames(const cplx<T>* __restrict__ bands, const RowBands& rb, cplx<T>* __restrict__ spec,
                                                long long kspec_stride, const cplx<T>* __restrict__ kp,
                                                long long kmain_stride, const cplx<T>* __restrict__ kn, long long knyq_stride,
                                                int n_kernels, const cplx<T>* tw, const T* wy, cplx<T>* stage0, bool valid_in,
                                                bool special, int a, int tile, int c, int n1, int slot, int lt, int f_begin,
                                                int f_end, const ApplyGeom& g) {
  using TL = Tile<P>;
  const bool valid = TL::SLOTS == 1 ? true : valid_in;
  constexpr int N1 = TL::N1, N2 = TL::N2, HALF = TL::HALF, C = TL::C;
  constexpr int STAGE = TL::SLOTS * P * C;
  constexpr int CH = 16 / (int)sizeof(cplx<T>);
  constexpr int ROW_CHUNKS = C / CH;
  constexpr int PER_THREAD = (P * ROW_CHUNKS) / TL::SLOT_THREADS;
  constexpr int ROWS_PER_PASS = TL::SLOT_THREADS / ROW_CHUNKS;
  static_assert(C % CH == 0 && (P * ROW_CHUNKS) % TL::SLOT_THREADS == 0, "tile does not split into 16-byte chunks");
  auto sync = []() { __syncthreads(); };
  auto nosync = []() {};

  const long long frame_stride = (long long)g.n_active * P * HALF;
  const long long band_frame_stride = (long long)rb.frame_rows * HALF;
  cplx<T>* tile_base = spec + ((long long)a * P) * HALF + tile * C;
  const int row0 = lt / ROW_CHUNKS, part = lt % ROW_CHUNKS;
  const cplx<T>* src0 = bands + ((long long)(valid ? rb.patch_row[a] : 0) + row0) * HALF + tile * C + part * CH;
  const int dst0 = slot * (P * C) + row0 * C + part * CH;
  const int n_it = f_end - f_begin;
  auto issue = [&](int it, cplx<T>* stage) {
    if (valid) {
      const cplx<T>* src = src0 + (f_begin + it) * band_frame_stride;
#pragma unroll
      for (int i = 0; i < PER_THREAD; ++i)
        cp_async16(stage + dst0 + i * (ROWS_PER_PASS * C), src + (long long)i * (ROWS_PER_PASS * HALF));
    }
    cp_async_commit();
  };
  auto ex = [=](int k2, int nn) { return ((slot * N2 + k2) * N1 + nn) * C + c; };

  constexpr int NS = K2_STAGES;
  int cur = 0;
  grid_dependency_wait();
  grid_launch_dependents();
#pragma unroll
  for (int s = 0; s < NS - 1; ++s) {
    if (s < n_it) issue(s, stage0 + s * STAGE);
    else cp_async_commit();
  }
  for (int it = 0; it < n_it; ++it, cur = (cur + 1 == NS ? 0 : cur + 1)) {
    const int f = f_begin + it;
    cplx<T>* xbuf = stage0 + cur * STAGE;
    cp_async_wait_pending<NS - 2>();
    __syncthreads();
    {
      const int nxt = cur + NS - 1 >= NS ? cur - 1 : cur + NS - 1;
      if (it + NS - 1 < n_it) issue(it + NS - 1, stage0 + nxt * STAGE);
      else cp_async_commit();
    }
    cplx<T> vf[N2];
    static_for<0, N2>([&](auto jj) {
      constexpr int j = decltype(jj)::value;
      vf[j] = cscale_rn(xbuf[ex(j, n1)], wy[n1 + N1 * j]);
    });
    coop_fft_forward<P, T>(vf, n1, xbuf, tw, ex, sync);
    cplx<T> zm[TILE0 ? N2 : 1];
    if constexpr (TILE0) {
      cplx<T>* zs = xbuf + slot * P;
      if (special) {
        static_for<0, N2>([&](auto ee) {
          constexpr int e = decltype(ee)::value;
          constexpr int m = e / N1, k1 = e % N1;
          zs[(n1 + N1 * m) + N2 * k1] = vf[e];
        });
      }
      __syncthreads();
      static_for<0, N2>([&](auto ee) {
        constexpr int e = decltype(ee)::value;
        constexpr int m = e / N1, k1 = e % N1;
        const int k = (n1 + N1 * m) + N2 * k1;
        zm[e] = vf[e];
        if (special) {
          const cplx<T> zr = zs[(P - k) & (P - 1)];
          zm[e] = mk<T>(zr.x, -zr.y);
        }
      });
      __syncthreads();                                      // zs is read: the inverse transforms may reuse the buffer
    }
    for (int km = 0; km < n_kernels; ++km) {
      const cplx<T>* kpm = kp + km * kmain_stride;
      cplx<T> v[N2];
      if constexpr (TILE0) {
        const cplx<T>* knm = kn + km * knyq_stride;
        static_for<0, N2>([&](auto ee) {
          constexpr int e = decltype(ee)::value;
          const cplx<T> kval = valid ? kpm[(long long)e * (N1 * C)] : mk<T>(T(0), T(0));
          const cplx<T> kny = special ? knm[e * N1] : mk<T>(T(0), T(0));
          const cplx<T> sum = mk<T>(T(0.5) * (vf[e].x + zm[e].x), T(0.5) * (vf[e].y + zm[e].y));
          const cplx<T> dif = mk<T>(T(0.5) * (vf[e].x - zm[e].x), T(0.5) * (vf[e].y - zm[e].y));
          v[e] = cadd(cmul(sum, kval), cmul(dif, kny));
        });
      } else {
        static_for<0, N2>([&](auto ee) {
          constexpr int e = decltype(ee)::value;
          v[e] = cmul(vf[e], valid ? kpm[(long long)e * (N1 * C)] : mk<T>(T(0), T(0)));
        });
      }
      // the exchange slots of one inverse transform are read before the next writes them (`sync` after the reads);
      // after the last one, the next frame's top barrier orders them before the stage is refilled
      if (km + 1 < n_kernels) coop_fft_inverse<P, T>(v, n1, xbuf, tw, ex, sync, sync);
      else coop_fft_inverse<P, T>(v, n1, xbuf, tw, ex, sync, nosync);
      if (valid) {
        cplx<T>* base = tile_base + km * kspec_stride + f * frame_stride + c;
        static_for<0, N2>([&](auto jj) {
          constexpr int j = decltype(jj)::value;
          base[(long long)(n1 + N1 * j) * HALF] = v[j];
        });
      }
    }
  }
}

template <int P, typename T>
__global__ void __launch_bounds__(Tile<P>::K2_THREADS, 2)
k2_stack(const cplx<T>* __restrict__ bands, const RowBands rb, cplx<T>* __restrict__ spec, long long kspec_stride,
         const cplx<T>* __restrict__ kmain, long long kmain_stride, const cplx<T>* __restrict__ knyq, long long knyq_stride,
         int n_kernels, const int* __restrict__ active, const cplx<T>* __restrict__ tw_g, const T* __restrict__ win_g,
         int batch, int frames_per_cta, ApplyGeom g) {
  using TL = Tile<P>;
  constexpr int N1 = TL::N1, N2 = TL::N2, C = TL::C, NTILE = TL::NTILE;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  T* wy = reinterpret_cast<T*>(tw + P);
  cplx<T>* stage0 = reinterpret_cast<cplx<T>*>(wy + P);
  for (int i = threadIdx.x; i < P; i += blockDim.x) { tw[i] = tw_g[i]; wy[i] = T(0.5) * win_g[i]; }

  const int c = threadIdx.x % C;
  const int n1 = (threadIdx.x / C) % N1;
  const int slot = threadIdx.x / (C * N1);
  const int lt = threadIdx.x % TL::SLOT_THREADS;
  const long long first = (long long)blockIdx.x * TL::SLOTS;
  const long long sitem = first + slot;
  const long long total = (long long)g.n_active * NTILE;
  const bool valid = sitem < total;
  const int a = valid ? int(sitem / NTILE) : 0;
  const int tile = valid ? int(sitem % NTILE) : 1;
  bool any_tile0 = false;
#pragma unroll
  for (int s = 0; s < TL::SLOTS; ++s) any_tile0 |= (first + s < total) && ((first + s) % NTILE == 0);
  if constexpr (TL::SLOTS == 1) { if (!valid) return; }
  const bool special = valid && tile == 0 && c == 0;
  const int gp = valid ? active[a] : 0;
  const cplx<T>* kp = kmain + (((long long)gp * NTILE + (valid ? tile : 0)) * N2) * (N1 * C) + n1 * C + c;
  const cplx<T>* kn = knyq + (long long)gp * P + n1;
  const int f_begin = blockIdx.y * frames_per_cta;
  const int f_end = min(batch, f_begin + frames_per_cta);
  if (any_tile0)
    k2_stack_frames<P, T, true>(bands, rb, spec, kspec_stride, kp, kmain_stride, kn, knyq_stride, n_kernels, tw, wy, stage0,
                                valid, special, a, tile, c, n1, slot, lt, f_begin, f_end, g);
  else
    k2_stack_frames<P, T, false>(bands, rb, spec, kspec_stride, kp, kmain_stride, kn, knyq_stride, n_kernels, tw, wy, stage0,
                                 valid, special, a, tile, c, n1, slot, lt, f_begin, f_end, g);
}

// ============================================================================ K3
// row IFFT + window + overlap-add.  transform.py:164-177 (second IFFT axis, np.real, window,
// `+=` into the canvas, crop).  Launched once per colour class: patches of one colour never
// overlap, so plain read-modify-write is race-free and the per-pixel summation order is the
// colour order — for calculate_covering inputs that is the reference's own order.
template <int P, typename T>
__global__ void __launch_bounds__(Tile<P>::ROW_THREADS)
k3_rowifft_window_overlap_add(const cplx<T>* __restrict__ spec, T* __restrict__ out,
                              const int2* __restrict__ corners, const int* __restrict__ items, int n_items,
                              const cplx<T>* __restrict__ tw_g, const T* __restrict__ win_g, int store_only,
                              ApplyGeom g) {
  using TL = Tile<P>;
  constexpr int N1 = TL::N1, N2 = TL::N2, HALF = TL::HALF;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  T* win = reinterpret_cast<T*>(tw + P);
  cplx<T>* scratch_all = reinterpret_cast<cplx<T>*>(win + P);
  for (int i = threadIdx.x; i < P; i += blockDim.x) { tw[i] = tw_g[i]; win[i] = win_g[i]; }
  __syncthreads();

  const int team = threadIdx.x / N1, t = threadIdx.x % N1;
  cplx<T>* scr = scratch_all + team * TL::SCR;
  const int idx = blockIdx.x * TL::TEAMS + team;
  if (idx >= n_items) return;
  const int item = items[idx];
  const int a = item / HALF, pair = item % HALF;
  const unsigned mask = team_mask(N1);
  auto ex = [](int k2, int n1) { return k2 * TL::EX_STRIDE + n1; };
  auto sync = [mask]() { __syncwarp(mask); };

  const int2 corner = corners[a];
  const int ra = 2 * pair, rb = ra + 1;
  const cplx<T>* ua = spec + (((long long)blockIdx.y * g.n_active + a) * P + ra) * HALF;
  const cplx<T>* ub = ua + HALF;

  // Z[k] = Ua[k] + i*Ub[k] for k <= P/2, Hermitian mirror above; bin 0 unpacks (DC, Nyquist).
  cplx<T> v[N2];
  static_for<0, N2>([&](auto ee) {
    constexpr int e = decltype(ee)::value;
    constexpr int m = e / N1, k1 = e % N1;
    const int k = (t + N1 * m) + N2 * k1;
    const int src = k <= HALF ? k : P - k;
    const cplx<T> pa = ua[src == HALF ? 0 : src];
    const cplx<T> pb = ub[src == HALF ? 0 : src];
    cplx<T> z;
    if (k == 0)           z = mk<T>(pa.x, pb.x);
    else if (k == HALF)   z = mk<T>(pa.y, pb.y);
    else if (k < HALF)    z = mk<T>(pa.x - pb.y, pa.y + pb.x);
    else                  z = mk<T>(pa.x + pb.y, pb.x - pa.y);
    v[e] = z;
  });

  coop_fft_inverse<P, T>(v, t, scr, tw, ex, sync);

  const int ya = corner.x + ra, yb = corner.x + rb;
  const bool oka = ya >= g.row_begin && ya < g.row_end;
  const bool okb = yb >= g.row_begin && yb < g.row_end;
  T* frame = out + (long long)blockIdx.y * g.out_frame_stride;
  T* oa = frame + (long long)(ya - g.out_row0) * g.out_pitch;
  T* ob = frame + (long long)(yb - g.out_row0) * g.out_pitch;
  const T wa = win[ra], wb = win[rb];
  static_for<0, N2>([&](auto jj) {
    constexpr int j = decltype(jj)::value;
    const int n = t + N1 * j;
    const int x = corner.y + n;
    if (x >= 0 && x < g.W && n < g.win_len) {
      const T w = win[n];
      if (oka && ra < g.win_len) { const T val = v[j].x * w * wa; oa[x] = store_only ? val : oa[x] + val; }
      if (okb && rb < g.win_len) { const T val = v[j].y * w * wb; ob[x] = store_only ? val : ob[x] + val; }
    }
  });
}

// ============================================================================ K3 (row-pair gather)
// Same arithmetic as the colour-phase kernel above, restructured so that no output pixel is
// ever read back from HBM.  A CTA owns one pair of output rows (x one column segment).  The
// (patch, row pair) items that land on it are grouped by patch corner column.  The items of a
// group cover the same columns and differ only in their row windows, and the inverse FFT is
// linear — so a team sums the group's half-spectra first, each scaled by its row windows
// (wa*Ua + i*wb*Ub, accumulated in colour order), and runs ONE inverse FFT for the group: for a
// calculate_covering grid that halves the row IFFTs (34 items -> 17 groups per row pair).
// Groups are split into (at most two) layers of pairwise disjoint groups — the patches whose
// corner column is a multiple of P, and the half-offset ones.  Layer 0 then layer 1 add their
// rows into one zero-initialised shared-memory plane, a barrier apart, so the per-pixel order
// is fixed (bit-stable, slab-sharded runs stitch bit-identically); the two rows are stored with
// coalesced 16-byte writes.
// A team's inputs arrive by cp.async into its 2-row buffer, which then serves as the exchange
// scratch of its inverse FFT.  Needs every patch corner row to share one parity (patch row
// pairs line up with output row pairs) and at most two layers; the planner falls back to the
// colour-phase kernel otherwise.
struct RowTile { int group_begin, group_count, y, x0; };              // output rows y, y+1; columns [x0, x0+seg)
struct RowGroup { int item_begin, item_count, cx, layer, clipped; };  // items: active*HALF + pair, colour order
constexpr int K3G_SMEM_MAX = 200 * 1024;                              // dynamic shared memory the kernel may ask for

template <int P, typename T>
__global__ void __launch_bounds__(288, 3)
k3_rowpair_gather(const cplx<T>* __restrict__ spec, T* __restrict__ out, const RowTile* __restrict__ tiles,
                  const RowGroup* __restrict__ groups, const int* __restrict__ items,
                  const cplx<T>* __restrict__ tw_g, const T* __restrict__ win_g, int seg_w, ApplyGeom g) {
  using TL = Tile<P>;
  constexpr int N1 = TL::N1, N2 = TL::N2, HALF = TL::HALF;
  constexpr int BUF = TL::SCR > P ? TL::SCR : P;             // complex elements per team buffer (>= 2 spectrum rows)
  constexpr int CH = 16 / (int)sizeof(cplx<T>);
  constexpr int V = 16 / (int)sizeof(T);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  T* win = reinterpret_cast<T*>(tw + P);
  T* plane = win + P;                                        // [row 2][seg_w]
  cplx<T>* bufs = reinterpret_cast<cplx<T>*>(plane + 2 * seg_w);   // [team][BUF]
  for (int i = threadIdx.x; i < P; i += blockDim.x) { tw[i] = tw_g[i]; win[i] = win_g[i]; }
  for (int i = threadIdx.x * V; i < 2 * seg_w; i += blockDim.x * V) {
    if constexpr (sizeof(T) == 4) *reinterpret_cast<float4*>(plane + i) = make_float4(0.f, 0.f, 0.f, 0.f);
    else *reinterpret_cast<double2*>(plane + i) = make_double2(0.0, 0.0);
  }

  const RowTile tile = tiles[blockIdx.x];
  const int teams = blockDim.x / N1;
  const int team = threadIdx.x / N1, t = threadIdx.x % N1;
  const unsigned mask = team_mask(N1);
  auto ex = [](int k2, int n1) { return k2 * TL::EX_STRIDE + n1; };
  auto sync = [mask]() { __syncwarp(mask); };
  const int x_end = min(tile.x0 + seg_w, g.W);
  cplx<T>* buf = bufs + (long long)team * BUF;
  __syncthreads();                                           // tables and the zeroed plane visible

  for (int base = 0; base < tile.group_count; base += teams) {
    const int gi = base + team;
    const bool live = gi < tile.group_count;
    RowGroup grp;
    grp.item_begin = 0; grp.item_count = 0; grp.cx = 0; grp.layer = -1; grp.clipped = 0;
    cplx<T> v[N2];
    if (live) {
      grp = groups[tile.group_begin + gi];
      static_for<0, N2>([&](auto ee) { v[decltype(ee)::value] = mk<T>(T(0), T(0)); });
      for (int it = 0; it < grp.item_count; ++it) {
        const int item = items[grp.item_begin + it];
        const int a = item / HALF, ra = 2 * (item % HALF);
        const cplx<T>* src = spec + (((long long)blockIdx.y * g.n_active + a) * P + ra) * HALF;
#pragma unroll
        for (int q = t; q < P / CH; q += N1) cp_async16(buf + q * CH, src + q * CH);
        cp_async_commit();
        const cplx<T> wa = mk<T>(win[ra], win[ra]), wb = mk<T>(win[ra + 1], win[ra + 1]);
        cp_async_wait_all();
        sync();
        const cplx<T>* ua = buf;
        const cplx<T>* ub = buf + HALF;
        // Z[k] += wa*Ua[k] + i*wb*Ub[k] for k <= P/2, Hermitian mirror above; bin 0 unpacks (DC, Nyquist)
        static_for<0, N2>([&](auto ee) {
          constexpr int e = decltype(ee)::value;
          constexpr int m = e / N1, k1 = e % N1;
          const int k = (t + N1 * m) + N2 * k1;
          const int srck = k <= HALF ? k : P - k;
          const cplx<T> pa = ua[srck == HALF ? 0 : srck];
          const cplx<T> pb = ub[srck == HALF ? 0 : srck];
          cplx<T> a2 = k > HALF ? mk<T>(pa.x, -pa.y) : pa;
          cplx<T> b2 = k > HALF ? mk<T>(pb.y, pb.x) : mk<T>(-pb.y, pb.x);
          if (k == 0)    { a2 = mk<T>(pa.x, T(0)); b2 = mk<T>(T(0), pb.x); }
          if (k == HALF) { a2 = mk<T>(pa.y, T(0)); b2 = mk<T>(T(0), pb.y); }
          v[e] = pfma(b2, wb, pfma(a2, wa, v[e]));
        });
        sync();                                              // whole team has read the rows: buffer is free again
      }
      coop_fft_inverse<P, T>(v, t, buf, tw, ex, sync, sync);
      static_for<0, N2>([&](auto jj) {
        constexpr int j = decltype(jj)::value;
        v[j] = cscale(v[j], win[t + N1 * j]);
      });
    }
#pragma unroll
    for (int layer = 0; layer < 2; ++layer) {
      if (live && grp.layer == layer) {
        if (!grp.clipped) {
          static_for<0, N2>([&](auto jj) {
            constexpr int j = decltype(jj)::value;
            const int x = grp.cx + t + N1 * j - tile.x0;
            plane[x] += v[j].x;
            plane[seg_w + x] += v[j].y;
          });
        } else {
          static_for<0, N2>([&](auto jj) {
            constexpr int j = decltype(jj)::value;
            const int x = grp.cx + t + N1 * j;
            if (x >= tile.x0 && x < x_end) {
              plane[x - tile.x0] += v[j].x;
              plane[seg_w + x - tile.x0] += v[j].y;
            }
          });
        }
      }
      __syncthreads();
    }
  }
  T* frame = out + (long long)blockIdx.y * g.out_frame_stride;
  const int len = x_end - tile.x0;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int y = tile.y + r;
    if (y < g.row_begin || y >= g.row_end) continue;
    T* dst = frame + (long long)(y - g.out_row0) * g.out_pitch + tile.x0;
    const T* p0 = plane + r * seg_w;
    if ((reinterpret_cast<size_t>(dst) & 15) == 0) {
      for (int i = threadIdx.x * V; i + V <= len; i += blockDim.x * V) {
        if constexpr (sizeof(T) == 4) *reinterpret_cast<float4*>(dst + i) = *reinterpret_cast<const float4*>(p0 + i);
        else *reinterpret_cast<double2*>(dst + i) = *reinterpret_cast<const double2*>(p0 + i);
      }
      for (int i = (len / V) * V + threadIdx.x; i < len; i += blockDim.x) dst[i] = p0[i];
    } else {
      for (int i = threadIdx.x; i < len; i += blockDim.x) dst[i] = p0[i];
    }
  }
}

// ============================================================================ kernel prep
// Reference-layout cube K[n][r][c] (complex TK, full unshifted spectrum) -> private layout.
//   Kh[r][c] = (K[r][c] + conj K[-r][-c]) / (2 P^2),  c in [0, P/2]
//   kmain[((n*NTILE + tile)*N2 + e)*(N1*C) + n1*C + cc] = Kh[(n1 + N1*m) + N2*k1][tile*C + cc],  e = m*N1 + k1
//   knyq [n*P + e*N1 + n1]                              = Kh[(n1 + N1*m) + N2*k1][P/2]
template <int P, typename T, typename TK>
__global__ void prep_transfer_kernel(const TK* __restrict__ full, cplx<T>* __restrict__ kmain,
                                     cplx<T>* __restrict__ knyq, int n_patches) {
  using TL = Tile<P>;
  constexpr int N1 = TL::N1, N2 = TL::N2, HALF = TL::HALF, C = TL::C, NTILE = TL::NTILE;
  const long long per_patch = (long long)P * HALF;
  const long long total = (long long)n_patches * (per_patch + P);
  const double scale = 0.5 / (double(P) * double(P));
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const bool nyq = i >= (long long)n_patches * per_patch;
    int n, k, col; long long dst;
    if (!nyq) {
      long long r = i;
      const int cc = int(r % C); r /= C;
      const int n1 = int(r % N1); r /= N1;
      const int e = int(r % N2); r /= N2;
      const int tile = int(r % NTILE); r /= NTILE;
      n = int(r);
      k = (n1 + N1 * (e / N1)) + N2 * (e % N1);
      col = tile * C + cc;
      dst = i;
    } else {
      long long r = i - (long long)n_patches * per_patch;
      const int n1 = int(r % N1); r /= N1;
      const int e = int(r % N2); r /= N2;
      n = int(r);
      k = (n1 + N1 * (e / N1)) + N2 * (e % N1);
      col = HALF;
      dst = i - (long long)n_patches * per_patch;
    }
    const TK p = full[((long long)n * P + k) * P + col];
    const TK q = full[((long long)n * P + ((P - k) & (P - 1))) * P + ((P - col) & (P - 1))];
    const cplx<T> val = mk<T>(T((double(p.x) + double(q.x)) * scale), T((double(p.y) - double(q.y)) * scale));
    if (nyq) knyq[dst] = val; else kmain[dst] = val;
  }
}

// ============================================================================ construct
// transform.py:78-82:  K = conj(S) |S|^(a-1) / (|S|^(a+1) + (eps |T|)^(a+1)) * T, in the cubes'
// dtype, IEEE-faithful (no zero guard: 0/0 -> NaN like the reference).  The small-exponent
// branches mirror numpy's scalar-power fast paths (x**0, x**0.5, x**1, x**2, x**-1) so the
// same bins take the same arithmetic; the division mirrors numpy's complex/real quotient.
template <typename T> __device__ __forceinline__ T pow_like_numpy(T x, T p) {
  if (p == T(0)) return T(1);
  if (p == T(1)) return x;
  if (p == T(2)) return x * x;
  if (p == T(0.5)) return sqrt(x);
  if (p == T(-1)) return T(1) / x;
  return pow(x, p);
}
// DEV: alpha and epsilon are read from two device doubles (`ae`), once per CTA, and converted to T as the host-scalar
// entry point converts its arguments, so the same bins take the same arithmetic (rpsf_construct_kernel_dev).
template <typename T, bool DEV = false>
__global__ void construct_transfer_kernel(const cplx<T>* __restrict__ S, const cplx<T>* __restrict__ Tg,
                                          cplx<T>* __restrict__ K, long long count, T alpha, T epsilon,
                                          const double* __restrict__ ae = nullptr) {
  if constexpr (DEV) {
    __shared__ T scalars[2];
    if (threadIdx.x == 0) { scalars[0] = T(ae[0]); scalars[1] = T(ae[1]); }
    __syncthreads();
    alpha = scalars[0];
    epsilon = scalars[1];
  }
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (long long)gridDim.x * blockDim.x) {
    const cplx<T> s = S[i], tg = Tg[i];
    const T sa = hypot(s.x, s.y), ta = hypot(tg.x, tg.y);
    const T pw = pow_like_numpy<T>(sa, alpha - T(1));
    const T nx = s.x * pw, ny = -s.y * pw;
    const T den = pow_like_numpy<T>(sa, alpha + T(1)) + pow_like_numpy<T>(epsilon * ta, alpha + T(1));
    T qx, qy;
    if (den == T(0)) { qx = nx / fabs(den); qy = ny / fabs(den); }
    else { const T scl = T(1) / den; qx = nx * scl; qy = ny * scl; }
    // explicit non-fused complex product, same operation order as numpy
    K[i] = mk<T>(qx * tg.x - qy * tg.y, qx * tg.y + qy * tg.x);
  }
}

// M kernels from one read of S and T: kernel m (m < n_kernels) goes to K + m * count, with (alpha, epsilon) =
// pairs[2m], pairs[2m + 1] converted to T as construct_transfer_kernel's entry points convert theirs.  The per-bin
// arithmetic is construct_transfer_kernel's, statement for statement, so every kernel is bit-identical to it.
// DEV: `pairs` is device memory (rpsf_construct_kernels_dev); otherwise the host pairs arrive in `host_pairs`.
constexpr int CONSTRUCT_BATCH = 64;     // kernels per launch: the host pairs travel as a 1 KB kernel parameter
struct ConstructPairs { double v[2 * CONSTRUCT_BATCH]; };
template <typename T, bool DEV = false>
__global__ void construct_transfer_kernels(const cplx<T>* __restrict__ S, const cplx<T>* __restrict__ Tg,
                                           cplx<T>* __restrict__ K, long long count, int n_kernels,
                                           ConstructPairs host_pairs, const double* __restrict__ pairs) {
  __shared__ T scalars[2 * CONSTRUCT_BATCH];
  for (int j = threadIdx.x; j < 2 * n_kernels; j += blockDim.x) scalars[j] = T(DEV ? pairs[j] : host_pairs.v[j]);
  __syncthreads();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count;
       i += (long long)gridDim.x * blockDim.x) {
    const cplx<T> s = S[i], tg = Tg[i];
    const T sa = hypot(s.x, s.y), ta = hypot(tg.x, tg.y);
    for (int m = 0; m < n_kernels; ++m) {
      const T alpha = scalars[2 * m], epsilon = scalars[2 * m + 1];
      const T pw = pow_like_numpy<T>(sa, alpha - T(1));
      const T nx = s.x * pw, ny = -s.y * pw;
      const T den = pow_like_numpy<T>(sa, alpha + T(1)) + pow_like_numpy<T>(epsilon * ta, alpha + T(1));
      T qx, qy;
      if (den == T(0)) { qx = nx / fabs(den); qy = ny / fabs(den); }
      else { const T scl = T(1) / den; qx = nx * scl; qy = ny * scl; }
      K[(long long)m * count + i] = mk<T>(qx * tg.x - qy * tg.y, qx * tg.y + qy * tg.x);
    }
  }
}

// ============================================================================ PSF FFT cube
// psf.py:216-219: fft2 over the last two axes, full spectrum, reference layout.
// rows: one team per row (real input promoted to complex); cols: K2-style tiles, in place.
template <int P, typename T, typename TIn>
__global__ void __launch_bounds__(Tile<P>::ROW_THREADS)
fft2_rows(const TIn* __restrict__ values, cplx<T>* __restrict__ out, const cplx<T>* __restrict__ tw_g,
          long long n_rows) {
  using TL = Tile<P>;
  constexpr int N1 = TL::N1, N2 = TL::N2;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  cplx<T>* scratch_all = tw + P;
  for (int i = threadIdx.x; i < P; i += blockDim.x) tw[i] = tw_g[i];
  __syncthreads();
  const int team = threadIdx.x / N1, t = threadIdx.x % N1;
  cplx<T>* scr = scratch_all + team * TL::SCR;
  const long long row = (long long)blockIdx.x * TL::TEAMS + team;
  if (row >= n_rows) return;
  const unsigned mask = team_mask(N1);
  auto ex = [](int k2, int n1) { return k2 * TL::EX_STRIDE + n1; };
  auto sync = [mask]() { __syncwarp(mask); };
  cplx<T> v[N2];
  static_for<0, N2>([&](auto jj) {
    constexpr int j = decltype(jj)::value;
    v[j] = mk<T>(T(values[row * P + t + N1 * j]), T(0));
  });
  coop_fft_forward<P, T>(v, t, scr, tw, ex, sync);
  static_for<0, N2>([&](auto ee) {
    constexpr int e = decltype(ee)::value;
    scr[(t + N1 * (e / N1)) + N2 * (e % N1)] = v[e];
  });
  sync();
#pragma unroll
  for (int i = 0; i < P / N1; ++i) out[row * P + t + N1 * i] = scr[t + N1 * i];
}

template <int P, typename T>
__global__ void __launch_bounds__(Tile<P>::K2_THREADS)
fft2_cols(cplx<T>* __restrict__ data, const cplx<T>* __restrict__ tw_g, long long n_patches) {
  using TL = Tile<P>;
  constexpr int N1 = TL::N1, N2 = TL::N2, C = TL::C;
  constexpr int NT = P / C;                                  // tiles across the full width
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  cplx<T>* xbuf = tw + P;
  for (int i = threadIdx.x; i < P; i += blockDim.x) tw[i] = tw_g[i];
  const int c = threadIdx.x % C;
  const int n1 = (threadIdx.x / C) % N1;
  const int slot = threadIdx.x / (C * N1);
  const long long sitem = (long long)blockIdx.x * TL::SLOTS + slot;
  const bool valid = sitem < n_patches * NT;
  const long long n = valid ? sitem / NT : 0;
  const int tile = valid ? int(sitem % NT) : 0;
  cplx<T>* base = data + n * P * P + tile * C + c;
  cplx<T> v[N2];
  static_for<0, N2>([&](auto jj) {
    constexpr int j = decltype(jj)::value;
    v[j] = valid ? base[(long long)(n1 + N1 * j) * P] : mk<T>(T(0), T(0));
  });
  __syncthreads();
  auto ex = [=](int k2, int nn) { return ((slot * N2 + k2) * N1 + nn) * C + c; };
  auto sync = []() { __syncthreads(); };
  coop_fft_forward<P, T>(v, n1, xbuf, tw, ex, sync);
  if (valid) {
    static_for<0, N2>([&](auto ee) {
      constexpr int e = decltype(ee)::value;
      base[(long long)((n1 + N1 * (e / N1)) + N2 * (e % N1)) * P] = v[e];
    });
  }
}

// ============================================================================ patch sizes without a native FFT length
// transform.py:163-164 for a P that is not a power of two in 16..512.  np.real(ifft2(fft2(x) * K)) is the circular
// convolution of the windowed patch x (P x P) with k = ifft2(K).  With M a power of two >= 2 P - 1, the same values
// come out of M-point transforms of the zero-padded patch and of k periodically extended over (-P, P)^2:
//     K'[u][v] = sum_{p,q} A[u][p] K[p][q] A[v][q],   A[u][p] = (1/P) sum_{i=-(P-1)}^{P-1} exp(2 pi i (p/P - u/M) i)
// (A is made on the host in double).  K' then goes through prep_transfer_kernel like any M x M cube, and apply()
// runs the M-point kernels with a window that ends at P.  Setup cost only: two small dense products per patch.
template <typename TK>
__global__ void embed_pass1(const TK* __restrict__ K, const double2* __restrict__ A, double2* __restrict__ T1,
                            int n_patches, int P, int M) {
  // T1[n][u][q] = sum_p A[u][p] K[n][p][q]
  const long long total = (long long)n_patches * M * P;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int q = int(i % P);
    const int u = int((i / P) % M);
    const long long n = i / ((long long)P * M);
    double re = 0.0, im = 0.0;
    for (int p = 0; p < P; ++p) {
      const double2 a = A[(long long)u * P + p];
      const TK k = K[(n * P + p) * P + q];
      re += a.x * double(k.x) - a.y * double(k.y);
      im += a.x * double(k.y) + a.y * double(k.x);
    }
    T1[i] = make_double2(re, im);
  }
}
template <typename TOut>      // (a template so that the header may be included by several translation units)
__global__ void embed_pass2(const double2* __restrict__ T1, const double2* __restrict__ A, TOut* __restrict__ Kp,
                            int n_patches, int P, int M) {
  // K'[n][u][v] = sum_q T1[n][u][q] A[v][q]
  const long long total = (long long)n_patches * M * M;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int v = int(i % M);
    const long long nu = i / M;
    double re = 0.0, im = 0.0;
    for (int q = 0; q < P; ++q) {
      const double2 a = A[(long long)v * P + q];
      const double2 t = T1[nu * P + q];
      re += t.x * a.x - t.y * a.y;
      im += t.x * a.y + t.y * a.x;
    }
    Kp[i].x = re; Kp[i].y = im;
  }
}
// psf.py:216-219 for such a P: separable direct DFT, out[n][k][l] = sum_{r,c} x[n][r][c] w^(k r + l c), w = exp(-2 pi i / P)
// (twiddle table tw[m] = w^m, m < P, made on the host in double; double accumulation; O(P^3) per patch, setup only).
template <typename TIn>
__global__ void dft_rows_direct(const TIn* __restrict__ x, const double2* __restrict__ tw, double2* __restrict__ tmp,
                                long long n_rows, int P) {
  const long long total = n_rows * P;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int l = int(i % P);
    const long long row = i / P;
    double re = 0.0, im = 0.0;
    int m = 0;
    for (int c = 0; c < P; ++c) {
      const double2 w = tw[m];
      const double v = double(x[row * P + c]);
      re += v * w.x; im += v * w.y;
      m += l; if (m >= P) m -= P;
    }
    tmp[i] = make_double2(re, im);
  }
}
template <typename TOut>
__global__ void dft_cols_direct(const double2* __restrict__ tmp, const double2* __restrict__ tw, TOut* __restrict__ out,
                                long long n_patches, int P) {
  const long long total = n_patches * P * P;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int l = int(i % P);
    const int k = int((i / P) % P);
    const long long n = i / ((long long)P * P);
    double re = 0.0, im = 0.0;
    int m = 0;
    for (int r = 0; r < P; ++r) {
      const double2 w = tw[m];
      const double2 t = tmp[(n * P + r) * P + l];
      re += t.x * w.x - t.y * w.y;
      im += t.x * w.y + t.y * w.x;
      m += k; if (m >= P) m -= P;
    }
    out[i].x = decltype(out[i].x)(re);
    out[i].y = decltype(out[i].y)(im);
  }
}

// ============================================================================ dtype conversion
template <typename TI, typename TO>
__global__ void convert_2d(const TI* __restrict__ src, long long src_pitch, TO* __restrict__ dst,
                           long long dst_pitch, int rows, int cols) {
  const long long total = (long long)rows * cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols, cidx = i % cols;
    dst[r * dst_pitch + cidx] = TO(src[r * src_pitch + cidx]);
  }
}

}  // namespace rpsf
