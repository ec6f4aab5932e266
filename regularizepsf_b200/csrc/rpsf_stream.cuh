// rpsf_stream.cuh — persistent, bulk-async (TMA 1-D) versions of the two row kernels.
//
// K1 (transform.py:141-163) and K3 (transform.py:164-177) each touch every row of every patch
// exactly once, so the kernels are streaming passes whose only enemies are memory latency and
// issue slots spent on address arithmetic.  Here a warp is a self-contained pipeline:
//
//   * one elected lane per row issues `cp.async.bulk.shared::cluster.global` copies (UBLKCP, the
//     1-D TMA path) that land whole patch rows in a ring of per-warp shared-memory stages and
//     signal an mbarrier with the byte count — no register staging, no per-element addresses;
//   * the warp's teams (N1 lanes each, see rpsf_fft.cuh) wait on the mbarrier of the oldest
//     stage, pull their samples out of shared memory with constant offsets, and reuse the very
//     same stage as the FFT exchange buffer;
//   * the grid is persistent (one CTA per SM), warps walk the item list with a fixed stride, and
//     the copy for item i+STAGES-1 is in flight while item i is transformed.
//
// Items the bulk path cannot serve (patches that hang over the frame edge in x, unaligned
// corners, `constant` padding rows) are gathered through pad_index() by the warp itself into
// the same stage and then take the same compute path.
#pragma once
#include <cstdint>
#include "rpsf_kernels.cuh"
#include "rpsf_bands.cuh"

namespace rpsf {

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  const unsigned addr = smem_u32(bar);
  unsigned done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}
// global -> shared bulk copy (bytes: multiple of 16, both addresses 16-byte aligned)
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// orders this thread's earlier generic-proxy shared-memory accesses before later async-proxy ones
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

constexpr int STREAM_SMEM_BUDGET = 224 * 1024;
constexpr int STREAM_MAX_WARPS = 16;
constexpr int STREAM_STAGES = 3;

template <int P, typename T, int STAGES_REQ = STREAM_STAGES> struct Stream {
  static constexpr int N1 = Split<P>::N1, N2 = Split<P>::N2, HALF = P / 2;
  static constexpr int TPW = 32 / N1;                                      // teams per warp
  static constexpr int ROWS = 2 * TPW;                                     // patch rows per warp item
  static constexpr int IPP = HALF / TPW;                                   // warp items per patch
  // A team's slot holds its row pair and, later, its padded N2 x (N1+1) exchange matrix (constant offsets for
  // every access, conflict-free).  A skew of N1 reals per team puts the sample reads of the teams of a warp on
  // disjoint banks — the row kernels are bound by the shared-memory data pipe (128 B/cycle/SM), so every
  // avoidable wavefront counts.  (This is also why rows arrive as 1-D bulk copies and not as one tiled
  // tensor-map box per item: a box lands densely, 128-byte aligned, and the 2-way conflict that costs was
  // measured to outweigh the cheaper issue.)
  static constexpr int EX_STRIDE = N1 + 1;
  static constexpr int SLOT_ELEMS = N2 * EX_STRIDE > P ? N2 * EX_STRIDE : P;            // complex elements
  static constexpr int TEAM_BYTES = SLOT_ELEMS * (int)sizeof(cplx<T>) + N1 * (int)sizeof(T);
  static constexpr int STAGE_BYTES = TPW * TEAM_BYTES;
  static constexpr int TABLE_BYTES = P * (int)sizeof(cplx<T>) + P * (int)sizeof(T);
  static constexpr int RING_OFFSET = (TABLE_BYTES + 1024 + 127) / 128 * 128;   // tables, mbarriers, then the ring (128-byte aligned)
  static constexpr int AVAIL = STREAM_SMEM_BUDGET - RING_OFFSET;
  static constexpr int WS = AVAIL / (STAGES_REQ * STAGE_BYTES);
  static constexpr int STAGES = WS >= 8 ? STAGES_REQ : 2;
  static constexpr int WFIT = AVAIL / (STAGES * STAGE_BYTES);
  static constexpr int WARPS = WFIT > STREAM_MAX_WARPS ? STREAM_MAX_WARPS : WFIT;
  static constexpr int THREADS = WARPS * 32;
  static constexpr size_t SMEM = RING_OFFSET + (size_t)WARPS * STAGES * STAGE_BYTES;
  static_assert(WARPS >= 2, "stage ring does not fit shared memory");
  static_assert(WARPS * STAGES * 8 <= 768, "mbarriers must fit the room reserved between the tables and the ring");
  static_assert(TEAM_BYTES % 16 == 0, "team slots must keep 16-byte alignment for bulk copies");

  __device__ static __forceinline__ int ex(int k2, int n1) { return k2 * EX_STRIDE + n1; }
};

// The gather kernel's own ring.  At 128 px three stages leave room for 15 warps (4 + 4 + 4 + 3 on the schedulers); its
// items are short enough that two stages and 16 warps are faster (single 1024^2 frame: 17.0 -> 15.1 us, 8 frames: 7.0
// -> 6.8 us per frame), while the overlap-add kernel keeps three (6.2 vs 6.5 us).
template <int P, typename T>
using StreamK1 = Stream<P, T, (P == 128 && sizeof(T) == 4) ? 2 : STREAM_STAGES>;

// K1's spectrum stores carry an L2 evict_last hint: K2 reads them next, and the tail of K1's output then survives in L2
// (K2 -0.5 us per frame at B=8, -2.6 us on a single frame)
__device__ __forceinline__ unsigned long long l2_policy_evict_last() {
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void st_spec(float2* p, float2 v, unsigned long long pol) {
  asm volatile("st.global.L2::cache_hint.v2.f32 [%0], {%1, %2}, %3;" ::"l"(p), "f"(v.x), "f"(v.y), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_spec(double2* p, double2 v, unsigned long long) { *p = v; }

// ============================================================================ K1, streaming
// gather + apodize + row FFT (same arithmetic as k1_gather_window_rowfft).  Warp item = one BandItem (ROWS consecutive
// rows of one band) of one frame; team tm of the warp owns rows (2*tm, 2*tm+1) of it.  The rows are stored to the band
// buffer without the row window (rpsf_bands.cuh).  The body stays a function apart from its kernel (as K3's does):
// written into the kernel, the same source compiles to different instructions.
template <int P, typename T, typename ST>
__device__ __forceinline__ void
k1_stream_body(const T* __restrict__ image, cplx<T>* __restrict__ spec, const RowBands rb,
               const cplx<T>* __restrict__ tw_g, const T* __restrict__ win_g, const ApplyGeom& g, int batch, int bulk_ok,
               unsigned cta, unsigned n_cta, unsigned char* smem_raw) {
  constexpr int N1 = ST::N1, N2 = ST::N2, HALF = ST::HALF, ROWS = ST::ROWS;
  constexpr int STAGES = ST::STAGES, WARPS = ST::WARPS;
  constexpr unsigned ROW_BYTES = P * sizeof(T);
  constexpr unsigned ALL_LIVE = (1u << ROWS) - 1u;
  static_assert(ROWS == band_quantum<P>(), "a band item is one warp item");
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  T* win = reinterpret_cast<T*>(tw + P);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + ST::TABLE_BYTES);            // [WARPS][STAGES]
  unsigned char* ring = smem_raw + ST::RING_OFFSET;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tm = lane / N1, t = lane % N1;
  for (int i = threadIdx.x; i < P; i += blockDim.x) { tw[i] = tw_g[i]; win[i] = win_g[i]; }
  uint64_t* bar = bars + warp * STAGES;
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) mbar_init(bar + s, 1);
    mbar_fence_init();
  }
  __syncthreads();
  grid_dependency_wait();         // tables and barriers are ready; frames / spectra may come from the kernel before
  grid_launch_dependents();

  unsigned char* my_ring = ring + (size_t)warp * STAGES * ST::STAGE_BYTES;
  const unsigned long long l2_keep = l2_policy_evict_last();
  const unsigned n_items = (unsigned)batch * (unsigned)rb.n_items;           // host guarantees batch * frame_rows < 2^30
  const unsigned stride = n_cta * WARPS;
  const unsigned first = cta * WARPS + warp;
  const bool direct = g.pad_mode == PAD_NONE;

  // How an item's rows reach its stage:
  //   BULK    every column lies inside the frame: one bulk copy per row
  //   PARTIAL the band hangs over the left/right frame edge: bulk copy of the in-frame span, then the
  //           overhanging columns are filled from their pad_index() sources (mirrored columns are
  //           read back from the stage itself when the source lies in the copied span)
  //   MANUAL  unaligned corners, `constant` rows above/below the frame, zero rows of the band: the warp gathers every
  //           sample
  enum : unsigned { BULK = 0, PARTIAL = 1, MANUAL = 2 };

  // ---- the head of the pipeline: the next item to be issued, decoded incrementally ----------
  // item = f * n_items + i; one step adds `stride` = (df, di) with a carry
  unsigned head = first;
  int hi = int(first % (unsigned)rb.n_items), hf = int(first / (unsigned)rb.n_items);
  const int di = int(stride % (unsigned)rb.n_items), df = int(stride / (unsigned)rb.n_items);
  BandItem hitem{0, 0, 0, 0};
  auto load_item = [&](int i) {
    const int4 v = __ldg(reinterpret_cast<const int4*>(rb.items) + i);
    return BandItem{v.x, v.y, v.z, (unsigned)v.w};
  };
  if (head < n_items) hitem = load_item(hi);
  auto advance_head = [&]() {
    head += stride;
    hi += di; hf += df;
    if (hi >= rb.n_items) { hi -= rb.n_items; ++hf; }
    if (head < n_items) hitem = load_item(hi);      // consumed one iteration later
  };

  unsigned phase = 0;      // bit s: parity the next wait on stage s must see

  // issue the head item into stage `st`; returns (band-buffer row index << 2) | kind
  auto issue_head = [&](int st) -> unsigned {
    const unsigned rowidx = (unsigned)hf * (unsigned)rb.frame_rows + (unsigned)hitem.buf_row;
    unsigned char* stage = my_ring + st * ST::STAGE_BYTES;
    const int x_lo = direct ? hitem.cx : max(hitem.cx, 0);
    const int x_hi = direct ? hitem.cx + P : min(hitem.cx + P, g.W);
    // source span AND its landing offset inside the stage row must keep the 16-byte granularity of bulk copies
    // (a band overhanging both frame edges can have aligned ends but a misaligned offset x_lo - cx)
    const bool aligned = bulk_ok && x_hi > x_lo && ((x_lo * (int)sizeof(T)) & 15) == 0 && ((x_hi * (int)sizeof(T)) & 15) == 0 &&
                         (((x_lo - hitem.cx) * (int)sizeof(T)) & 15) == 0;
    int y = 0;
    if (lane < ROWS) y = pad_index(hitem.row + lane, g.H, g.pad_mode);
    const bool rows_ok = __all_sync(0xffffffffu, direct || y >= 0) && hitem.live == ALL_LIVE;
    const unsigned kind = !(aligned && rows_ok) ? MANUAL : (x_hi - x_lo == P ? BULK : PARTIAL);
    if (kind != MANUAL) {
      const unsigned bytes = (unsigned)(x_hi - x_lo) * (unsigned)sizeof(T);
      // The stage was last written through the generic proxy (exchange matrix, PARTIAL / MANUAL fills); the
      // closing __syncwarp of that iteration ordered those stores before lane 0, whose proxy fence now orders
      // them before the async-proxy writes of the refill.
      if (lane == 0) {
        fence_proxy_async();
        mbar_expect_tx(bar + st, ROWS * bytes);
      }
      __syncwarp();
      if (lane < ROWS) {
        const T* src = image + (long long)hf * g.img_frame_stride + (long long)(y - g.img_row0) * g.img_pitch + x_lo;
        bulk_load(stage + (lane >> 1) * ST::TEAM_BYTES + (lane & 1) * ROW_BYTES + (x_lo - hitem.cx) * (int)sizeof(T), src, bytes,
                  bar + st);
      }
    }
    return (rowidx << 2) | kind;
  };

  unsigned pend[STAGES - 1], pend_item[STAGES - 1];    // (band-buffer row << 2) | kind, and the item's number
#pragma unroll
  for (int k = 0; k < STAGES - 1; ++k) {
    pend[k] = 0; pend_item[k] = 0;
    if (head < n_items) { pend_item[k] = head; pend[k] = issue_head(k); advance_head(); }
  }

  // per-thread constants: offset inside a stage, column window of this thread's samples
  const unsigned team_off = tm * ST::TEAM_BYTES;
  T wcol[N2];
  static_for<0, N2>([&](auto jj) { wcol[decltype(jj)::value] = win[t + N1 * decltype(jj)::value]; });

  int s = 0;
  for (unsigned it = first; it < n_items; it += stride) {
    const unsigned cur = pend[0], item = pend_item[0];
#pragma unroll
    for (int k = 0; k + 1 < STAGES - 1; ++k) { pend[k] = pend[k + 1]; pend_item[k] = pend_item[k + 1]; }
    // the stage the previous iteration released receives the head item
    if (head < n_items) {
      pend_item[STAGES - 2] = head;
      pend[STAGES - 2] = issue_head(s == 0 ? STAGES - 1 : s - 1);
      advance_head();
    }
    const unsigned kind = cur & 3u, rowidx = cur >> 2;
    unsigned char* stage = my_ring + s * ST::STAGE_BYTES;
    if (kind != MANUAL) {
      mbar_wait(bar + s, (phase >> s) & 1u);
      phase ^= 1u << s;
    }
    if (kind >= PARTIAL) {
      // rare path: recover the item from its number
      const int f = int(item / (unsigned)rb.n_items);
      const BandItem bi = load_item(int(item - (unsigned)f * (unsigned)rb.n_items));
      const T* img = image + (long long)f * g.img_frame_stride;
      const int lo_c = kind == PARTIAL ? max(-bi.cx, 0) : 0;                      // bulk-copied columns [lo_c, hi_c)
      const int hi_c = kind == PARTIAL ? min(g.W - bi.cx, P) : 0;
      const int n_fill = lo_c + (P - hi_c);                                       // columns outside [lo_c, hi_c)
#pragma unroll 1
      for (int ci = lane; ci < n_fill; ci += 32) {
        const int c = ci < lo_c ? ci : ci - lo_c + hi_c;
        const int x = pad_index(bi.cx + c, g.W, g.pad_mode);
        const int cs = x - bi.cx;                                                 // source column inside the stage?
        const bool in_stage = !direct && x >= 0 && cs >= lo_c && cs < hi_c;
#pragma unroll 1
        for (int r = 0; r < ROWS; ++r) {
          T* dst = reinterpret_cast<T*>(stage + (r >> 1) * ST::TEAM_BYTES + (r & 1) * ROW_BYTES);
          T val = T(0);
          if (in_stage) {
            val = dst[cs];
          } else if ((bi.live >> r) & 1u) {
            const int y = pad_index(bi.row + r, g.H, g.pad_mode);
            if (direct || (x >= 0 && y >= 0)) val = img[(long long)(y - g.img_row0) * g.img_pitch + x];
          }
          dst[c] = val;
        }
      }
      __syncwarp();
    }

    const T* ra_p = reinterpret_cast<const T*>(stage + team_off);
    const T* rb_p = ra_p + P;
    cplx<T>* scr = reinterpret_cast<cplx<T>*>(stage + team_off);
    cplx<T> v[N2];
    static_for<0, N2>([&](auto jj) {
      constexpr int j = decltype(jj)::value;
      const int n = t + N1 * j;
      v[j] = cscale(mk<T>(ra_p[n], rb_p[n]), wcol[j]);
    });
    __syncwarp();                                            // samples are in registers: the slot becomes the exchange buffer
    auto sync = []() { __syncwarp(); };
    coop_fft_forward<P, T>(v, t, scr, tw, [](int k2, int n1) { return ST::ex(k2, n1); }, sync);

    // This thread holds Z[k] for k = (t + N1*m) + N2*k1 in v[m*N1 + k1].  Split into the two rows' Hermitian
    // half-spectra times two: A[k] = Z[k] + conj Z[P-k], B[k] = -i (Z[k] - conj Z[P-k]); the factor 1/2 and the row
    // window are applied by the reader (rpsf_bands.cuh).  Z[P-k] for k = t + N1*i sits in lane N1-t of the team at a
    // compile-time register, so it comes by shuffle — no second pass through shared memory (the data pipe is this
    // kernel's bound).
    cplx<T>* outa = spec + ((size_t)rowidx + 2 * tm) * HALF + t;
    constexpr int R = N2 / N1;
    auto reg_of = [](int i) constexpr { return (i % R) * N1 + i / R; };   // register holding bin (lane) + N1*i
    const int partner = (N1 - t) & (N1 - 1);
    static_for<0, HALF / N1>([&](auto ii) {
      constexpr int i = decltype(ii)::value;
      const cplx<T> z1 = v[reg_of(i)];
      const cplx<T> mine = v[reg_of((N2 - i) % N2)];                     // lane 0: bin P - N1*i is its own
      const cplx<T> theirs = v[reg_of(N2 - 1 - i)];                      // lane t > 0: bin P - t - N1*i = (N1-t) + N1*(N2-1-i)
      cplx<T> z2;
      z2.x = __shfl_sync(0xffffffffu, theirs.x, partner, N1);
      z2.y = __shfl_sync(0xffffffffu, theirs.y, partner, N1);
      if (t == 0) z2 = mine;
      const cplx<T> D = padd(z1, mk<T>(-z2.x, z2.y));
      cplx<T> A = padd(z1, mk<T>(z2.x, -z2.y));
      cplx<T> B = mk<T>(D.y, -D.x);
      if constexpr (i == 0) {
        if (t == 0) {                                        // pack (DC, Nyquist): both real
          const cplx<T> zn = v[reg_of(N2 / 2)];
          A = mk<T>(T(2) * z1.x, T(2) * zn.x);
          B = mk<T>(T(2) * z1.y, T(2) * zn.y);
        }
      }
      st_spec(outa + N1 * i, A, l2_keep);
      st_spec(outa + HALF + N1 * i, B, l2_keep);
    });
    // coop_fft_forward ended with a team barrier after its last exchange read: the stage may be refilled
    s = s + 1 == STAGES ? 0 : s + 1;
  }
  __syncwarp();
}

template <int P, typename T>
__global__ void __launch_bounds__(StreamK1<P, T>::THREADS, 1)
k1_stream(const T* __restrict__ image, cplx<T>* __restrict__ spec, RowBands rb, const cplx<T>* __restrict__ tw_g,
          const T* __restrict__ win_g, ApplyGeom g, int batch, int bulk_ok) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  k1_stream_body<P, T, StreamK1<P, T>>(image, spec, rb, tw_g, win_g, g, batch, bulk_ok, blockIdx.x, gridDim.x, smem_raw);
}

// ============================================================================ K3, streaming
// row IFFT + window + overlap-add (transform.py:164-177; same arithmetic as k3_rowpair_gather).
//
// For a covering the (patch, row pair) items that land on one pair of output rows form a chain of
// groups: group g holds the items whose patch corner column is cx0 + g*P/2 (one per overlapping
// patch row, summed in the frequency domain in colour order, one inverse FFT per group), and
// consecutive groups overlap by half a patch.  A team walks a chain left to right keeping the right
// half of the previous group's rows in registers:
//
//     out[cx_g .. cx_g + P/2) = right half of group g-1  +  left half of group g
//
// so every output pixel is produced exactly once, straight from registers — no shared-memory
// plane, no zero fill, no read-modify-write, and a fixed two-term sum per pixel (bit-stable; the
// same sum on every slab and every chunking).  Chains are cut into chunks for parallelism; a
// chunk that does not start its chain recomputes the group before it (flag SEAM) only for its
// right half.  Items arrive by bulk copy into the warp's stage ring exactly like K1's rows; the
// stage of a group's last item doubles as the exchange buffer of the group's inverse FFT.
struct StreamTask {
  int y;            // output rows y, y+1
  int cx0;          // corner column of the first group this task computes
  int item_begin;   // into the item-code list
  int n_steps;      // item codes to walk; 0 = idle team
  int flags;        // TASK_SEAM | TASK_LAST
  int pad0, pad1, pad2;   // padding to 32 bytes
};
enum : int { TASK_SEAM = 1, TASK_LAST = 2 };
constexpr unsigned ITEM_LAST_OF_GROUP = 1u << 30;            // item code = (active*P/2 + pair) | flag

// Fused output gather for patch-row slabs across GPUs: besides `out`, every pixel is stored to the same
// position of up to 7 peer buffers (byte offsets from `out`; the peers' frames mapped over NVLink with
// CUDA IPC), so the band lands in every rank's full frame while the kernel runs and no all-gather follows.
struct OutMirrors {
  int n;
  long long delta[7];
};

// Item code = active * P/2 + pair; patch `a` of frame `f` sits at workspace slot f * n_active + a.
template <int P, typename T, bool MIRROR>
__device__ __forceinline__ void
k3_stream_body(const cplx<T>* __restrict__ spec, T* __restrict__ out, const StreamTask* __restrict__ tasks,
               const unsigned* __restrict__ codes, int n_warp_items, const cplx<T>* __restrict__ tw_g,
               const T* __restrict__ win_g, const ApplyGeom& g, int batch, const OutMirrors& mir, unsigned cta,
               unsigned n_cta, unsigned char* smem_raw) {
  auto put = [&](T* p, T val) {
    *p = val;
    if constexpr (MIRROR) {
      for (int d = 0; d < mir.n; ++d) *reinterpret_cast<T*>(reinterpret_cast<char*>(p) + mir.delta[d]) = val;
    }
  };
  using ST = Stream<P, T>;
  constexpr int N1 = ST::N1, N2 = ST::N2, HALF = ST::HALF, TPW = ST::TPW;
  constexpr int STAGES = ST::STAGES, WARPS = ST::WARPS;
  constexpr int HN = N2 / 2;                                 // registers per half row
  constexpr unsigned ITEM_BYTES = P * sizeof(cplx<T>);      // one row pair of half-spectra
  cplx<T>* tw = reinterpret_cast<cplx<T>*>(smem_raw);
  T* win = reinterpret_cast<T*>(tw + P);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + ST::TABLE_BYTES);
  unsigned char* ring = smem_raw + ST::RING_OFFSET;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tm = lane / N1, t = lane % N1;
  for (int i = threadIdx.x; i < P; i += blockDim.x) { tw[i] = tw_g[i]; win[i] = win_g[i]; }
  uint64_t* bar = bars + warp * STAGES;
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) mbar_init(bar + s, 1);
    mbar_fence_init();
  }
  __syncthreads();
  grid_dependency_wait();         // tables and barriers are ready; frames / spectra may come from the kernel before
  grid_launch_dependents();

  unsigned char* my_ring = ring + (size_t)warp * STAGES * ST::STAGE_BYTES;
  const unsigned team_off = tm * ST::TEAM_BYTES;
  T wcol[N2];                                                // column window of this thread's samples
  static_for<0, N2>([&](auto jj) { wcol[decltype(jj)::value] = win[t + N1 * decltype(jj)::value]; });

  const unsigned total = (unsigned)n_warp_items * (unsigned)batch;
  const unsigned stride = n_cta * WARPS;
  unsigned phase = 0;
  int s = 0;                                                 // stage of the next step to consume

  for (unsigned wi = cta * WARPS + warp; wi < total; wi += stride) {
    const int f = int(wi / (unsigned)n_warp_items);
    const unsigned local = wi - (unsigned)f * (unsigned)n_warp_items;
    const StreamTask task = tasks[(size_t)local * TPW + tm];
    const int K = __reduce_max_sync(0xffffffffu, task.n_steps);
    const bool live = task.n_steps > 0;
    const unsigned live_teams = __popc(__ballot_sync(0xffffffffu, live && t == 0));
    const unsigned* my_codes = codes + task.item_begin;

    // issue step k into stage st: every live team's row pair of half-spectra, one bulk copy each
    auto issue = [&](unsigned code, int st) {
      if (lane == 0) {
        fence_proxy_async();
        mbar_expect_tx(bar + st, live_teams * ITEM_BYTES);
      }
      __syncwarp();
      if (live && t == 0) {
        const cplx<T>* src = spec + ((size_t)f * g.n_active * (P / 2) + (code & (ITEM_LAST_OF_GROUP - 1))) * P;
        bulk_load(my_ring + st * ST::STAGE_BYTES + team_off, src, ITEM_BYTES, bar + st);
      }
    };

    // prologue: STAGES-1 steps in flight, the code of the next one to issue in a register
    unsigned inflight[STAGES - 1];
#pragma unroll
    for (int k = 0; k < STAGES - 1; ++k) {
      inflight[k] = 0;
      if (k < K) {
        inflight[k] = live ? __ldg(my_codes + k) : 0u;
        int st = s + k; if (st >= STAGES) st -= STAGES;
        issue(inflight[k], st);
      }
    }
    unsigned next_code = (live && STAGES - 1 < K) ? __ldg(my_codes + STAGES - 1) : 0u;

    cplx<T> v[N2];
    static_for<0, N2>([&](auto ee) { v[decltype(ee)::value] = mk<T>(T(0), T(0)); });
    cplx<T> prev[HN];
    static_for<0, HN>([&](auto jj) { prev[decltype(jj)::value] = mk<T>(T(0), T(0)); });
    int cx = task.cx0;
    bool emit_left = !(task.flags & TASK_SEAM);
    const bool oka = live && task.y >= g.row_begin && task.y < g.row_end;
    const bool okb = live && task.y + 1 >= g.row_begin && task.y + 1 < g.row_end;
    T* oa = out + (size_t)f * g.out_frame_stride + (long long)(task.y - g.out_row0) * g.out_pitch + t;
    T* ob = oa + g.out_pitch;
    // 16-byte stores: row starts aligned in `out` (and hence in the mirrors, whose offsets are checked on the host)
    const bool vec_ok = MIRROR && ((reinterpret_cast<uintptr_t>(oa - t) | (uintptr_t)(g.out_pitch * sizeof(T))) & 15) == 0;

    for (int k = 0; k < K; ++k) {
      const unsigned code = inflight[0];
#pragma unroll
      for (int q = 0; q + 1 < STAGES - 1; ++q) inflight[q] = inflight[q + 1];
      if (k + STAGES - 1 < K) {
        inflight[STAGES - 2] = next_code;
        issue(next_code, s == 0 ? STAGES - 1 : s - 1);
        next_code = (live && k + STAGES < K) ? __ldg(my_codes + k + STAGES) : 0u;
      }
      mbar_wait(bar + s, (phase >> s) & 1u);
      phase ^= 1u << s;
      cplx<T>* slot = reinterpret_cast<cplx<T>*>(my_ring + s * ST::STAGE_BYTES + team_off);

      if (live) {
        // Z[k] += wa*Ua[k] + i*wb*Ub[k] for k <= P/2, Hermitian mirror above; bin 0 packs (DC, Nyquist)
        // row windows of the item's two rows (transform.py:165)
        const int pair = int((code & (ITEM_LAST_OF_GROUP - 1)) % (P / 2));
        const T wa_s = win[2 * pair], wb_s = win[2 * pair + 1];
        const cplx<T> wa = mk<T>(wa_s, wa_s), wb = mk<T>(wb_s, wb_s);
        const cplx<T>* lo = slot + t;                      // Ua[bin] = lo[bin - t], Ub[bin] = lo[P/2 + bin - t]
        const cplx<T>* neg = slot - t;                     // Ua[P - bin] = neg[P - (bin - t)]
        const cplx<T> p0a = slot[0], p0b = slot[HALF];     // packed (DC, Nyquist) of the two rows
        static_for<0, N2>([&](auto ee) {
          constexpr int e = decltype(ee)::value;
          constexpr int m = e / N1, k1 = e % N1;
          constexpr int base = N1 * m + N2 * k1;            // bin = base + t; [base, base + N1) never straddles P/2
          cplx<T> a2, b2;
          if constexpr (base < HALF) {
            const cplx<T> pa = lo[base], pb = lo[HALF + base];
            a2 = pa; b2 = mk<T>(-pb.y, pb.x);
            if constexpr (base == 0) {
              if (t == 0) { a2 = mk<T>(p0a.x, T(0)); b2 = mk<T>(T(0), p0b.x); }
            }
          } else {
            // bin > P/2: conjugate mirror of bin P - (base + t).  (base == P/2, t == 0 is the Nyquist bin:
            // the generic read lands on a harmless in-slot word and is replaced below.)
            const cplx<T> pa = neg[P - base], pb = neg[HALF + P - base];
            a2 = mk<T>(pa.x, -pa.y); b2 = mk<T>(pb.y, pb.x);
            if constexpr (base == HALF) {
              if (t == 0) { a2 = mk<T>(p0a.y, T(0)); b2 = mk<T>(T(0), p0b.y); }
            }
          }
          v[e] = pfma(b2, wb, pfma(a2, wa, v[e]));
        });
      }
      __syncwarp();                                        // every lane has read the item

      if (__any_sync(0xffffffffu, (code & ITEM_LAST_OF_GROUP) != 0)) {
        auto sync = []() { __syncwarp(); };
        coop_fft_inverse<P, T>(v, t, slot, tw, [](int k2, int n1) { return ST::ex(k2, n1); }, sync, sync);
        // Column window: the right half is scaled and kept for the next group; the left half meets the
        // previous group's right half in ONE fused multiply-add, o = v * w + prev, written out as such so
        // that every instantiation of this kernel rounds the same way (left to the compiler, the packed
        // multiply and add were contracted in one instantiation and not in another).
        static_for<HN, N2>([&](auto jj) { v[decltype(jj)::value] = cscale(v[decltype(jj)::value], wcol[decltype(jj)::value]); });
        auto left = [&](auto jj) -> cplx<T> {
          constexpr int j = decltype(jj)::value;
          return pfma(v[j], mk<T>(wcol[j], wcol[j]), prev[j]);
        };
        bool wide = false;
        if constexpr (MIRROR && sizeof(T) == 4 && HN % 4 == 0) {
          // Mirrored stores travel over NVLink, where 64-byte pieces are expensive: transpose the two half
          // rows through the (now idle) exchange slot so that every lane holds 4 consecutive pixels, and
          // store 16 bytes per lane — 256 contiguous bytes per team and instruction — to `out` and every mirror.
          wide = emit_left && live && cx >= 0 && cx + HALF <= g.W && vec_ok;
          T* plane = reinterpret_cast<T*>(slot);
          if (wide) {
            static_for<0, HN>([&](auto jj) {
              constexpr int j = decltype(jj)::value;
              const cplx<T> o = left(jj);
              plane[t + N1 * j] = o.x;
              plane[HALF + t + N1 * j] = o.y;
            });
          }
          __syncwarp();
          if (wide) {
            static_for<0, HN / 4>([&](auto qq) {
              constexpr int q = decltype(qq)::value;
              const int i0 = q * 4 * N1 + 4 * t;
              const float4 pa = *reinterpret_cast<const float4*>(plane + i0);
              const float4 pb = *reinterpret_cast<const float4*>(plane + HALF + i0);
              float* da = reinterpret_cast<float*>(oa - t + cx + i0);       // oa / ob carry + t
              float* db = reinterpret_cast<float*>(ob - t + cx + i0);
              if (oka) {
                *reinterpret_cast<float4*>(da) = pa;
                for (int d = 0; d < mir.n; ++d) *reinterpret_cast<float4*>(reinterpret_cast<char*>(da) + mir.delta[d]) = pa;
              }
              if (okb) {
                *reinterpret_cast<float4*>(db) = pb;
                for (int d = 0; d < mir.n; ++d) *reinterpret_cast<float4*>(reinterpret_cast<char*>(db) + mir.delta[d]) = pb;
              }
            });
          }
          __syncwarp();                                     // the slot goes back to the ring after this step
        }
        if (emit_left && !wide) {
          const bool inside = cx >= 0 && cx + HALF <= g.W;
          static_for<0, HN>([&](auto jj) {
            constexpr int j = decltype(jj)::value;
            const cplx<T> o = left(jj);
            const int x = cx + N1 * j;                      // + t folded into oa / ob
            if (inside || (x + t >= 0 && x + t < g.W)) {
              if (oka) put(oa + x, o.x);
              if (okb) put(ob + x, o.y);
            }
          });
        }
        static_for<0, HN>([&](auto jj) { prev[decltype(jj)::value] = v[HN + decltype(jj)::value]; });
        if (k == K - 1 && (task.flags & TASK_LAST)) {
          const int cr = cx + HALF;                         // the chain ends: its right half stands alone
          static_for<0, HN>([&](auto jj) {
            constexpr int j = decltype(jj)::value;
            const int x = cr + N1 * j;
            if (x + t >= 0 && x + t < g.W) {
              if (oka) put(oa + x, prev[j].x);
              if (okb) put(ob + x, prev[j].y);
            }
          });
        }
        static_for<0, N2>([&](auto ee) { v[decltype(ee)::value] = mk<T>(T(0), T(0)); });
        cx += HALF;
        emit_left = true;
      }
      s = s + 1 == STAGES ? 0 : s + 1;
    }
  }
}

template <int P, typename T, bool MIRROR>
__global__ void __launch_bounds__(Stream<P, T>::THREADS, 1)
k3_stream(const cplx<T>* __restrict__ spec, T* __restrict__ out, const StreamTask* __restrict__ tasks,
          const unsigned* __restrict__ codes, int n_warp_items, const cplx<T>* __restrict__ tw_g,
          const T* __restrict__ win_g, ApplyGeom g, int batch, OutMirrors mir) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  k3_stream_body<P, T, MIRROR>(spec, out, tasks, codes, n_warp_items, tw_g, win_g, g, batch, mir, blockIdx.x, gridDim.x,
                               smem_raw);
}

}  // namespace rpsf
