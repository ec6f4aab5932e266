// rpsf_inst.cu — instantiates every kernel for one patch size (compile with -DRPSF_P=<P>).
#include "rpsf_ops.h"
#include "rpsf_kgrad.cuh"
#include "rpsf_construct_grad.cuh"

#ifndef RPSF_P
#error "compile with -DRPSF_P=<patch size>"
#endif

namespace rpsf {
namespace {

constexpr int P = RPSF_P;
using TL = Tile<P>;

template <typename T> constexpr size_t row_smem() {
  return sizeof(cplx<T>) * P + sizeof(T) * P + sizeof(cplx<T>) * size_t(TL::TEAMS) * TL::SCR;
}
template <typename T> constexpr size_t col_smem() {
  return sizeof(cplx<T>) * P + sizeof(cplx<T>) * size_t(TL::SLOTS) * P * TL::C;
}
// the column pass keeps the row window (P reals) beside the twiddles
template <typename T> constexpr size_t col_k2_smem() { return col_smem<T>() + sizeof(T) * P; }
template <typename T> constexpr size_t col_pipe_smem() {
  return sizeof(cplx<T>) * P + sizeof(T) * P + K2_STAGES * sizeof(cplx<T>) * size_t(TL::SLOTS) * P * TL::C;
}
// the pipelined column kernel needs K2_STAGES tile stages per CTA; use it while a stage is at most
// 32 KB (two or three CTAs then fit an SM)
template <typename T> constexpr bool use_col_pipe() {
  return sizeof(cplx<T>) * size_t(TL::SLOTS) * P * TL::C <= 32 * 1024 + 4096;
}
template <typename T> constexpr size_t fft2_row_smem() {
  return sizeof(cplx<T>) * P + sizeof(cplx<T>) * size_t(TL::TEAMS) * TL::SCR;
}

// Launch one of the chained kernels (k1_stream -> k2_pipelined -> k3_stream -> the next call's k1_stream) so that its
// CTAs may start while the kernel before it in the stream drains (programmatic dependent launch; the kernels wait in
// grid_dependency_wait() before they touch anything a predecessor wrote).  `which`: 1 = k1_stream, 2 = k2_pipelined,
// 4 = k3_stream.  Measured: all three start early at P <= 128 (one 1024^2 frame: 41.1 -> 34.1 us at 128 px,
// 39.4 -> 31.8 at 64 px); at P >= 256 an early column pass costs 1 % (its first wave of CTAs is placed on the SMs the
// row pass leaves first), so only the row kernels start early there (2048^2 / 256 px: 97.0 -> 95.2 us for one frame,
// 64.4 -> 63.5 per frame at 8).
constexpr int PDL_MASK = P <= 128 ? 7 : 5;
template <typename... KArgs, typename... Args>
int launch_chain(int which, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (PDL_MASK & which) ? 1 : 0;
  return (int)cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

template <typename F> int set_smem(F* fn, size_t bytes) {
  return (int)cudaFuncSetAttribute(reinterpret_cast<const void*>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

int init() {
  int e = 0;
  if ((e = set_smem(k1_gather_window_rowfft<P, float>, row_smem<float>()))) return e;
  if ((e = set_smem(k1_gather_window_rowfft<P, double>, row_smem<double>()))) return e;
  if ((e = set_smem(k1_stream<P, float>, StreamK1<P, float>::SMEM))) return e;
  if ((e = set_smem(k1_stream<P, double>, StreamK1<P, double>::SMEM))) return e;
  if ((e = set_smem(k3_stream<P, float, false>, Stream<P, float>::SMEM))) return e;
  if ((e = set_smem(k3_stream<P, double, false>, Stream<P, double>::SMEM))) return e;
  if ((e = set_smem(k3_stream<P, float, true>, Stream<P, float>::SMEM))) return e;
  if ((e = set_smem(k3_stream<P, double, true>, Stream<P, double>::SMEM))) return e;
  if ((e = set_smem(k2_colfft_mul_colifft<P, float>, col_k2_smem<float>()))) return e;
  if ((e = set_smem(k2_colfft_mul_colifft<P, double>, col_k2_smem<double>()))) return e;
  if ((e = set_smem(k2_colfft_mul_colifft<P, float, true>, col_k2_smem<float>()))) return e;
  if ((e = set_smem(k2_colfft_mul_colifft<P, double, true>, col_k2_smem<double>()))) return e;
  if constexpr (use_col_pipe<float>())
    if ((e = set_smem(k2_pipelined<P, float, 1, true>, col_pipe_smem<float>()))) return e;
  if constexpr (use_col_pipe<double>())
    if ((e = set_smem(k2_pipelined<P, double, 1, true>, col_pipe_smem<double>()))) return e;
  if constexpr (use_col_pipe<float>())
    if ((e = set_smem(k2_pipelined<P, float>, col_pipe_smem<float>()))) return e;
  if constexpr (use_col_pipe<double>())
    if ((e = set_smem(k2_pipelined<P, double>, col_pipe_smem<double>()))) return e;
  if constexpr (use_col_pipe<float>() && TL::SLOTS == 1 && TL::NTILE % 2 == 0)
    if ((e = set_smem(k2_pipelined<P, float, 2>, col_pipe_smem<float>()))) return e;
  if constexpr (use_col_pipe<double>() && TL::SLOTS == 1 && TL::NTILE % 2 == 0)
    if ((e = set_smem(k2_pipelined<P, double, 2>, col_pipe_smem<double>()))) return e;
  if constexpr (use_col_pipe<float>())
    if ((e = set_smem(k2_stack<P, float>, col_pipe_smem<float>()))) return e;
  if constexpr (use_col_pipe<double>())
    if ((e = set_smem(k2_stack<P, double>, col_pipe_smem<double>()))) return e;
  if ((e = set_smem(k3_rowifft_window_overlap_add<P, float>, row_smem<float>()))) return e;
  if ((e = set_smem(k3_rowifft_window_overlap_add<P, double>, row_smem<double>()))) return e;
  if ((e = set_smem(k3_rowpair_gather<P, float>, K3G_SMEM_MAX))) return e;
  if ((e = set_smem(k3_rowpair_gather<P, double>, K3G_SMEM_MAX))) return e;
  if ((e = set_smem(fft2_rows<P, float, float>, fft2_row_smem<float>()))) return e;
  if ((e = set_smem(fft2_rows<P, double, double>, fft2_row_smem<double>()))) return e;
  if ((e = set_smem(fft2_cols<P, float>, col_smem<float>()))) return e;
  if ((e = set_smem(fft2_cols<P, double>, col_smem<double>()))) return e;
  if ((e = set_smem(kgrad<P, float>, GradTile<P, float>::SMEM))) return e;
  if ((e = set_smem(kgrad<P, double>, GradTile<P, double>::SMEM))) return e;
  if ((e = set_smem(fft2_rows_conj<P, float>, fft2_row_smem<float>()))) return e;
  if ((e = set_smem(fft2_rows_conj<P, double>, fft2_row_smem<double>()))) return e;
  if ((e = set_smem(fft2_cols_real<P, float>, col_smem<float>()))) return e;
  if ((e = set_smem(fft2_cols_real<P, double>, col_smem<double>()))) return e;
  return 0;
}

inline unsigned cdiv(long long a, long long b) { return (unsigned)((a + b - 1) / b); }

template <typename T>
int k1_t(const void* image, void* bands, const RowBands& rb, const void* tw, const void* win, const ApplyGeom& g, int batch,
         cudaStream_t s) {
  if (rb.n_items == 0) return 0;
  dim3 grid(cdiv((long long)rb.n_items * (band_quantum<P>() / 2), TL::TEAMS), batch);
  k1_gather_window_rowfft<P, T><<<grid, TL::ROW_THREADS, row_smem<T>(), s>>>(
      (const T*)image, (cplx<T>*)bands, rb, (const cplx<T>*)tw, (const T*)win, g);
  return (int)cudaGetLastError();
}
int k1(int dt, const void* image, void* bands, const RowBands& rb, const void* tw, const void* win, const ApplyGeom& g,
       int batch, cudaStream_t s) {
  return dt == DT_F32 ? k1_t<float>(image, bands, rb, tw, win, g, batch, s)
                      : k1_t<double>(image, bands, rb, tw, win, g, batch, s);
}

template <typename T>
int k1s_t(const void* image, void* bands, const RowBands& rb, const void* tw, const void* win, const ApplyGeom& g,
          int batch, int bulk_ok, int sm_count, cudaStream_t s) {
  using ST = StreamK1<P, T>;
  const long long items = (long long)batch * rb.n_items;
  if (items == 0) return 0;
  const long long ctas = (items + ST::WARPS - 1) / ST::WARPS;
  const unsigned grid = (unsigned)(ctas < sm_count ? ctas : sm_count);
  return launch_chain(1, k1_stream<P, T>, dim3(grid), dim3(ST::THREADS), ST::SMEM, s, (const T*)image, (cplx<T>*)bands, rb,
                      (const cplx<T>*)tw, (const T*)win, g, batch, bulk_ok);
}
int k1s(int dt, const void* image, void* bands, const RowBands& rb, const void* tw, const void* win, const ApplyGeom& g,
        int batch, int bulk_ok, int sm_count, cudaStream_t s) {
  return dt == DT_F32 ? k1s_t<float>(image, bands, rb, tw, win, g, batch, bulk_ok, sm_count, s)
                      : k1s_t<double>(image, bands, rb, tw, win, g, batch, bulk_ok, sm_count, s);
}

template <typename T>
int k2_t(const void* bands, const RowBands& rb, void* spec, const void* kmain, const void* knyq, const int* active,
         const void* tw, const void* win, const ApplyGeom& g, int batch, int sm_count, cudaStream_t s) {
  // Walk several frames per CTA so the transfer-kernel tile is read once per batch, but keep
  // at least ~4 waves of CTAs in flight (SMs x 3 resident CTAs).
  const long long ctas = cdiv((long long)g.n_active * TL::NTILE, TL::SLOTS);
  int fpc = batch;
  while (fpc > 1 && ctas * cdiv(batch, fpc) < (long long)sm_count * 3 * 4) fpc = (fpc + 1) / 2;
  dim3 grid((unsigned)ctas, cdiv(batch, fpc));
  const cplx<T>* bnd = (const cplx<T>*)bands;
  if (g.win_len < P) {
    // embedded patch size: only the first win_len rows of a patch carry data (rpsf_kernels.cuh: PRUNED)
    if constexpr (use_col_pipe<T>())
      return launch_chain(2, k2_pipelined<P, T, 1, true>, grid, dim3(TL::K2_THREADS), col_pipe_smem<T>(), s, bnd, rb,
                          (cplx<T>*)spec, (const cplx<T>*)kmain, (const cplx<T>*)knyq, active, (const cplx<T>*)tw,
                          (const T*)win, batch, fpc, g);
    else
      k2_colfft_mul_colifft<P, T, true><<<grid, TL::K2_THREADS, col_k2_smem<T>(), s>>>(
          bnd, rb, (cplx<T>*)spec, (const cplx<T>*)kmain, (const cplx<T>*)knyq, active, (const cplx<T>*)tw, (const T*)win,
          batch, fpc, g);
    return (int)cudaGetLastError();
  }
  if constexpr (use_col_pipe<T>() && TL::SLOTS == 1 && TL::NTILE % 2 == 0) {
    // few frames per CTA: walk two adjacent tiles per CTA so that the stage ring and the transfer-kernel loads have
    // something to overlap with.  Only for one-slot CTAs (P >= 256): with two slots per CTA (P = 128) the same change
    // was measured 2 % (1024^2) to 8 % (2048^2) slower, at P = 64 1 % faster.  Four tiles per CTA (2048^2 / 256 px:
    // 89.9 vs 87.3 us) and two tiles at 8 frames per call (4 % slower) lost.
    if (fpc <= 1) {
      grid.x = (unsigned)cdiv(ctas, 2);
      return launch_chain(2, k2_pipelined<P, T, 2>, grid, dim3(TL::K2_THREADS), col_pipe_smem<T>(), s, bnd, rb,
                          (cplx<T>*)spec, (const cplx<T>*)kmain, (const cplx<T>*)knyq, active, (const cplx<T>*)tw,
                          (const T*)win, batch, fpc, g);
    }
  }
  if constexpr (use_col_pipe<T>())
    return launch_chain(2, k2_pipelined<P, T>, grid, dim3(TL::K2_THREADS), col_pipe_smem<T>(), s, bnd, rb, (cplx<T>*)spec,
                        (const cplx<T>*)kmain, (const cplx<T>*)knyq, active, (const cplx<T>*)tw, (const T*)win, batch, fpc,
                        g);
  else
    k2_colfft_mul_colifft<P, T><<<grid, TL::K2_THREADS, col_k2_smem<T>(), s>>>(
        bnd, rb, (cplx<T>*)spec, (const cplx<T>*)kmain, (const cplx<T>*)knyq, active, (const cplx<T>*)tw, (const T*)win,
        batch, fpc, g);
  return (int)cudaGetLastError();
}
int k2(int dt, const void* bands, const RowBands& rb, void* spec, const void* kmain, const void* knyq, const int* active,
       const void* tw, const void* win, const ApplyGeom& g, int batch, int sm_count, cudaStream_t s) {
  return dt == DT_F32 ? k2_t<float>(bands, rb, spec, kmain, knyq, active, tw, win, g, batch, sm_count, s)
                      : k2_t<double>(bands, rb, spec, kmain, knyq, active, tw, win, g, batch, sm_count, s);
}

template <typename T>
int k2s_t(const void* bands, const RowBands& rb, void* spec, long long kspec_stride, const void* kmain,
          long long kmain_stride, const void* knyq, long long knyq_stride, int n_kernels, const int* active, const void* tw,
          const void* win, const ApplyGeom& g, int batch, int sm_count, cudaStream_t s) {
  if constexpr (use_col_pipe<T>()) {
    // k2_t's grid: several frames per CTA while at least ~4 waves of CTAs stay in flight
    const long long ctas = cdiv((long long)g.n_active * TL::NTILE, TL::SLOTS);
    int fpc = batch;
    while (fpc > 1 && ctas * cdiv(batch, fpc) < (long long)sm_count * 3 * 4) fpc = (fpc + 1) / 2;
    return launch_chain(2, k2_stack<P, T>, dim3((unsigned)ctas, cdiv(batch, fpc)), dim3(TL::K2_THREADS), col_pipe_smem<T>(),
                        s, (const cplx<T>*)bands, rb, (cplx<T>*)spec, kspec_stride, (const cplx<T>*)kmain, kmain_stride,
                        (const cplx<T>*)knyq, knyq_stride, n_kernels, active, (const cplx<T>*)tw, (const T*)win, batch, fpc,
                        g);
  } else {
    return (int)cudaErrorNotSupported;
  }
}
int k2s(int dt, const void* bands, const RowBands& rb, void* spec, long long kspec_stride, const void* kmain,
        long long kmain_stride, const void* knyq, long long knyq_stride, int n_kernels, const int* active, const void* tw,
        const void* win, const ApplyGeom& g, int batch, int sm_count, cudaStream_t s) {
  return dt == DT_F32 ? k2s_t<float>(bands, rb, spec, kspec_stride, kmain, kmain_stride, knyq, knyq_stride, n_kernels, active,
                                     tw, win, g, batch, sm_count, s)
                      : k2s_t<double>(bands, rb, spec, kspec_stride, kmain, kmain_stride, knyq, knyq_stride, n_kernels,
                                      active, tw, win, g, batch, sm_count, s);
}
int k2s_ok(int dt) { return dt == DT_F32 ? use_col_pipe<float>() : use_col_pipe<double>(); }

template <typename T>
int k3_t(const void* spec, void* out, const int2* corners, const int* items, int n_items, const void* tw,
         const void* win, int store_only, const ApplyGeom& g, int batch, cudaStream_t s) {
  if (n_items == 0) return 0;
  dim3 grid(cdiv(n_items, TL::TEAMS), batch);
  k3_rowifft_window_overlap_add<P, T><<<grid, TL::ROW_THREADS, row_smem<T>(), s>>>(
      (const cplx<T>*)spec, (T*)out, corners, items, n_items, (const cplx<T>*)tw, (const T*)win, store_only, g);
  return (int)cudaGetLastError();
}
int k3(int dt, const void* spec, void* out, const int2* corners, const int* items, int n_items, const void* tw,
       const void* win, int store_only, const ApplyGeom& g, int batch, cudaStream_t s) {
  return dt == DT_F32 ? k3_t<float>(spec, out, corners, items, n_items, tw, win, store_only, g, batch, s)
                      : k3_t<double>(spec, out, corners, items, n_items, tw, win, store_only, g, batch, s);
}

template <typename T> size_t gather_smem(int teams, int seg_w) {
  constexpr size_t BUF = TL::SCR > P ? TL::SCR : P;
  return sizeof(cplx<T>) * P + sizeof(T) * P + sizeof(T) * 2 * (size_t)seg_w + sizeof(cplx<T>) * (size_t)teams * BUF;
}
size_t k3g_smem(int dt, int teams, int seg_w) {
  return dt == DT_F32 ? gather_smem<float>(teams, seg_w) : gather_smem<double>(teams, seg_w);
}
template <typename T>
int k3g_t(const void* spec, void* out, const RowTile* tiles, int n_tiles, const RowGroup* groups, const int* items,
          const void* tw, const void* win, int teams, int seg_w, const ApplyGeom& g, int batch, cudaStream_t s) {
  if (n_tiles == 0) return 0;
  dim3 grid(n_tiles, batch);
  k3_rowpair_gather<P, T><<<grid, teams * TL::N1, gather_smem<T>(teams, seg_w), s>>>(
      (const cplx<T>*)spec, (T*)out, tiles, groups, items, (const cplx<T>*)tw, (const T*)win, seg_w, g);
  return (int)cudaGetLastError();
}
int k3g(int dt, const void* spec, void* out, const RowTile* tiles, int n_tiles, const RowGroup* groups,
        const int* items, const void* tw, const void* win, int teams, int seg_w, const ApplyGeom& g, int batch,
        cudaStream_t s) {
  return dt == DT_F32 ? k3g_t<float>(spec, out, tiles, n_tiles, groups, items, tw, win, teams, seg_w, g, batch, s)
                      : k3g_t<double>(spec, out, tiles, n_tiles, groups, items, tw, win, teams, seg_w, g, batch, s);
}

template <typename T>
int k3s_t(const void* spec, void* out, const StreamTask* tasks, const unsigned* codes, int n_warp_items, const void* tw,
          const void* win, const ApplyGeom& g, int batch, int sm_count, const OutMirrors* mirrors, cudaStream_t s) {
  using ST = Stream<P, T>;
  const long long items = (long long)n_warp_items * batch;
  if (items == 0) return 0;
  const long long ctas = (items + ST::WARPS - 1) / ST::WARPS;
  const unsigned grid = (unsigned)(ctas < sm_count ? ctas : sm_count);
  if (mirrors && mirrors->n > 0)
    return launch_chain(4, k3_stream<P, T, true>, dim3(grid), dim3(ST::THREADS), ST::SMEM, s, (const cplx<T>*)spec, (T*)out,
                        tasks, codes, n_warp_items, (const cplx<T>*)tw, (const T*)win, g, batch, *mirrors);
  return launch_chain(4, k3_stream<P, T, false>, dim3(grid), dim3(ST::THREADS), ST::SMEM, s, (const cplx<T>*)spec, (T*)out,
                      tasks, codes, n_warp_items, (const cplx<T>*)tw, (const T*)win, g, batch, OutMirrors{});
}
int k3s(int dt, const void* spec, void* out, const StreamTask* tasks, const unsigned* codes, int n_warp_items,
        const void* tw, const void* win, const ApplyGeom& g, int batch, int sm_count, const OutMirrors* mirrors,
        cudaStream_t s) {
  return dt == DT_F32 ? k3s_t<float>(spec, out, tasks, codes, n_warp_items, tw, win, g, batch, sm_count, mirrors, s)
                      : k3s_t<double>(spec, out, tasks, codes, n_warp_items, tw, win, g, batch, sm_count, mirrors, s);
}
int stream_tpw() { return Stream<P, float>::TPW; }

template <typename T, typename TK>
int prep_t(const void* full, void* kmain, void* knyq, int n, cudaStream_t s) {
  const long long total = (long long)n * ((long long)P * TL::HALF + P);
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long long cap = (long long)sms * 32;
  const unsigned blocks = (unsigned)((total + 255) / 256 < cap ? (total + 255) / 256 : cap);
  prep_transfer_kernel<P, T, TK><<<blocks ? blocks : 1, 256, 0, s>>>((const TK*)full, (cplx<T>*)kmain, (cplx<T>*)knyq, n);
  return (int)cudaGetLastError();
}
int prep(int dt, int kdt, const void* full, void* kmain, void* knyq, int n, cudaStream_t s) {
  if (dt == DT_F32) return kdt == DT_F32 ? prep_t<float, float2>(full, kmain, knyq, n, s)
                                         : prep_t<float, double2>(full, kmain, knyq, n, s);
  return kdt == DT_F32 ? prep_t<double, float2>(full, kmain, knyq, n, s)
                       : prep_t<double, double2>(full, kmain, knyq, n, s);
}

template <typename T>
int fft2_t(const void* values, void* out, const void* tw, long long n, cudaStream_t s) {
  if (n == 0) return 0;
  fft2_rows<P, T, T><<<cdiv(n * P, TL::TEAMS), TL::ROW_THREADS, fft2_row_smem<T>(), s>>>(
      (const T*)values, (cplx<T>*)out, (const cplx<T>*)tw, n * P);
  int e = (int)cudaGetLastError();
  if (e) return e;
  fft2_cols<P, T><<<cdiv(n * (P / TL::C), TL::SLOTS), TL::K2_THREADS, col_smem<T>(), s>>>(
      (cplx<T>*)out, (const cplx<T>*)tw, n);
  return (int)cudaGetLastError();
}
int fft2(int dt, int in_dt, const void* values, void* out, const void* tw, long long n, cudaStream_t s) {
  if (dt != in_dt) return (int)cudaErrorInvalidValue;
  return dt == DT_F32 ? fft2_t<float>(values, out, tw, n, s) : fft2_t<double>(values, out, tw, n, s);
}

template <typename T>
int fft2_adjoint_t(const void* grad, void* scratch, void* out, const void* tw, long long n, cudaStream_t s) {
  if (n == 0) return 0;
  fft2_rows_conj<P, T><<<cdiv(n * P, TL::TEAMS), TL::ROW_THREADS, fft2_row_smem<T>(), s>>>(
      (const cplx<T>*)grad, (cplx<T>*)scratch, (const cplx<T>*)tw, n * P);
  int e = (int)cudaGetLastError();
  if (e) return e;
  fft2_cols_real<P, T><<<cdiv(n * (P / TL::C), TL::SLOTS), TL::K2_THREADS, col_smem<T>(), s>>>(
      (const cplx<T>*)scratch, (T*)out, (const cplx<T>*)tw, n);
  return (int)cudaGetLastError();
}
int fft2_adjoint(int dt, const void* grad, void* scratch, void* out, const void* tw, long long n, cudaStream_t s) {
  return dt == DT_F32 ? fft2_adjoint_t<float>(grad, scratch, out, tw, n, s)
                      : fft2_adjoint_t<double>(grad, scratch, out, tw, n, s);
}

// launched plainly (no programmatic dependent launch): it reads both plans' spectra, written by the kernels before it
template <typename T>
int kgrad_t(const void* xspec, const RowBands& xb, const void* gspec, const RowBands& gb, void* out, const int* active,
            const void* tw, const void* win, int n_active, int batch, cudaStream_t s) {
  using GT = GradTile<P, T>;
  if (n_active == 0) return 0;
  kgrad<P, T><<<cdiv((long long)n_active * GT::NTILE, GT::SLOTS), GT::THREADS, GT::SMEM, s>>>(
      (const cplx<T>*)xspec, xb, (const cplx<T>*)gspec, gb, (cplx<T>*)out, active, (const cplx<T>*)tw, (const T*)win,
      n_active, batch);
  return (int)cudaGetLastError();
}
int kgrad_launch(int dt, const void* xspec, const RowBands& xb, const void* gspec, const RowBands& gb, void* out,
                 const int* active, const void* tw, const void* win, int n_active, int batch, cudaStream_t s) {
  return dt == DT_F32 ? kgrad_t<float>(xspec, xb, gspec, gb, out, active, tw, win, n_active, batch, s)
                      : kgrad_t<double>(xspec, xb, gspec, gb, out, active, tw, win, n_active, batch, s);
}

const Ops kOps = {P, init, k1, k1s, k2, k2s, k2s_ok, k3, k3g, k3s, stream_tpw, k3g_smem, prep, fft2, kgrad_launch, fft2_adjoint};

}  // namespace

#define RPSF_CAT2(a, b) a##b
#define RPSF_CAT(a, b) RPSF_CAT2(a, b)
const Ops* RPSF_CAT(ops_p, RPSF_P)() { return &kOps; }

}  // namespace rpsf
