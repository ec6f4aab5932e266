// rpsf_api.cu — C ABI (include/rpsf_b200.h) over the sm_100a kernels.
// Host-side planning: coordinate validation, colour classes of the patch overlap graph,
// per-colour work lists, resident-row range, workspace ownership.
#include <algorithm>
#include <atomic>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <type_traits>
#include <vector>

#include "../../include/rpsf_b200.h"
#include "rpsf_ops.h"
#include "rpsf_saturation.cuh"
#include "rpsf_builder.cuh"
#include "rpsf_adjoint.cuh"
#include "rpsf_construct_grad.cuh"

namespace rpsf {
const Ops* ops_for(int P) {
  switch (P) {
    case 16: return ops_p16();
    case 32: return ops_p32();
    case 64: return ops_p64();
    case 128: return ops_p128();
    case 256: return ops_p256();
    case 512: return ops_p512();
    default: return nullptr;
  }
}
}  // namespace rpsf

using namespace rpsf;

namespace {

thread_local std::string g_error;
std::atomic<long long> g_launches{0};

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_error = buf;
  return code;
}

#define CU(expr)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(RPSF_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

#define LAUNCH(expr)                                                                               \
  do {                                                                                             \
    int e_ = (expr);                                                                               \
    g_launches.fetch_add(1, std::memory_order_relaxed);                                            \
    if (e_ != 0)                                                                                   \
      return fail(RPSF_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString((cudaError_t)e_));       \
  } while (0)

size_t real_size(int dt) { return dt == DT_F32 ? 4 : 8; }
size_t elem_size(int dt) {
  switch (dt) {
    case RPSF_F32: case RPSF_I32: case RPSF_U32: return 4;
    case RPSF_F64: case RPSF_I64: return 8;
    case RPSF_U8: return 1;
    case RPSF_I16: case RPSF_U16: return 2;
    default: return 0;
  }
}

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ---- CUDA graph capture (DESIGN.md section 5) ---------------------------------------------------------------------
// Streams this library has seen capturing: the entry points that take no stream (plan creation, upload, IPC, the host
// path) look here to refuse while a capture that went through the library is still open.
std::mutex g_capture_mu;
std::vector<cudaStream_t> g_capture_streams;
std::atomic<int> g_capture_count{0};      // g_capture_streams.size(), read without the mutex by eager calls

// 1 when `s` is capturing, 0 when not.  The legacy stream cannot be asked while another stream captures
// (cudaErrorStreamCaptureImplicit): that counts as capturing, since work on it would invalidate the capture.
int stream_capturing(cudaStream_t s, unsigned long long* id = nullptr) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  unsigned long long cid = 0;
  const cudaError_t e = cudaStreamGetCaptureInfo(s, &st, &cid);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return e == cudaErrorStreamCaptureImplicit ? 1 : 0;
  }
  if (id) *id = cid;
  return st != cudaStreamCaptureStatusNone ? 1 : 0;
}

void note_capture(cudaStream_t s) {
  std::lock_guard<std::mutex> lock(g_capture_mu);
  if (std::find(g_capture_streams.begin(), g_capture_streams.end(), s) == g_capture_streams.end()) {
    g_capture_streams.push_back(s);
    g_capture_count.store((int)g_capture_streams.size());
  }
}

// an eager call on `s`: a capture on it has ended, so it leaves the list (cheap when the list is empty)
void forget_capture(cudaStream_t s) {
  if (g_capture_count.load() == 0) return;
  std::lock_guard<std::mutex> lock(g_capture_mu);
  auto it = std::find(g_capture_streams.begin(), g_capture_streams.end(), s);
  if (it != g_capture_streams.end()) g_capture_streams.erase(it);
  g_capture_count.store((int)g_capture_streams.size());
}

// whether a capture the library has taken part in is still open (finished ones are forgotten)
bool capture_open() {
  std::lock_guard<std::mutex> lock(g_capture_mu);
  bool open = false;
  for (size_t i = 0; i < g_capture_streams.size();) {
    if (stream_capturing(g_capture_streams[i])) { open = true; ++i; }
    else g_capture_streams.erase(g_capture_streams.begin() + (long)i);
  }
  g_capture_count.store((int)g_capture_streams.size());
  return open;
}

int refuse_capture(const char* what) {
  return fail(RPSF_E_UNSUPPORTED, "%s cannot run while a CUDA graph is being captured (it allocates or synchronises): "
              "run the call once before capturing so that its plans, workspaces and kernel layout exist", what);
}

// refuse a stream-less entry point while a capture is open
#define REFUSE_IN_CAPTURE(what) do { if (capture_open()) return refuse_capture(what); } while (0)
// refuse an entry point that would allocate or synchronise on `s` while `s` captures
#define REFUSE_ON_CAPTURING(s, what) do { if (stream_capturing(s) || capture_open()) return refuse_capture(what); } while (0)

// the calls on this thread between the halves of an OrderedCall on a capturing stream (lazy allocations refuse)
thread_local bool t_capturing = false;

// FFT length for a patch size without a native one: the next power of two >= 2 P - 1 (0 if none fits 16..512)
int embedded_length(int P) {
  if (P < 2) return 0;
  int m = 16;
  while (m < 2 * P - 1) m *= 2;
  return m <= 512 ? m : 0;
}

int sm_count_of(int device) {
  static std::mutex mu;
  static std::map<int, int> cache;
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(device);
  if (it != cache.end()) return it->second;
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || n < 1) n = 148;
  cache[device] = n;
  return n;
}
int current_sm_count() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  return sm_count_of(dev);
}

template <typename T>
int upload_tables(int P, void** tw_out, void** win_out) {
  const int N1 = P == 16 ? 4 : P == 32 ? 4 : P == 64 ? 8 : P == 128 ? 8 : 16;
  const int N2 = P / N1;
  std::vector<T> tw(2 * (size_t)P), win(P);
  const double two_pi = 6.283185307179586476925286766559;
  for (int k2 = 0; k2 < N2; ++k2)
    for (int n1 = 0; n1 < N1; ++n1) {
      // exp(-2*pi*i*n1*k2/P); reduce the product mod P first so the angle stays exact
      const int r = (n1 * k2) % P;
      const double ang = two_pi * double(r) / double(P);
      tw[2 * (k2 * N1 + n1)] = T(std::cos(ang));
      tw[2 * (k2 * N1 + n1) + 1] = T(-std::sin(ang));
    }
  // apodization window, transform.py:151-154: sin((n + 0.5) * (pi / P)) per axis
  const double pi = 3.14159265358979323846264338327950288;
  for (int n = 0; n < P; ++n) win[n] = T(std::sin((n + 0.5) * (pi / P)));
  CU(cudaMalloc(tw_out, tw.size() * sizeof(T)));
  CU(cudaMalloc(win_out, win.size() * sizeof(T)));
  CU(cudaMemcpy(*tw_out, tw.data(), tw.size() * sizeof(T), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(*win_out, win.data(), win.size() * sizeof(T), cudaMemcpyHostToDevice));
  return 0;
}

// Twiddle / window tables are a pure function of (P, dtype): one copy per device for the life of the
// library (3 KB at P = 256), shared by every transform and by rpsf_psf_fft2 — nothing to free, no
// synchronisation when a call returns.
struct TableEntry { void* tw; void* win; };
std::mutex g_tables_mu;
std::map<std::tuple<int, int, int>, TableEntry> g_tables;

int shared_tables(int P, int dtype, int device, void** tw, void** win) {
  std::lock_guard<std::mutex> lock(g_tables_mu);
  const auto key = std::make_tuple(P, dtype, device);
  auto it = g_tables.find(key);
  if (it == g_tables.end()) {
    TableEntry e{nullptr, nullptr};
    int rc = dtype == RPSF_F32 ? upload_tables<float>(P, &e.tw, &e.win) : upload_tables<double>(P, &e.tw, &e.win);
    if (rc) { cudaFree(e.tw); cudaFree(e.win); return rc; }
    it = g_tables.emplace(key, e).first;
  }
  *tw = it->second.tw; *win = it->second.win;
  return 0;
}

// whether the tables of (P, dtype, device) exist already, so that a call can take them while a graph is captured
bool tables_ready(int P, int dtype, int device) {
  std::lock_guard<std::mutex> lock(g_tables_mu);
  return g_tables.count(std::make_tuple(P, dtype, device)) != 0;
}

}  // namespace

namespace {
template <typename TI, typename TO>
void launch_convert(const void* src, long long sp, void* dst, long long dp, int rows, int cols, cudaStream_t s) {
  const long long total = (long long)rows * cols;
  const unsigned blocks = (unsigned)std::min<long long>((total + 255) / 256, (long long)current_sm_count() * 16);
  convert_2d<TI, TO><<<blocks ? blocks : 1, 256, 0, s>>>((const TI*)src, sp, (TO*)dst, dp, rows, cols);
}
template <typename TO>
int convert_to(const void* src, int sdt, long long sp, void* dst, long long dp, int rows, int cols, cudaStream_t s) {
  switch (sdt) {
    case RPSF_F32: launch_convert<float, TO>(src, sp, dst, dp, rows, cols, s); break;
    case RPSF_F64: launch_convert<double, TO>(src, sp, dst, dp, rows, cols, s); break;
    case RPSF_U8: launch_convert<uint8_t, TO>(src, sp, dst, dp, rows, cols, s); break;
    case RPSF_I16: launch_convert<int16_t, TO>(src, sp, dst, dp, rows, cols, s); break;
    case RPSF_U16: launch_convert<uint16_t, TO>(src, sp, dst, dp, rows, cols, s); break;
    case RPSF_I32: launch_convert<int32_t, TO>(src, sp, dst, dp, rows, cols, s); break;
    case RPSF_U32: launch_convert<uint32_t, TO>(src, sp, dst, dp, rows, cols, s); break;
    case RPSF_I64: launch_convert<long long, TO>(src, sp, dst, dp, rows, cols, s); break;
    default: return -1;
  }
  return 0;
}
}  // namespace

namespace {
// Tables of the streaming overlap-add (k3_stream): per owned row pair the (patch, row pair) items are
// grouped by corner column (colour order inside a group); the kernel needs the groups of a row pair
// to form one chain cx, cx + P/2, cx + P, ... that covers [0, W).  Chains are cut into `chunks`
// pieces for parallelism; teams of one warp must walk identically shaped tasks, so tasks are packed
// `tpw` at a time and padded with idle tasks where the shape changes.
struct StreamTables {
  std::vector<StreamTask> tasks;
  std::vector<unsigned> codes;
  int n_warp_items = 0;
  int chunks = 0;              // chunks per chain
  bool ok = false;
};

StreamTables build_stream_tables(const std::vector<int2>& corners, const std::vector<int>& colours, int P, int W,
                                 int row_begin, int row_end, int tpw, long long team_slots, int max_batch) {
  StreamTables st;
  const int half = P / 2;
  if (corners.empty() || row_end <= row_begin) return st;
  const int parity = ((corners[0].x % 2) + 2) % 2;
  for (const int2& c : corners)
    if (((c.x % 2) + 2) % 2 != parity) return st;
  struct Entry { int item, colour, cx; };
  const int y_start = row_begin - ((((row_begin - parity) % 2) + 2) % 2);
  const int n_rp = (row_end - y_start + 1) / 2;
  std::vector<std::vector<Entry>> bucket(n_rp);
  for (size_t a = 0; a < corners.size(); ++a) {
    const int2 c = corners[a];
    if (c.y + P <= 0 || c.y >= W) continue;
    for (int pair = 0; pair < half; ++pair) {
      const int y = c.x + 2 * pair;
      if (y + 1 < row_begin || y >= row_end) continue;
      bucket[(y - y_start) / 2].push_back({(int)a * half + pair, colours[a], c.y});
    }
  }
  struct Group { int cx; std::vector<int> items; };
  std::vector<std::vector<Group>> chains(n_rp);
  size_t min_groups = SIZE_MAX;
  for (int rp = 0; rp < n_rp; ++rp) {
    auto& b = bucket[rp];
    if (b.empty()) return st;
    std::stable_sort(b.begin(), b.end(), [](const Entry& u, const Entry& v) {
      return u.cx != v.cx ? u.cx < v.cx : u.colour < v.colour;
    });
    auto& ch = chains[rp];
    for (const Entry& e : b) {
      if (ch.empty() || ch.back().cx != e.cx) ch.push_back({e.cx, {}});
      ch.back().items.push_back(e.item);
    }
    for (size_t i = 1; i < ch.size(); ++i)
      if (ch[i].cx != ch[i - 1].cx + half) return st;
    if (ch.front().cx > 0 || ch.back().cx + P < W) return st;
    min_groups = std::min(min_groups, ch.size());
  }
  // chunks per chain.  A chunk that does not start its chain recomputes one seam group, so c chunks cost a team
  // ceil(groups / c) + 1 transforms per task, and the launch takes ceil(tasks / teams) rounds of them: pick the c
  // that minimises the product (small launches want many short tasks, large ones whole chains).
  long long chunks = 1;
  const long long whole = (long long)n_rp * std::max(max_batch, 1);
  if (team_slots > 0) {
    long long best = LLONG_MAX;
    for (long long c = 1; c <= (long long)min_groups; ++c) {
      const long long per_task = ((long long)min_groups + c - 1) / c + (c > 1 ? 1 : 0);
      const long long rounds = (whole * c + team_slots - 1) / team_slots;
      if (per_task * rounds < best) { best = per_task * rounds; chunks = c; }
    }
  }
  std::vector<std::vector<int>> shape;        // per task: items per computed group
  for (long long chn = 0; chn < chunks; ++chn) {
    for (int rp = 0; rp < n_rp; ++rp) {
      const auto& ch = chains[rp];
      const size_t n_g = ch.size();
      const size_t gb = n_g * chn / chunks, ge = n_g * (chn + 1) / chunks;
      if (gb >= ge) continue;
      const size_t g0 = gb > 0 ? gb - 1 : 0;
      StreamTask t{};
      t.y = y_start + 2 * rp;
      t.cx0 = ch[g0].cx;
      t.item_begin = (int)st.codes.size();
      t.flags = (gb > 0 ? TASK_SEAM : 0) | (ge == n_g ? TASK_LAST : 0);
      std::vector<int> sh;
      for (size_t gi = g0; gi < ge; ++gi) {
        for (size_t k = 0; k < ch[gi].items.size(); ++k)
          st.codes.push_back((unsigned)ch[gi].items[k] | (k + 1 == ch[gi].items.size() ? ITEM_LAST_OF_GROUP : 0u));
        sh.push_back((int)ch[gi].items.size());
      }
      t.n_steps = (int)st.codes.size() - t.item_begin;
      // pack: a warp item holds `tpw` tasks of one shape
      const size_t fill = st.tasks.size() % tpw;
      if (fill != 0 && shape.back() != sh)
        for (size_t k = fill; k < (size_t)tpw; ++k) { st.tasks.push_back(StreamTask{}); shape.push_back(sh); }
      st.tasks.push_back(t);
      shape.push_back(sh);
    }
  }
  while (st.tasks.size() % tpw) st.tasks.push_back(StreamTask{});
  st.n_warp_items = (int)(st.tasks.size() / tpw);
  st.chunks = (int)chunks;
  st.ok = st.n_warp_items > 0;
  return st;
}
}  // namespace

struct rpsf_transform {
  int device = 0, P = 0, n = 0, dtype = 0;
  const Ops* ops = nullptr;
  std::vector<int2> corners;       // (row, col)
  std::vector<int> colour;         // greedy colouring in list order
  int n_colours = 0;
  void* tw = nullptr;
  void* win = nullptr;
  void* kmain = nullptr;           // private kernel layout of the KEPT patches, in list order
  void* knyq = nullptr;
  std::vector<int> kslot;          // patch -> index into kmain / knyq, or -1 (no kernel on this device: row-slab shards)
  int n_kept = 0;
  // patch sizes without a native FFT length run embedded in P = the next power of two >= 2 * win_len - 1
  // (embed_transfer_kernel); win_len == P otherwise
  int win_len = 0;
  bool own_win = false;            // the window table belongs to this transform (embedded sizes), not to the shared cache
  bool has_kernel = false;
  int sm_count = 148;
  // conj of kmain / knyq: the transfer kernel of the transpose (rpsf_plan_create_adjoint); allocated at the first
  // adjoint plan, refreshed by every rpsf_transform_set_kernel after that
  void* kconj_main = nullptr;
  void* kconj_nyq = nullptr;
  // stream order of the transform's device state (the kernel layouts above, and the workspaces, boxes and scratch of
  // its plans): recorded after the last launch of every call that touches it, on that call's stream (OrderedCall)
  std::mutex order_mu;
  cudaEvent_t order_ev = nullptr;
  cudaStream_t order_stream = nullptr;   // the stream order_ev was last recorded on
  bool order_recorded = false;
  // CUDA graphs: a capture makes order_ev an external dependency of the graph, so replays record it without the host
  // knowing; once captured, every eager call waits for it.  capture_ev orders the calls inside one capture (capture_id).
  bool captured = false;
  cudaEvent_t capture_ev = nullptr;
  unsigned long long capture_id = 0;
  bool capture_recorded = false;
  // embedded patch sizes: the (M, P) embedding matrix of set_kernel_on, uploaded at the first layout
  void* embed_A = nullptr;
};

namespace {
// Every entry point that reads or writes the transform's device state runs its launches between the two halves of an
// OrderedCall on its stream.  The first half makes the stream wait for the last call's record when that call ran on
// another stream (a call on the same stream is already behind it); the second records the event after this call's
// launches.  So a call sees the kernel laid out by the calls issued before it, and no two calls use one plan's
// workspace at once, whatever streams they use; a call on the stream of the previous one pays only the record.
// cudaStreamPerThread names a different stream on every thread, so it always waits.  The mutex keeps the bookkeeping
// whole for C callers that share a transform across threads.
//
// On a capturing stream the event becomes an external dependency of the graph: an external wait at the start (each
// replay waits for the calls issued before its launch) and an external record at the end (calls issued after the launch
// are ordered behind the replay).  A replay runs no library code, so the host cannot know which stream recorded the
// event last: once a transform has been captured, every eager call waits for it.  Calls inside one capture are also
// ordered among themselves through capture_ev, an ordinary record / wait pair that becomes a graph edge.
struct OrderedCall {
  rpsf_transform* t;
  cudaStream_t s;
  bool capturing = false;
  unsigned long long capture_id = 0;
  int begin() {
    capturing = stream_capturing(s, &capture_id) != 0;
    std::lock_guard<std::mutex> lock(t->order_mu);
    if (capturing) {
      note_capture(s);
      cudaError_t e = cudaStreamWaitEvent(s, t->order_ev, cudaEventWaitExternal);
      if (e == cudaSuccess && t->capture_recorded && t->capture_id == capture_id) e = cudaStreamWaitEvent(s, t->capture_ev, 0);
      if (e != cudaSuccess) return fail(RPSF_E_CUDA, "ordering a captured call after the transform's last call failed: %s", cudaGetErrorString(e));
      t->captured = true;
      t_capturing = true;
      return RPSF_OK;
    }
    forget_capture(s);
    if (t->order_recorded && (t->captured || s != t->order_stream || s == cudaStreamPerThread)) {
      const cudaError_t e = cudaStreamWaitEvent(s, t->order_ev, 0);
      if (e != cudaSuccess) return fail(RPSF_E_CUDA, "ordering after the transform's last call failed: %s", cudaGetErrorString(e));
    }
    return RPSF_OK;
  }
  // `rc`: the status of the launches; the record is made whatever it is, so that what was launched is ordered too
  int end(int rc) {
    std::lock_guard<std::mutex> lock(t->order_mu);
    if (capturing) {
      t_capturing = false;
      cudaError_t e = cudaEventRecordWithFlags(t->order_ev, s, cudaEventRecordExternal);
      if (e == cudaSuccess) e = cudaEventRecord(t->capture_ev, s);
      if (e != cudaSuccess) return rc ? rc : fail(RPSF_E_CUDA, "recording the transform's order event in a capture failed: %s", cudaGetErrorString(e));
      t->capture_id = capture_id;
      t->capture_recorded = true;
      t->order_recorded = true;           // replays record it: eager calls after them must wait
      return rc;
    }
    const cudaError_t e = cudaEventRecord(t->order_ev, s);
    if (e != cudaSuccess) return rc ? rc : fail(RPSF_E_CUDA, "recording the transform's order event failed: %s", cudaGetErrorString(e));
    t->order_stream = s;
    t->order_recorded = true;
    return rc;
  }
};

// body() between the two halves of an OrderedCall on `s`, with the transform's device current
template <typename F>
int ordered(rpsf_transform* t, cudaStream_t s, F&& body) {
  DeviceGuard guard(t->device);
  if (!guard.ok) return fail(RPSF_E_CUDA, "cannot select CUDA device %d", t->device);
  OrderedCall call{t, s};
  if (int rc = call.begin()) return rc;
  return call.end(body());
}

// kconj_* = conj(kmain / knyq), stream-ordered after whatever wrote kmain on `s`
int refresh_conj_kernel(rpsf_transform* t, cudaStream_t s) {
  if (!t->kconj_main || t->n_kept == 0) return RPSF_OK;
  const long long main_reals = (long long)t->n_kept * t->P * (t->P / 2) * 2, nyq_reals = (long long)t->n_kept * t->P * 2;
  const unsigned blocks = (unsigned)t->sm_count * 8;
  if (t->dtype == RPSF_F32) {
    conj_spectrum<float><<<blocks, 256, 0, s>>>((const float*)t->kmain, (float*)t->kconj_main, main_reals);
    conj_spectrum<float><<<blocks, 256, 0, s>>>((const float*)t->knyq, (float*)t->kconj_nyq, nyq_reals);
  } else {
    conj_spectrum<double><<<blocks, 256, 0, s>>>((const double*)t->kmain, (double*)t->kconj_main, main_reals);
    conj_spectrum<double><<<blocks, 256, 0, s>>>((const double*)t->knyq, (double*)t->kconj_nyq, nyq_reals);
  }
  g_launches.fetch_add(2, std::memory_order_relaxed);
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? RPSF_OK : fail(RPSF_E_CUDA, "conjugate kernel launch failed: %s", cudaGetErrorString(e));
}
}  // namespace

// The row pass (K1) and overlap-add (K3) kernels of a plan.  The overlap-add values are what rpsf_plan_info reports.
enum class K1Kernel { plain, bulk };
enum class Overlap { phases = 0, gather = 1, stream = 2 };

struct rpsf_plan {
  rpsf_transform* tr = nullptr;
  int H = 0, W = 0, pad_mode = 0, row_begin = 0, row_end = 0, max_batch = 1;
  int n_active = 0;
  int* active_dev = nullptr;       // active index -> kernel slot of the patch (rpsf_transform::kslot)
  std::vector<int> active_host;    // active index -> patch index (rpsf_kernel_gradient pairs two plans by it)
  int2* corners_dev = nullptr;     // per active patch
  std::vector<int*> items_dev;     // per colour: active*P/2 + pair
  std::vector<int> n_items;
  bool colour0_covers = false;
  // single-launch overlap-add (row-pair gather); falls back to colour phases when patch corner
  // rows do not share one parity or there are more than 15 colours
  bool gather = false;
  RowTile* tiles_dev = nullptr;
  RowGroup* groups_dev = nullptr;
  int* gitems_dev = nullptr;
  int n_tiles = 0, teams = 0, seg_w = 0;
  bool stream_ok = false;      // every owned row pair is a chain of half-overlapping groups covering [0, W)
  StreamTask* stasks_dev = nullptr;
  unsigned* scodes_dev = nullptr;
  int n_warp_items = 0;
  int stream_chunks = 0;       // chunks per chain of the streaming tables
  // the kernels apply runs: chosen by plan_build from the geometry (rpsf_plan_set_overlap_mode and
  // rpsf_plan_set_gather_mode let tests pick the others)
  K1Kernel k1 = K1Kernel::bulk;
  Overlap overlap = Overlap::phases;
  // workspace, allocated at the first apply: the spectrum of every active patch ([frame][active][P][P/2], what the
  // column pass writes and the overlap-add reads) at offset 0, then the band buffer the row pass writes
  // (rpsf_bands.cuh) at band_offset
  void* workspace = nullptr;
  size_t workspace_bytes = 0, band_offset = 0;
  BandItem* band_items_dev = nullptr;
  int* patch_row_dev = nullptr;
  int n_band_items = 0, band_frame_rows = 0;
  int img_lo = 0, img_hi = 0;      // resident frame rows needed: [img_lo, img_hi)
  // host path: a ring of HOST_SLOTS chunk buffers so the upload of chunk i+1, the kernels of
  // chunk i and the download of chunk i-1 run concurrently on three streams (two copy engines)
  static constexpr int HOST_SLOTS = 3;
  cudaStream_t s_in = nullptr, s_comp = nullptr, s_out = nullptr;
  cudaEvent_t ev_in[HOST_SLOTS] = {}, ev_comp[HOST_SLOTS] = {}, ev_out[HOST_SLOTS] = {};
  void* d_in_raw[HOST_SLOTS] = {}; size_t d_in_raw_bytes = 0;
  void* h_stage[HOST_SLOTS] = {}; size_t h_stage_bytes = 0;   // pinned staging of pageable input chunks
  void* d_in[HOST_SLOTS] = {};
  void* d_out[HOST_SLOTS] = {};
  void* d_out_conv[HOST_SLOTS] = {}; size_t d_out_conv_bytes = 0;
  // saturation branch (transform.py:125-138,171-172); threshold = +inf disables it
  double sat_threshold = INFINITY;
  int sat_dilation = 1, sat_width = 7;
  void* sat_pf = nullptr;                 // [max_batch][Hp][Wp] padded frames, compute dtype
  unsigned char* sat_mask[2] = {nullptr, nullptr};
  int* sat_list = nullptr;                // [max_batch][Hp*Wp] raster-ordered masked pixels
  int* sat_rows = nullptr;                // [max_batch][Hp+1] row offsets, total last
  int* sat_flags = nullptr;               // [2*max_batch]: any-masked flags, fill tickets
  // fused slab gather: peer buffers K3 stores to as well (same layout as `out`)
  std::vector<void*> mirrors;
  // transpose (rpsf_plan_create_adjoint): this plan is the forward plan of the box [box_y0, box_y0 + H) x
  // [box_x0, box_x0 + W) of the frame coordinates; rpsf_apply copies the frame of output gradients into box_in (zero
  // margins), runs the three kernels with the conjugated transfer kernel into box_out and folds box_out onto the
  // frame (fold_pad_adjoint)
  bool adjoint = false;
  int frame_H = 0, frame_W = 0, box_y0 = 0, box_x0 = 0;
  int frame_pad_mode = 0;             // the pad mode of the forward map this plan transposes
  long long box_pitch = 0;            // elements, a multiple of 16 bytes (K1's bulk row copies)
  void* box_in = nullptr; void* box_out = nullptr;
  int* fold_rows = nullptr;           // [frame_H + 1 offsets | box row indices], CSR preimages of the row pad map
  int* fold_cols = nullptr;           // the same for columns
  // masked transpose (rpsf_apply_masked on an adjoint plan): the same preimages over the whole padded frame (the fill
  // carries gradient out of the box), and, allocated at the first masked call, the padded-size buffers: v / shares in
  // sat_pf, the combined gradient in mask_out, contributor counts in mask_count (state, list, rows and tickets: sat_*)
  int* fold_prows = nullptr;
  int* fold_pcols = nullptr;
  void* mask_out = nullptr;
  int* mask_count = nullptr;
  // per-stage timing (bench only)
  bool timing = false;
  std::vector<cudaEvent_t> events;   // 4 per recorded apply call
  size_t events_used = 0;
  // the transform stack of a plan made by rpsf_plan_create_stack (null otherwise): the workspace holds the spectra of
  // stack->m * max_batch frames ([kernel][frame]) and the row bands of max_batch frames; only rpsf_apply_stack runs it
  rpsf_stack* stack = nullptr;
  // its column pass: 0 = k2_stack where it exists (native patch sizes whose stage ring fits), 1 = the per-kernel K2
  // (rpsf_plan_set_stack_mode, a test and benchmark hook)
  int stack_mode = 0;
};

// M transfer kernels on one set of patch corners: `t` holds the geometry, and its kmain / knyq hold kernel m's layout at
// slot m (n_kept patches each).  `t` is never exposed, so only stack calls touch it.
struct rpsf_stack {
  rpsf_transform* t = nullptr;
  int m = 0;
  std::vector<char> loaded;          // kernel m has been laid out
  size_t main_bytes = 0, nyq_bytes = 0;   // bytes of one kernel's kmain / knyq
};

extern "C" {

int rpsf_abi_version(void) { return RPSF_ABI_VERSION; }
const char* rpsf_last_error(void) { return g_error.c_str(); }
int rpsf_patch_size_supported(int P) { return ops_for(P) ? 1 : (embedded_length(P) && ops_for(embedded_length(P))) ? 2 : 0; }
int64_t rpsf_launch_count(void) { return g_launches.load(); }
int rpsf_pad_index(int i, int n, int pad_mode) { return n > 0 ? pad_index(i, n, pad_mode) : -1; }

int rpsf_transform_create_subset(rpsf_transform** out, const int32_t* coords, int n, int P, int dtype, int device,
                                 const uint8_t* keep) {
  if (!out || (!coords && n > 0) || n < 0) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (dtype != RPSF_F32 && dtype != RPSF_F64) return fail(RPSF_E_UNSUPPORTED, "compute dtype must be f32 or f64");
  REFUSE_IN_CAPTURE("rpsf_transform_create");
  const int win_len = P;
  const Ops* ops = ops_for(P);
  if (!ops) {
    P = embedded_length(win_len);                  // run embedded in the next power of two >= 2 P - 1
    ops = P ? ops_for(P) : nullptr;
  }
  if (!ops)
    return fail(RPSF_E_UNSUPPORTED, "patch size %d has no device path (supported: powers of two 16..512 natively, any size "
                "from 2 to 256 embedded in the next power of two >= 2 P - 1)", win_len);
  DeviceGuard guard(device);
  if (!guard.ok) return fail(RPSF_E_CUDA, "cannot select CUDA device %d", device);
  int e = ops->init();
  if (e) return fail(RPSF_E_CUDA, "kernel attribute setup failed: %s", cudaGetErrorString((cudaError_t)e));
  auto* t = new rpsf_transform;
  t->device = device; t->P = P; t->n = n; t->dtype = dtype; t->ops = ops; t->win_len = win_len;
  t->sm_count = sm_count_of(device);
  if (cudaEventCreateWithFlags(&t->order_ev, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&t->capture_ev, cudaEventDisableTiming) != cudaSuccess) {
    const cudaError_t ce = cudaGetLastError();
    if (t->order_ev) cudaEventDestroy(t->order_ev);
    delete t;
    return fail(RPSF_E_CUDA, "cannot create the transform's order event: %s", cudaGetErrorString(ce));
  }
  t->corners.resize(n);
  for (int i = 0; i < n; ++i) t->corners[i] = make_int2(coords[2 * i], coords[2 * i + 1]);
  // Greedy colouring in list order: same-colour patches are pairwise disjoint.  For
  // calculate_covering (util.py:27-53) this recovers its four grids, in its order.
  t->colour.assign(n, 0);
  {
    std::vector<std::vector<int>> members;
    for (int i = 0; i < n; ++i) {
      int c = 0;
      for (;; ++c) {
        if (c == (int)members.size()) { members.emplace_back(); break; }
        bool clash = false;
        for (int j : members[c]) {
          // (the footprint of a patch is its true size: an embedded transform's FFT length P is larger)
          if (std::abs(t->corners[i].x - t->corners[j].x) < win_len && std::abs(t->corners[i].y - t->corners[j].y) < win_len) {
            clash = true; break;
          }
        }
        if (!clash) break;
      }
      members[c].push_back(i);
      t->colour[i] = c;
    }
    t->n_colours = (int)members.size();
  }
  int rc = shared_tables(P, dtype, device, &t->tw, &t->win);     // owned by the library, not by the transform
  if (rc) { rpsf_transform_destroy(t); return rc; }
  if (win_len != P) {
    // the window of the true patch size, zero beyond it (transform.py:151-154 with P = win_len)
    const double pi = 3.14159265358979323846264338327950288;
    std::vector<double> w64(P, 0.0);
    for (int i = 0; i < win_len; ++i) w64[i] = std::sin((i + 0.5) * (pi / win_len));
    const size_t rsz = real_size(dtype);
    void* wdev = nullptr;
    if (cudaMalloc(&wdev, P * rsz) != cudaSuccess) { rpsf_transform_destroy(t); return fail(RPSF_E_CUDA, "out of device memory for the window table"); }
    cudaError_t ce;
    if (dtype == RPSF_F32) {
      std::vector<float> w32(w64.begin(), w64.end());
      ce = cudaMemcpy(wdev, w32.data(), P * rsz, cudaMemcpyHostToDevice);
    } else {
      ce = cudaMemcpy(wdev, w64.data(), P * rsz, cudaMemcpyHostToDevice);
    }
    if (ce != cudaSuccess) { cudaFree(wdev); rpsf_transform_destroy(t); return fail(RPSF_E_CUDA, "window upload failed: %s", cudaGetErrorString(ce)); }
    t->win = wdev; t->own_win = true;
  }
  const size_t cs = 2 * real_size(dtype);
  t->kslot.assign(n, -1);
  for (int i = 0; i < n; ++i)
    if (!keep || keep[i]) t->kslot[i] = t->n_kept++;
  if (t->n_kept > 0) {
    if (cudaMalloc(&t->kmain, (size_t)t->n_kept * P * (P / 2) * cs) != cudaSuccess ||
        cudaMalloc(&t->knyq, (size_t)t->n_kept * P * cs) != cudaSuccess) {
      rpsf_transform_destroy(t);
      return fail(RPSF_E_CUDA, "out of device memory for the transfer kernel (%d patches of %d)", t->n_kept, P);
    }
  }
  *out = t;
  return RPSF_OK;
}

int rpsf_transform_create(rpsf_transform** out, const int32_t* coords, int n, int P, int dtype, int device) {
  return rpsf_transform_create_subset(out, coords, n, P, dtype, device, nullptr);
}

int rpsf_transform_destroy(rpsf_transform* t) {
  if (!t) return RPSF_OK;
  DeviceGuard guard(t->device);
  cudaFree(t->kmain); cudaFree(t->knyq);
  cudaFree(t->kconj_main); cudaFree(t->kconj_nyq);
  if (t->own_win) cudaFree(t->win);
  cudaFree(t->embed_A);
  if (t->order_ev) cudaEventDestroy(t->order_ev);
  if (t->capture_ev) cudaEventDestroy(t->capture_ev);
  delete t;
  return RPSF_OK;
}

int rpsf_transform_num_colours(const rpsf_transform* t) { return t ? t->n_colours : 0; }

int rpsf_transform_order(rpsf_transform* t, void* stream) {
  if (!t) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  return ordered(t, (cudaStream_t)stream, []() -> int { return RPSF_OK; });
}

}  // extern "C"

namespace {
// the (M, P) embedding matrix of an embedded patch size, uploaded once per transform (at its first kernel layout, which
// is never captured): A[u][p] = (1/P) sum_{i=-(P-1)}^{P-1} exp(2 pi i (p/P - u/M) i), stored complex with a zero
// imaginary part
int upload_embed_matrix(rpsf_transform* t) {
  if (t->embed_A) return RPSF_OK;
  const int P = t->win_len, M = t->P;
  std::vector<double> A(2 * (size_t)M * P);
  const double two_pi = 6.283185307179586476925286766559;
  for (int u = 0; u < M; ++u)
    for (int p = 0; p < P; ++p) {
      // the phase reduced exactly: (p M - u P) i mod (P M) = sin((2P-1) theta/2) / sin(theta/2) / P with theta/2 = pi r /
      // (P M), r = (p M - u P) mod (P M); real, because the terms i and -i are conjugates
      const long long den = (long long)P * M;
      long long r = ((long long)p * M - (long long)u * P) % den; if (r < 0) r += den;
      double re = double(2 * P - 1);
      if (r != 0) {
        const long long rn = ((2LL * P - 1) * r) % (2 * den);         // numerator angle, reduced mod 2 pi
        re = std::sin(0.5 * two_pi * double(rn) / double(den)) / std::sin(0.5 * two_pi * double(r) / double(den));
      }
      A[2 * ((size_t)u * P + p)] = re / P; A[2 * ((size_t)u * P + p) + 1] = 0.0;
    }
  void* dA = nullptr;
  if (cudaMalloc(&dA, sizeof(double2) * M * P) != cudaSuccess) {
    cudaGetLastError();
    return fail(RPSF_E_CUDA, "out of device memory for the embedding matrix (%d x %d)", M, P);
  }
  const cudaError_t e = cudaMemcpy(dA, A.data(), sizeof(double2) * M * P, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { cudaFree(dA); return fail(RPSF_E_CUDA, "embedding matrix upload failed: %s", cudaGetErrorString(e)); }
  t->embed_A = dA;
  return RPSF_OK;
}

// the layout of rpsf_transform_set_kernel into `kmain` / `knyq` (the transform's own, or a stack's slot), stream-ordered
// on `s`; on a capturing stream it allocates only with cudaMallocAsync (allocation nodes of the graph)
int layout_kernel(rpsf_transform* t, const void* kernel_full, int kernel_dtype, void* kmain, void* knyq, cudaStream_t s) {
  if (t->n_kept > 0 && t->win_len != t->P) {
    // embedded patch size: K (n, P, P) -> K' (n, M, M) = A K A^T in double (rpsf_kernels.cuh), then the usual layout
    const int P = t->win_len, M = t->P;
    if (!t->embed_A && t_capturing) return refuse_capture("the first kernel layout of an embedded patch size");
    if (int rc = upload_embed_matrix(t)) return rc;
    const double2* dA = (const double2*)t->embed_A;
    double2 *dT = nullptr, *dK = nullptr;
    auto release = [&]() { for (void* q : {(void*)dT, (void*)dK}) if (q) cudaFreeAsync(q, s); };
    const size_t n = (size_t)t->n_kept;
    if (cudaMallocAsync((void**)&dT, sizeof(double2) * n * M * P, s) != cudaSuccess ||
        cudaMallocAsync((void**)&dK, sizeof(double2) * n * M * M, s) != cudaSuccess) {
      release(); cudaGetLastError();
      return fail(RPSF_E_CUDA, "out of device memory embedding %zu kernels of %d in %d", n, P, M);
    }
    const unsigned blocks = (unsigned)t->sm_count * 16;
    if (kernel_dtype == RPSF_F32) embed_pass1<float2><<<blocks, 256, 0, s>>>((const float2*)kernel_full, dA, dT, (int)n, P, M);
    else embed_pass1<double2><<<blocks, 256, 0, s>>>((const double2*)kernel_full, dA, dT, (int)n, P, M);
    LAUNCH((int)cudaGetLastError());
    embed_pass2<double2><<<blocks, 256, 0, s>>>(dT, dA, dK, (int)n, P, M);
    LAUNCH((int)cudaGetLastError());
    int e = t->ops->prep(t->dtype, RPSF_F64, dK, kmain, knyq, t->n_kept, s);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    release();
    if (e) return fail(RPSF_E_CUDA, "kernel layout launch failed: %s", cudaGetErrorString((cudaError_t)e));
    return RPSF_OK;
  }
  if (t->n_kept > 0) LAUNCH(t->ops->prep(t->dtype, kernel_dtype, kernel_full, kmain, knyq, t->n_kept, s));
  return RPSF_OK;
}

int set_kernel_on(rpsf_transform* t, const void* kernel_full, int kernel_dtype, cudaStream_t s) {
  if (int rc = layout_kernel(t, kernel_full, kernel_dtype, t->kmain, t->knyq, s)) return rc;
  t->has_kernel = true;
  return refresh_conj_kernel(t, s);
}
}  // namespace

extern "C" {

int rpsf_transform_set_kernel(rpsf_transform* t, const void* kernel_full, int kernel_dtype, void* stream) {
  if (!t || (!kernel_full && t->n_kept > 0)) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (kernel_dtype != RPSF_F32 && kernel_dtype != RPSF_F64)
    return fail(RPSF_E_UNSUPPORTED, "kernel dtype must be complex64 (RPSF_F32) or complex128 (RPSF_F64)");
  cudaStream_t s = (cudaStream_t)stream;
  return ordered(t, s, [&]() -> int { return set_kernel_on(t, kernel_full, kernel_dtype, s); });
}

int rpsf_stack_create(rpsf_stack** out, const int32_t* coords, int n, int P, int dtype, int device, int n_kernels) {
  if (!out) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (n_kernels < 1) return fail(RPSF_E_INVALID_ARGUMENT, "a stack needs at least one kernel, got %d", n_kernels);
  rpsf_transform* t = nullptr;
  if (int rc = rpsf_transform_create(&t, coords, n, P, dtype, device)) return rc;
  auto* st = new rpsf_stack;
  st->t = t; st->m = n_kernels;
  st->loaded.assign(n_kernels, 0);
  const size_t cs = 2 * real_size(dtype);
  st->main_bytes = (size_t)t->n_kept * t->P * (t->P / 2) * cs;
  st->nyq_bytes = (size_t)t->n_kept * t->P * cs;
  if (n_kernels > 1 && t->n_kept > 0) {
    DeviceGuard guard(device);
    cudaFree(t->kmain); cudaFree(t->knyq);
    t->kmain = t->knyq = nullptr;
    if (cudaMalloc(&t->kmain, st->main_bytes * n_kernels) != cudaSuccess ||
        cudaMalloc(&t->knyq, st->nyq_bytes * n_kernels) != cudaSuccess) {
      cudaGetLastError();
      rpsf_stack_destroy(st);
      return fail(RPSF_E_CUDA, "out of device memory for %d transfer kernels (%d patches of %d)", n_kernels, n, P);
    }
  }
  *out = st;
  return RPSF_OK;
}

int rpsf_stack_set_kernel(rpsf_stack* st, int index, const void* kernel_full, int kernel_dtype, void* stream) {
  if (!st || (!kernel_full && st->t->n_kept > 0)) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (index < 0 || index >= st->m) return fail(RPSF_E_INVALID_ARGUMENT, "kernel %d outside [0, %d)", index, st->m);
  if (kernel_dtype != RPSF_F32 && kernel_dtype != RPSF_F64)
    return fail(RPSF_E_UNSUPPORTED, "kernel dtype must be complex64 (RPSF_F32) or complex128 (RPSF_F64)");
  rpsf_transform* t = st->t;
  cudaStream_t s = (cudaStream_t)stream;
  return ordered(t, s, [&]() -> int {
    void* kmain = t->kmain ? (char*)t->kmain + st->main_bytes * index : nullptr;
    void* knyq = t->knyq ? (char*)t->knyq + st->nyq_bytes * index : nullptr;
    if (int rc = layout_kernel(t, kernel_full, kernel_dtype, kmain, knyq, s)) return rc;
    st->loaded[index] = 1;
    return RPSF_OK;
  });
}

int rpsf_stack_destroy(rpsf_stack* st) {
  if (!st) return RPSF_OK;
  rpsf_transform_destroy(st->t);
  delete st;
  return RPSF_OK;
}

}  // extern "C"

namespace {
// rpsf_construct_kernel (ae == nullptr: the host scalars alpha, epsilon) and rpsf_construct_kernel_dev (ae: two device
// doubles); launches only, so a capture may hold it
int construct_kernel(const void* S, const void* Tg, void* K, int64_t count, int dtype, double alpha, double epsilon,
                     const double* ae, int device, void* stream) {
  if (count < 0 || (count > 0 && (!S || !Tg || !K))) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (dtype != RPSF_F32 && dtype != RPSF_F64) return fail(RPSF_E_UNSUPPORTED, "dtype must be f32 or f64");
  if (count == 0) return RPSF_OK;
  DeviceGuard guard(device);
  const unsigned blocks = (unsigned)std::min<long long>((count + 255) / 256, (long long)sm_count_of(device) * 16);
  const cudaStream_t s = (cudaStream_t)stream;
  if (dtype == RPSF_F32) {
    if (ae) construct_transfer_kernel<float, true><<<blocks, 256, 0, s>>>((const float2*)S, (const float2*)Tg, (float2*)K,
                                                                        count, 0.f, 0.f, ae);
    else construct_transfer_kernel<float><<<blocks, 256, 0, s>>>((const float2*)S, (const float2*)Tg, (float2*)K, count,
                                                                 (float)alpha, (float)epsilon);
  } else {
    if (ae) construct_transfer_kernel<double, true><<<blocks, 256, 0, s>>>((const double2*)S, (const double2*)Tg,
                                                                         (double2*)K, count, 0.0, 0.0, ae);
    else construct_transfer_kernel<double><<<blocks, 256, 0, s>>>((const double2*)S, (const double2*)Tg, (double2*)K,
                                                                  count, alpha, epsilon);
  }
  LAUNCH((int)cudaGetLastError());
  return RPSF_OK;
}

// rpsf_construct_kernel_backward and its _dev form (ae: alpha and epsilon as two device doubles)
int construct_kernel_backward(const void* S, const void* Tg, const void* G, int64_t count, int dtype, double alpha,
                              double epsilon, const double* ae, void* source_grad, void* target_grad,
                              double* alpha_epsilon_grad, int device, void* stream) {
  if (count < 0 || (count > 0 && (!S || !Tg || !G))) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (dtype != RPSF_F32 && dtype != RPSF_F64) return fail(RPSF_E_UNSUPPORTED, "dtype must be f32 or f64");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(RPSF_E_CUDA, "cannot select CUDA device %d", device);
  cudaStream_t s = (cudaStream_t)stream;
  if (count == 0) {
    if (alpha_epsilon_grad) CU(cudaMemsetAsync(alpha_epsilon_grad, 0, 2 * sizeof(double), s));
    return RPSF_OK;
  }
  if (!source_grad && !target_grad && !alpha_epsilon_grad) return RPSF_OK;
  const int ctas = (int)std::min<long long>((count + CGRAD_THREADS - 1) / CGRAD_THREADS, CGRAD_MAX_CTAS);
  double2* partial = nullptr;
  if (alpha_epsilon_grad) {
    cudaError_t e = cudaMallocAsync((void**)&partial, sizeof(double2) * ctas, s);
    if (e != cudaSuccess) return fail(RPSF_E_CUDA, "cudaMallocAsync of %d partial sums failed: %s", ctas, cudaGetErrorString(e));
  }
  if (dtype == RPSF_F32) {
    if (ae)
      construct_transfer_kernel_backward<float, true><<<ctas, CGRAD_THREADS, 0, s>>>(
          (const float2*)S, (const float2*)Tg, (const float2*)G, count, 0.f, 0.f, (float2*)source_grad,
          (float2*)target_grad, partial, ae);
    else
      construct_transfer_kernel_backward<float><<<ctas, CGRAD_THREADS, 0, s>>>(
          (const float2*)S, (const float2*)Tg, (const float2*)G, count, (float)alpha, (float)epsilon, (float2*)source_grad,
          (float2*)target_grad, partial);
  } else {
    if (ae)
      construct_transfer_kernel_backward<double, true><<<ctas, CGRAD_THREADS, 0, s>>>(
          (const double2*)S, (const double2*)Tg, (const double2*)G, count, 0.0, 0.0, (double2*)source_grad,
          (double2*)target_grad, partial, ae);
    else
      construct_transfer_kernel_backward<double><<<ctas, CGRAD_THREADS, 0, s>>>(
          (const double2*)S, (const double2*)Tg, (const double2*)G, count, alpha, epsilon, (double2*)source_grad,
          (double2*)target_grad, partial);
  }
  cudaError_t e = cudaGetLastError();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (e == cudaSuccess && partial) {
    construct_grad_sum<CGRAD_THREADS><<<1, CGRAD_THREADS, 0, s>>>(partial, ctas, alpha_epsilon_grad);
    e = cudaGetLastError();
    g_launches.fetch_add(1, std::memory_order_relaxed);
  }
  if (partial) cudaFreeAsync(partial, s);
  if (e != cudaSuccess) return fail(RPSF_E_CUDA, "construct backward launch failed: %s", cudaGetErrorString(e));
  return RPSF_OK;
}

// rpsf_construct_kernels (host pairs `hp`) and rpsf_construct_kernels_dev (device pairs `dp`): CONSTRUCT_BATCH kernels
// per launch, each launch reading S and T once
int construct_kernels(const void* S, const void* Tg, void* K, int64_t count, int dtype, const double* hp,
                      const double* dp, int n_kernels, int device, void* stream) {
  if (count < 0 || n_kernels < 0 || (count > 0 && n_kernels > 0 && (!S || !Tg || !K || !(hp || dp))))
    return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (dtype != RPSF_F32 && dtype != RPSF_F64) return fail(RPSF_E_UNSUPPORTED, "dtype must be f32 or f64");
  if (count == 0 || n_kernels == 0) return RPSF_OK;
  DeviceGuard guard(device);
  if (!guard.ok) return fail(RPSF_E_CUDA, "cannot select CUDA device %d", device);
  const unsigned blocks = (unsigned)std::min<long long>((count + 255) / 256, (long long)sm_count_of(device) * 16);
  const cudaStream_t s = (cudaStream_t)stream;
  const size_t cs = dtype == RPSF_F32 ? sizeof(float2) : sizeof(double2);
  for (int m0 = 0; m0 < n_kernels; m0 += CONSTRUCT_BATCH) {
    const int mb = std::min(CONSTRUCT_BATCH, n_kernels - m0);
    ConstructPairs pairs{};
    if (hp) std::copy(hp + 2 * (size_t)m0, hp + 2 * (size_t)(m0 + mb), pairs.v);
    const double* dpm = dp ? dp + 2 * (size_t)m0 : nullptr;
    void* Km = (char*)K + (size_t)m0 * (size_t)count * cs;
    if (dtype == RPSF_F32) {
      if (dp) construct_transfer_kernels<float, true><<<blocks, 256, 0, s>>>((const float2*)S, (const float2*)Tg, (float2*)Km,
                                                                           count, mb, pairs, dpm);
      else construct_transfer_kernels<float><<<blocks, 256, 0, s>>>((const float2*)S, (const float2*)Tg, (float2*)Km, count,
                                                                    mb, pairs, nullptr);
    } else {
      if (dp) construct_transfer_kernels<double, true><<<blocks, 256, 0, s>>>((const double2*)S, (const double2*)Tg,
                                                                            (double2*)Km, count, mb, pairs, dpm);
      else construct_transfer_kernels<double><<<blocks, 256, 0, s>>>((const double2*)S, (const double2*)Tg, (double2*)Km,
                                                                     count, mb, pairs, nullptr);
    }
    LAUNCH((int)cudaGetLastError());
  }
  return RPSF_OK;
}
}  // namespace

extern "C" {

int rpsf_construct_kernel(const void* S, const void* Tg, void* K, int64_t count, int dtype, double alpha,
                          double epsilon, int device, void* stream) {
  return construct_kernel(S, Tg, K, count, dtype, alpha, epsilon, nullptr, device, stream);
}

int rpsf_construct_kernel_dev(const void* S, const void* Tg, void* K, int64_t count, int dtype,
                              const double* alpha_epsilon, int device, void* stream) {
  if (!alpha_epsilon) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  return construct_kernel(S, Tg, K, count, dtype, 0.0, 0.0, alpha_epsilon, device, stream);
}

int rpsf_construct_kernels(const void* S, const void* Tg, void* K, int64_t count, int dtype, const double* alpha_epsilon,
                           int n_kernels, int device, void* stream) {
  if (!alpha_epsilon && n_kernels > 0) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  return construct_kernels(S, Tg, K, count, dtype, alpha_epsilon, nullptr, n_kernels, device, stream);
}

int rpsf_construct_kernels_dev(const void* S, const void* Tg, void* K, int64_t count, int dtype,
                               const double* alpha_epsilon, int n_kernels, int device, void* stream) {
  if (!alpha_epsilon && n_kernels > 0) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  return construct_kernels(S, Tg, K, count, dtype, nullptr, alpha_epsilon, n_kernels, device, stream);
}

int rpsf_construct_kernel_backward(const void* S, const void* Tg, const void* G, int64_t count, int dtype, double alpha,
                                   double epsilon, void* source_grad, void* target_grad, double* alpha_epsilon_grad,
                                   int device, void* stream) {
  return construct_kernel_backward(S, Tg, G, count, dtype, alpha, epsilon, nullptr, source_grad, target_grad,
                                   alpha_epsilon_grad, device, stream);
}

int rpsf_construct_kernel_backward_dev(const void* S, const void* Tg, const void* G, int64_t count, int dtype,
                                       const double* alpha_epsilon, void* source_grad, void* target_grad,
                                       double* alpha_epsilon_grad, int device, void* stream) {
  if (!alpha_epsilon) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  return construct_kernel_backward(S, Tg, G, count, dtype, 0.0, 0.0, alpha_epsilon, source_grad, target_grad,
                                   alpha_epsilon_grad, device, stream);
}

int rpsf_psf_fft2_adjoint(const void* spectrum_grad, void* values_grad, int64_t n, int P, int dtype, int device,
                          void* stream) {
  if (n < 0 || (n > 0 && (!spectrum_grad || !values_grad))) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (dtype != RPSF_F32 && dtype != RPSF_F64) return fail(RPSF_E_UNSUPPORTED, "dtype must be f32 or f64");
  const Ops* ops = ops_for(P);
  if (!ops) return fail(RPSF_E_UNSUPPORTED, "the PSF FFT adjoint is implemented for the patch sizes 16, 32, ..., 512, not %d", P);
  if (n == 0) return RPSF_OK;
  DeviceGuard guard(device);
  if (!guard.ok) return fail(RPSF_E_CUDA, "cannot select CUDA device %d", device);
  cudaStream_t s = (cudaStream_t)stream;
  if (!tables_ready(P, dtype, device) && stream_capturing(s)) return refuse_capture("the first rpsf_psf_fft2_adjoint of a patch size");
  int e = ops->init();
  if (e) return fail(RPSF_E_CUDA, "kernel attribute setup failed: %s", cudaGetErrorString((cudaError_t)e));
  void* tw = nullptr; void* win = nullptr;
  int rc = shared_tables(P, dtype, device, &tw, &win);
  if (rc) return rc;
  void* scratch = nullptr;                                        // the complex row spectra, (n, P, P)
  const size_t bytes = 2 * real_size(dtype) * (size_t)n * P * P;
  cudaError_t ce = cudaMallocAsync(&scratch, bytes, s);
  if (ce != cudaSuccess) return fail(RPSF_E_CUDA, "cudaMallocAsync of %zu scratch bytes failed: %s", bytes, cudaGetErrorString(ce));
  e = ops->fft2_adjoint(dtype, spectrum_grad, scratch, values_grad, tw, n, s);
  g_launches.fetch_add(2, std::memory_order_relaxed);
  cudaFreeAsync(scratch, s);
  if (e) return fail(RPSF_E_CUDA, "fft2 adjoint launch failed: %s", cudaGetErrorString((cudaError_t)e));
  return RPSF_OK;
}

int rpsf_psf_fft2(const void* values, void* out, int64_t n, int P, int dtype, int device, void* stream) {
  if (n < 0 || (n > 0 && (!values || !out))) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (dtype != RPSF_F32 && dtype != RPSF_F64) return fail(RPSF_E_UNSUPPORTED, "dtype must be f32 or f64");
  const Ops* ops = ops_for(P);
  if (!ops && (P < 1 || P > 512)) return fail(RPSF_E_UNSUPPORTED, "patch size %d has no device path", P);
  if (n == 0) return RPSF_OK;
  DeviceGuard guard(device);
  if ((!ops || !tables_ready(P, dtype, device)) && stream_capturing((cudaStream_t)stream))
    return refuse_capture(ops ? "the first rpsf_psf_fft2 of a patch size" : "rpsf_psf_fft2 of a patch size without a native FFT length");
  if (!ops) {
    // no native FFT length: separable direct DFT in double (setup cost only, O(P^3) per patch)
    cudaStream_t s = (cudaStream_t)stream;
    std::vector<double> tw(2 * (size_t)P);
    const double two_pi = 6.283185307179586476925286766559;
    for (int m = 0; m < P; ++m) { tw[2 * m] = std::cos(two_pi * m / P); tw[2 * m + 1] = -std::sin(two_pi * m / P); }
    double2 *d_tw = nullptr, *d_tmp = nullptr;
    if (cudaMallocAsync((void**)&d_tw, sizeof(double2) * P, s) != cudaSuccess ||
        cudaMallocAsync((void**)&d_tmp, sizeof(double2) * (size_t)n * P * P, s) != cudaSuccess) {
      if (d_tw) cudaFreeAsync(d_tw, s);
      cudaGetLastError();
      return fail(RPSF_E_CUDA, "out of device memory for the direct DFT of %lld patches of %d", (long long)n, P);
    }
    CU(cudaMemcpyAsync(d_tw, tw.data(), sizeof(double2) * P, cudaMemcpyHostToDevice, s));
    const unsigned blocks = (unsigned)sm_count_of(device) * 16;
    if (dtype == RPSF_F32) dft_rows_direct<float><<<blocks, 256, 0, s>>>((const float*)values, d_tw, d_tmp, n * P, P);
    else dft_rows_direct<double><<<blocks, 256, 0, s>>>((const double*)values, d_tw, d_tmp, n * P, P);
    LAUNCH((int)cudaGetLastError());
    if (dtype == RPSF_F32) dft_cols_direct<float2><<<blocks, 256, 0, s>>>(d_tmp, d_tw, (float2*)out, n, P);
    else dft_cols_direct<double2><<<blocks, 256, 0, s>>>(d_tmp, d_tw, (double2*)out, n, P);
    LAUNCH((int)cudaGetLastError());
    cudaFreeAsync(d_tw, s); cudaFreeAsync(d_tmp, s);
    return RPSF_OK;
  }
  int e = ops->init();
  if (e) return fail(RPSF_E_CUDA, "kernel attribute setup failed: %s", cudaGetErrorString((cudaError_t)e));
  void* tw = nullptr; void* win = nullptr;
  int rc = shared_tables(P, dtype, device, &tw, &win);           // cached per (P, dtype, device): no sync, no free
  if (rc) return rc;
  e = ops->fft2(dtype, dtype, values, out, tw, n, (cudaStream_t)stream);
  g_launches.fetch_add(2, std::memory_order_relaxed);
  if (e) return fail(RPSF_E_CUDA, "fft2 launch failed: %s", cudaGetErrorString((cudaError_t)e));
  return RPSF_OK;
}

int rpsf_average_patches(const double* cutouts, int64_t n_cutouts, int P, const int64_t* cell_offsets,
                         const int32_t* cell_items, int64_t n_cells, int method, double percentile, double* out,
                         int device, void* stream) {
  if (P <= 0 || n_cutouts < 0 || n_cells < 0) return fail(RPSF_E_INVALID_ARGUMENT, "negative size");
  if (n_cells == 0) return RPSF_OK;
  if (!cell_offsets || !out) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  REFUSE_ON_CAPTURING((cudaStream_t)stream, "rpsf_average_patches");
  if (method != RPSF_AVG_MEAN && method != RPSF_AVG_MEDIAN && method != RPSF_AVG_PERCENTILE)
    return fail(RPSF_E_UNSUPPORTED, "unknown averaging method %d", method);
  if (method == RPSF_AVG_PERCENTILE && !(percentile >= 0.0 && percentile <= 100.0))
    return fail(RPSF_E_INVALID_ARGUMENT, "percentile must be in [0, 100]");
  if (method == RPSF_AVG_PERCENTILE && percentile == 50.0) method = RPSF_AVG_MEDIAN;      // builder.py:79-82
  const long long total = cell_offsets[n_cells];
  if (cell_offsets[0] != 0 || total < 0 || (total > 0 && (!cell_items || !cutouts)))
    return fail(RPSF_E_INVALID_ARGUMENT, "bad cell index arrays");
  for (int64_t c = 0; c < n_cells; ++c)
    if (cell_offsets[c + 1] < cell_offsets[c] || cell_offsets[c + 1] - cell_offsets[c] > INT_MAX)
      return fail(RPSF_E_INVALID_ARGUMENT, "cell offsets must be non-decreasing");
  for (long long i = 0; i < total; ++i)
    if (cell_items[i] < 0 || cell_items[i] >= n_cutouts)
      return fail(RPSF_E_INVALID_ARGUMENT, "cell item %lld refers to cutout %d of %lld", i, cell_items[i], (long long)n_cutouts);
  DeviceGuard guard(device);
  if (!guard.ok) return fail(RPSF_E_CUDA, "cannot select CUDA device %d", device);
  cudaStream_t s = (cudaStream_t)stream;
  const int pp = P * P, centre = (P / 2) * P + P / 2;
  const unsigned gx = (unsigned)((pp + AVG_TPB - 1) / AVG_TPB);

  // launch lists: staged classes by stack depth, then the stacks too deep for shared memory
  const int caps[] = {16, AVG_SHALLOW, 64, 128, 256, AVG_MAX_STAGED};
  constexpr int NCLASS = 7;
  std::vector<int> lists[NCLASS];
  std::vector<long long> big_off;
  long long scratch_elems = 0;
  if (method != RPSF_AVG_MEAN)
    for (int64_t c = 0; c < n_cells; ++c) {
      const long long n = cell_offsets[c + 1] - cell_offsets[c];
      int k = 0;
      while (k < NCLASS - 1 && n > caps[k]) ++k;
      lists[k].push_back((int)c);
      if (k == NCLASS - 1) { big_off.push_back(scratch_elems); scratch_elems += (long long)gx * AvgLayout<AVG_SUBS>::STRIDE * n; }
    }
  std::vector<int> cells_flat;
  for (auto& l : lists) cells_flat.insert(cells_flat.end(), l.begin(), l.end());

  long long* d_off = nullptr; int* d_items = nullptr; int* d_cells = nullptr;
  long long* d_big = nullptr; unsigned long long* d_scratch = nullptr;
  // stream-ordered temporaries: freed behind the kernels, no host synchronisation
  auto release = [&]() {
    for (void* ptr : {(void*)d_off, (void*)d_items, (void*)d_cells, (void*)d_big, (void*)d_scratch})
      if (ptr) cudaFreeAsync(ptr, s);
  };
#define AVG_CU(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) { release(); \
    return fail(RPSF_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e_)); } } while (0)
  static_assert(sizeof(long long) == sizeof(int64_t), "offset width");
  AVG_CU(cudaMallocAsync(&d_off, sizeof(long long) * (size_t)(n_cells + 1), s));
  AVG_CU(cudaMemcpyAsync(d_off, cell_offsets, sizeof(long long) * (size_t)(n_cells + 1), cudaMemcpyHostToDevice, s));
  if (total > 0) {
    AVG_CU(cudaMallocAsync(&d_items, sizeof(int) * (size_t)total, s));
    AVG_CU(cudaMemcpyAsync(d_items, cell_items, sizeof(int) * (size_t)total, cudaMemcpyHostToDevice, s));
  }
  if (!cells_flat.empty()) {
    AVG_CU(cudaMallocAsync(&d_cells, sizeof(int) * cells_flat.size(), s));
    AVG_CU(cudaMemcpyAsync(d_cells, cells_flat.data(), sizeof(int) * cells_flat.size(), cudaMemcpyHostToDevice, s));
  }
  if (!big_off.empty()) {
    AVG_CU(cudaMallocAsync(&d_big, sizeof(long long) * big_off.size(), s));
    AVG_CU(cudaMemcpyAsync(d_big, big_off.data(), sizeof(long long) * big_off.size(), cudaMemcpyHostToDevice, s));
    AVG_CU(cudaMallocAsync(&d_scratch, sizeof(unsigned long long) * (size_t)scratch_elems, s));
  }
  const double quantile = percentile / 100.0;             // np.true_divide(q, 100)
  if (method == RPSF_AVG_MEAN) {
    const unsigned mx = (unsigned)((pp + 255) / 256);
    for (int64_t c0 = 0; c0 < n_cells; c0 += 65535) {
      const unsigned gy = (unsigned)std::min<int64_t>(65535, n_cells - c0);
      average_mean<<<dim3(mx, gy), 256, 0, s>>>(cutouts, d_off + c0, d_items, pp, centre, out + c0 * pp);
      g_launches.fetch_add(1, std::memory_order_relaxed);
      AVG_CU(cudaGetLastError());
    }
  } else {
    using Deep = AvgLayout<AVG_SUBS>;
    AVG_CU(cudaFuncSetAttribute(reinterpret_cast<const void*>(average_select<true, AVG_SUBS>),
                                cudaFuncAttributeMaxDynamicSharedMemorySize, AVG_MAX_STAGED * Deep::STRIDE * 8));
    size_t first = 0;
    for (int k = 0; k < NCLASS; ++k) {
      const size_t count = lists[k].size();
      for (size_t c0 = 0; c0 < count; c0 += 65535) {
        const unsigned gy = (unsigned)std::min<size_t>(65535, count - c0);
        const int* cl = d_cells + first + c0;
        if (k < NCLASS - 1 && caps[k] <= AVG_SHALLOW)
          average_select<true, 1><<<dim3(gx, gy), AvgLayout<1>::THREADS, (size_t)caps[k] * AvgLayout<1>::STRIDE * 8, s>>>(
              cutouts, d_off, d_items, cl, pp, centre, method, quantile, nullptr, nullptr, out);
        else if (k < NCLASS - 1)
          average_select<true, AVG_SUBS><<<dim3(gx, gy), Deep::THREADS, (size_t)caps[k] * Deep::STRIDE * 8, s>>>(
              cutouts, d_off, d_items, cl, pp, centre, method, quantile, nullptr, nullptr, out);
        else
          average_select<false, AVG_SUBS><<<dim3(gx, gy), Deep::THREADS, 0, s>>>(
              cutouts, d_off, d_items, cl, pp, centre, method, quantile, d_scratch, d_big + c0, out);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        AVG_CU(cudaGetLastError());
      }
      first += count;
    }
  }
#undef AVG_CU
  release();
  return RPSF_OK;
}

namespace {
// the two per-patch builder stages share their argument checks and the stream-ordered byte scratch
int patch_stage(const double* in, double* out, int64_t n, int P, int device, void* stream, bool isolate) {
  if (P <= 0 || n < 0) return fail(RPSF_E_INVALID_ARGUMENT, "negative size");
  if (n == 0) return RPSF_OK;
  if (!out || (!isolate && !in)) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (n > INT_MAX || (long long)P * P > INT_MAX / 2) return fail(RPSF_E_UNSUPPORTED, "too many patches or patch too large");
  REFUSE_ON_CAPTURING((cudaStream_t)stream, isolate ? "rpsf_isolate_cores" : "rpsf_plane_background");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(RPSF_E_CUDA, "cannot select CUDA device %d", device);
  cudaStream_t s = (cudaStream_t)stream;
  unsigned char* scratch = nullptr;
  const size_t bytes = (size_t)n * P * P * (isolate ? 2 : 1);
  cudaError_t e = cudaMallocAsync(&scratch, bytes, s);
  if (e != cudaSuccess) return fail(RPSF_E_CUDA, "cudaMallocAsync of %zu scratch bytes failed: %s", bytes, cudaGetErrorString(e));
  if (isolate) isolate_cores<<<(unsigned)n, ISO_TPB, 0, s>>>(out, scratch, P);
  else plane_background<<<(unsigned)n, ISO_TPB, 0, s>>>(in, out, scratch, P);
  e = cudaGetLastError();
  cudaFreeAsync(scratch, s);
  if (e != cudaSuccess) return fail(RPSF_E_CUDA, "launch failed: %s", cudaGetErrorString(e));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return RPSF_OK;
}
}  // namespace

int rpsf_star_cutouts(const void* frame, int frame_dtype, int H, int W, const double* corners, int64_t n_stars, int width,
                      double saturation_threshold, double star_minimum, double star_maximum, double* out,
                      unsigned char* accepted, int device, void* stream) {
  if (H <= 0 || W <= 0 || width <= 0 || n_stars < 0) return fail(RPSF_E_INVALID_ARGUMENT, "negative size");
  if (n_stars == 0) return RPSF_OK;
  if (!frame || !corners || !out || !accepted) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (frame_dtype != RPSF_F32 && frame_dtype != RPSF_F64) return fail(RPSF_E_UNSUPPORTED, "frames must be float32 or float64");
  if (n_stars > INT_MAX || (long long)width * width > INT_MAX / 2) return fail(RPSF_E_UNSUPPORTED, "too many stars or cutout too large");
  REFUSE_ON_CAPTURING((cudaStream_t)stream, "rpsf_star_cutouts");
  for (int64_t i = 0; i < 2 * n_stars; ++i)
    if (!(std::fabs(corners[i]) < 1e9)) return fail(RPSF_E_INVALID_COORDINATE, "star corner %lld is not a finite pixel position", (long long)(i / 2));
  DeviceGuard guard(device);
  if (!guard.ok) return fail(RPSF_E_CUDA, "cannot select CUDA device %d", device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t pp = (size_t)width * width;
  double* d_corners = nullptr; double* d_coeffs = nullptr; unsigned char* d_scratch = nullptr;
  auto release = [&]() {
    for (void* ptr : {(void*)d_corners, (void*)d_coeffs, (void*)d_scratch})
      if (ptr) cudaFreeAsync(ptr, s);
  };
#define CUT_CU(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) { release(); \
    return fail(RPSF_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e_)); } } while (0)
  CUT_CU(cudaMallocAsync(&d_corners, sizeof(double) * 2 * (size_t)n_stars, s));
  CUT_CU(cudaMemcpyAsync(d_corners, corners, sizeof(double) * 2 * (size_t)n_stars, cudaMemcpyHostToDevice, s));
  CUT_CU(cudaMallocAsync(&d_coeffs, sizeof(double) * pp * (size_t)n_stars, s));
  CUT_CU(cudaMallocAsync(&d_scratch, pp * (size_t)n_stars, s));
  if (frame_dtype == RPSF_F32)
    star_cutouts<float><<<(unsigned)n_stars, ISO_TPB, 0, s>>>((const float*)frame, H, W, d_corners, width, saturation_threshold,
                                                               star_minimum, star_maximum, out, accepted, d_coeffs, d_scratch);
  else
    star_cutouts<double><<<(unsigned)n_stars, ISO_TPB, 0, s>>>((const double*)frame, H, W, d_corners, width, saturation_threshold,
                                                                star_minimum, star_maximum, out, accepted, d_coeffs, d_scratch);
  CUT_CU(cudaGetLastError());
#undef CUT_CU
  g_launches.fetch_add(1, std::memory_order_relaxed);
  // the corner list is pageable host memory: its copy must have left the caller's buffer before we return
  cudaError_t e = cudaStreamSynchronize(s);
  release();
  if (e != cudaSuccess) return fail(RPSF_E_CUDA, "star cutouts failed: %s", cudaGetErrorString(e));
  return RPSF_OK;
}

int rpsf_plane_background(const double* patches, int64_t n_patches, int P, double* out, int device, void* stream) {
  return patch_stage(patches, out, n_patches, P, device, stream, false);
}

int rpsf_isolate_cores(double* patches, int64_t n_patches, int P, int device, void* stream) {
  return patch_stage(nullptr, patches, n_patches, P, device, stream, true);
}

int rpsf_plan_set_output_mirrors(rpsf_plan* p, int n, void* const* ptrs) {
  if (!p || n < 0 || n > 7 || (n > 0 && !ptrs)) return fail(RPSF_E_INVALID_ARGUMENT, "0..7 mirror buffers");
  if (p->adjoint && n > 0) return fail(RPSF_E_UNSUPPORTED, "an adjoint plan has no output mirrors");
  p->mirrors.assign(ptrs, ptrs + n);
  return RPSF_OK;
}

int rpsf_ipc_alloc(void** ptr, int64_t bytes, int device, unsigned char handle[64]) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  if (!ptr || !handle || bytes <= 0) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  REFUSE_IN_CAPTURE("rpsf_ipc_alloc");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(RPSF_E_CUDA, "cannot select CUDA device %d", device);
  CU(cudaMalloc(ptr, (size_t)bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, *ptr);
  if (e != cudaSuccess) { cudaFree(*ptr); *ptr = nullptr; return fail(RPSF_E_CUDA, "cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e)); }
  memcpy(handle, &h, sizeof h);
  return RPSF_OK;
}

int rpsf_ipc_open(void** ptr, const unsigned char handle[64], int device) {
  if (!ptr || !handle) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  REFUSE_IN_CAPTURE("rpsf_ipc_open");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(RPSF_E_CUDA, "cannot select CUDA device %d", device);
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof h);
  CU(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return RPSF_OK;
}

int rpsf_ipc_close(void* ptr, int device) {
  if (!ptr) return RPSF_OK;
  REFUSE_IN_CAPTURE("rpsf_ipc_close");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(RPSF_E_CUDA, "cannot select CUDA device %d", device);
  CU(cudaDeviceSynchronize());
  CU(cudaIpcCloseMemHandle(ptr));
  return RPSF_OK;
}

}  // extern "C"

namespace {
// The reference pads 2P per side and slices [c+2P, c+3P) (transform.py:119-123,141-149); a corner outside [-2P, dim+P]
// makes that slice short and numpy raises.  Reject it up front.  (P here is the true patch size; an embedded
// transform's FFT length t->P is larger.)
int check_corners(const rpsf_transform* t, int H, int W) {
  const int P = t->win_len;
  for (int i = 0; i < t->n; ++i) {
    const int2 c = t->corners[i];
    if (c.x < -2 * P || c.x + P > H + 2 * P || c.y < -2 * P || c.y + P > W + 2 * P)
      return fail(RPSF_E_INVALID_COORDINATE,
                  "patch corner (%d, %d) lies outside the 2*P padded frame of shape (%d, %d)", c.x, c.y, H, W);
  }
  return RPSF_OK;
}

// The overlap-add kernel of a plan: streaming chains where every owned row pair forms one, else the row-pair gather
// where its tables exist, else colour phases.  Embedded patch sizes only have colour phases, the one overlap-add kernel
// that honours ApplyGeom::win_len.
Overlap default_overlap(const rpsf_plan* p) {
  if (p->tr->win_len != p->tr->P) return Overlap::phases;
  return p->stream_ok ? Overlap::stream : p->gather ? Overlap::gather : Overlap::phases;
}

// Where the plan of a transpose sits: the frame coordinates of box pixel (0, 0) and the frame shape.
struct AdjointBox { int y0, x0, frame_H, frame_W; };

// The forward plan of an H x W frame.  With `box`, the "frame" is the box of an adjoint plan: patch corners are shifted
// into box coordinates, a patch takes part when it touches the real frame (exactly the patches the forward reads), and
// only the default three-kernel path is prepared — the opt-in paths do not read the conjugated kernel.
int plan_build(rpsf_plan** out, rpsf_transform* t, int H, int W, int pad_mode, int row_begin, int row_end,
               int max_batch, const AdjointBox* box) {
  if (!out || !t) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (H <= 0 || W <= 0) return fail(RPSF_E_INCORRECT_SHAPE, "frame shape must be positive, got (%d, %d)", H, W);
  if (pad_mode < 0 || pad_mode > RPSF_PAD_MATERIALIZED) return fail(RPSF_E_UNSUPPORTED, "unknown pad mode %d", pad_mode);
  static_assert(RPSF_PAD_MATERIALIZED == PAD_NONE, "the materialised pad is the kernels' PAD_NONE");
  if (row_begin < 0 || row_end > H || row_begin > row_end)
    return fail(RPSF_E_INVALID_ARGUMENT, "row band [%d,%d) outside frame of %d rows", row_begin, row_end, H);
  if (max_batch < 1) return fail(RPSF_E_INVALID_ARGUMENT, "max_batch must be >= 1");
  const int P = t->P;
  if (!box)
    if (int rc = check_corners(t, H, W)) return rc;
  std::vector<int2> tcorners(t->corners);
  // the region a patch must touch to take part, in plan coordinates: the owned band, or the real frame inside the box
  int reach_r0 = row_begin, reach_r1 = row_end, reach_c0 = 0, reach_c1 = W;
  if (box) {
    for (int2& c : tcorners) { c.x -= box->y0; c.y -= box->x0; }
    reach_r0 = -box->y0; reach_r1 = box->frame_H - box->y0; reach_c0 = -box->x0; reach_c1 = box->frame_W - box->x0;
  }
  DeviceGuard guard(t->device);
  auto* p = new rpsf_plan;
  p->tr = t; p->H = H; p->W = W; p->pad_mode = pad_mode; p->row_begin = row_begin; p->row_end = row_end;
  p->max_batch = max_batch;
  const bool embedded = t->win_len != t->P;
  std::vector<int> active;
  std::vector<int2> corners;
  std::vector<std::vector<int>> items(std::max(t->n_colours, 1));
  long long colour0_area = 0;
  int lo = H, hi = 0;
  // active patches in (corner row, corner column) order: the row kernels walk the frame top to bottom
  std::vector<int> order;
  for (int i = 0; i < t->n; ++i) {
    const int2 c = tcorners[i];
    if (std::max(c.x, reach_r0) >= std::min(c.x + t->win_len, reach_r1) ||
        std::max(c.y, reach_c0) >= std::min(c.y + t->win_len, reach_c1)) continue;
    order.push_back(i);                                       // contributes to the owned band
  }
  std::stable_sort(order.begin(), order.end(), [&](int u, int v) {
    const int2 cu = tcorners[u], cv = tcorners[v];
    return cu.x != cv.x ? cu.x < cv.x : cu.y < cv.y;
  });
  for (int i : order) {
    const int2 c = tcorners[i];
    const int r0 = std::max(c.x, row_begin), r1 = std::min(c.x + t->win_len, row_end);
    const int c0 = std::max(c.y, 0), c1 = std::min(c.y + t->win_len, W);
    const int a = (int)active.size();
    if (t->kslot[i] < 0) {
      rpsf_plan_destroy(p);
      return fail(RPSF_E_INVALID_ARGUMENT,
                  "patch %d at (%d, %d) contributes to rows [%d, %d) but this transform was created without its kernel", i, c.x,
                  c.y, row_begin, row_end);
    }
    active.push_back(i);
    corners.push_back(c);
    for (int r = 0; r < t->win_len; ++r) {
      const int y = pad_index(c.x + r, H, pad_mode);
      if (y >= 0) { lo = std::min(lo, y); hi = std::max(hi, y + 1); }
    }
    for (int pair = 0; pair < (t->win_len + 1) / 2; ++pair) {         // row pairs past the window contribute nothing
      const int ya = c.x + 2 * pair, yb = ya + 1;
      if ((ya >= row_begin && ya < row_end) || (yb >= row_begin && yb < row_end))
        items[t->colour[i]].push_back(a * (P / 2) + pair);
    }
    if (t->colour[i] == 0) colour0_area += (long long)(r1 - r0) * (c1 - c0);
  }
  if (lo >= hi) { lo = 0; hi = 0; }
  p->img_lo = lo; p->img_hi = hi;
  p->n_active = (int)active.size();
  p->active_host = active;
  p->colour0_covers = !embedded && colour0_area == (long long)(row_end - row_begin) * W;
  auto destroy_fail = [&](const char* what) {
    rpsf_plan_destroy(p);
    return fail(RPSF_E_CUDA, "out of device memory for %s", what);
  };
  auto upload_fail = [&]() {
    const cudaError_t e = cudaGetLastError();
    rpsf_plan_destroy(p);
    return fail(RPSF_E_CUDA, "plan upload failed: %s", cudaGetErrorString(e));
  };
  if (p->n_active > 0) {
    if (cudaMalloc(&p->active_dev, sizeof(int) * active.size()) != cudaSuccess) return destroy_fail("patch list");
    if (cudaMalloc(&p->corners_dev, sizeof(int2) * corners.size()) != cudaSuccess) return destroy_fail("corner list");
    std::vector<int> slots_of_active(active.size());          // what the column kernel needs of a patch: where its kernel lives
    for (size_t a = 0; a < active.size(); ++a) slots_of_active[a] = t->kslot[active[a]];
    if (cudaMemcpy(p->active_dev, slots_of_active.data(), sizeof(int) * active.size(), cudaMemcpyHostToDevice) != cudaSuccess) return upload_fail();
    if (cudaMemcpy(p->corners_dev, corners.data(), sizeof(int2) * corners.size(), cudaMemcpyHostToDevice) != cudaSuccess) return upload_fail();
  }
  p->items_dev.assign(items.size(), nullptr);
  p->n_items.assign(items.size(), 0);
  for (size_t c = 0; c < items.size(); ++c) {
    p->n_items[c] = (int)items[c].size();
    if (items[c].empty()) continue;
    if (cudaMalloc(&p->items_dev[c], sizeof(int) * items[c].size()) != cudaSuccess) return destroy_fail("work list");
    if (cudaMemcpy(p->items_dev[c], items[c].data(), sizeof(int) * items[c].size(), cudaMemcpyHostToDevice) != cudaSuccess) return upload_fail();
  }
  // ---- row-pair gather tables: tiles -> groups (same corner column, summed in registers in colour
  // order) -> at most two layers of disjoint groups (one shared-memory plane each)
  {
    bool aligned = p->n_active > 0;
    const int parity = p->n_active ? ((corners[0].x % 2) + 2) % 2 : 0;
    for (const int2& c : corners) aligned = aligned && (((c.x % 2) + 2) % 2 == parity);
    if (aligned) {
      struct Entry { int item, colour, cx; };
      const int seg = std::min(W, 2048);
      const int n_seg = (W + seg - 1) / seg;
      const int y_start = row_begin - ((((row_begin - parity) % 2) + 2) % 2);
      const int n_rp = row_end > y_start ? (row_end - y_start + 1) / 2 : 0;
      std::vector<std::vector<Entry>> bucket((size_t)n_rp * n_seg);
      for (int a = 0; a < p->n_active; ++a) {
        const int2 c = corners[a];
        const int col = t->colour[active[a]];
        for (int pair = 0; pair < P / 2; ++pair) {
          const int y = c.x + 2 * pair;
          if (y + 1 < row_begin || y >= row_end) continue;
          const int rp = (y - y_start) / 2;
          for (int sgm = 0; sgm < n_seg; ++sgm) {
            const int x0 = sgm * seg, x1 = std::min(W, x0 + seg);
            if (c.y + P <= x0 || c.y >= x1) continue;
            bucket[(size_t)rp * n_seg + sgm].push_back({a * (P / 2) + pair, col, c.y});
          }
        }
      }
      std::vector<RowTile> tiles;
      std::vector<RowGroup> groups;
      std::vector<int> gitems;
      size_t most = 0;
      bool two_layers = true;
      for (int rp = 0; rp < n_rp && two_layers; ++rp)
        for (int sgm = 0; sgm < n_seg && two_layers; ++sgm) {
          auto& b = bucket[(size_t)rp * n_seg + sgm];
          std::stable_sort(b.begin(), b.end(), [](const Entry& u, const Entry& v) {
            return u.cx != v.cx ? u.cx < v.cx : u.colour < v.colour;
          });
          const int x0 = sgm * seg, x1 = std::min(W, x0 + seg);
          RowTile rt;
          rt.group_begin = (int)groups.size(); rt.group_count = 0;
          rt.y = y_start + 2 * rp; rt.x0 = x0;
          int layer_end[2] = {INT_MIN, INT_MIN};           // one past the last column a layer holds so far
          for (size_t i = 0; i < b.size();) {
            size_t j = i;
            while (j < b.size() && b[j].cx == b[i].cx) ++j;
            const int cx = b[i].cx;
            int layer = -1;
            for (int l = 0; l < 2; ++l)
              if (cx >= layer_end[l]) { layer = l; break; }
            if (layer < 0) { two_layers = false; break; }
            layer_end[layer] = cx + P;
            RowGroup gr;
            gr.item_begin = (int)gitems.size(); gr.item_count = (int)(j - i); gr.cx = cx; gr.layer = layer;
            gr.clipped = (cx < x0 || cx + P > x1) ? 1 : 0;
            for (size_t k = i; k < j; ++k) gitems.push_back(b[k].item);
            groups.push_back(gr);
            ++rt.group_count;
            i = j;
          }
          tiles.push_back(rt);                                  // a tile with no group still zero-fills its rows
          most = std::max(most, (size_t)rt.group_count);
        }
      if (two_layers && !tiles.empty()) {
        const int n1 = P == 16 || P == 32 ? 4 : P == 64 || P == 128 ? 8 : 16;
        int teams_max = std::min(288 / n1, 32);
        while (teams_max > 1 && t->ops->k3g_smem(t->dtype, teams_max, seg) > (size_t)K3G_SMEM_MAX) --teams_max;
        if (t->ops->k3g_smem(t->dtype, teams_max, seg) <= (size_t)K3G_SMEM_MAX) {
          const int rounds = most ? (int)((most + teams_max - 1) / teams_max) : 1;
          p->teams = most ? (int)((most + rounds - 1) / rounds) : 1;
          p->seg_w = seg;
          p->n_tiles = (int)tiles.size();
          if (cudaMalloc(&p->tiles_dev, sizeof(RowTile) * tiles.size()) != cudaSuccess) return destroy_fail("row tiles");
          if (cudaMemcpy(p->tiles_dev, tiles.data(), sizeof(RowTile) * tiles.size(), cudaMemcpyHostToDevice) != cudaSuccess) return upload_fail();
          if (!groups.empty()) {
            if (cudaMalloc(&p->groups_dev, sizeof(RowGroup) * groups.size()) != cudaSuccess) return destroy_fail("row groups");
            if (cudaMemcpy(p->groups_dev, groups.data(), sizeof(RowGroup) * groups.size(), cudaMemcpyHostToDevice) != cudaSuccess) return upload_fail();
            if (cudaMalloc(&p->gitems_dev, sizeof(int) * gitems.size()) != cudaSuccess) return destroy_fail("gather items");
            if (cudaMemcpy(p->gitems_dev, gitems.data(), sizeof(int) * gitems.size(), cudaMemcpyHostToDevice) != cudaSuccess) return upload_fail();
          }
          p->gather = true;
        }
      }
    }
  }
  // ---- streaming overlap-add tables
  if (p->n_active > 0 && (long long)p->n_active * (P / 2) < (1LL << 30)) {
    std::vector<int> colours(active.size());
    for (size_t a = 0; a < active.size(); ++a) colours[a] = t->colour[active[a]];
    const int tpw = t->ops->stream_tpw();
    StreamTables stt = build_stream_tables(corners, colours, P, W, row_begin, row_end, tpw,
                                           (long long)t->sm_count * 16 * tpw, max_batch);
    if (stt.ok) {
      if (cudaMalloc(&p->stasks_dev, sizeof(StreamTask) * stt.tasks.size()) != cudaSuccess) return destroy_fail("stream tasks");
      if (cudaMemcpy(p->stasks_dev, stt.tasks.data(), sizeof(StreamTask) * stt.tasks.size(), cudaMemcpyHostToDevice) != cudaSuccess) return upload_fail();
      if (cudaMalloc(&p->scodes_dev, sizeof(unsigned) * stt.codes.size()) != cudaSuccess) return destroy_fail("stream item codes");
      if (cudaMemcpy(p->scodes_dev, stt.codes.data(), sizeof(unsigned) * stt.codes.size(), cudaMemcpyHostToDevice) != cudaSuccess) return upload_fail();
      p->n_warp_items = stt.n_warp_items;
      p->stream_chunks = stt.chunks;
      p->stream_ok = true;
    }
  }
  // ---- row bands: each frame row is transformed once per band and shared by the band's patches
  if (p->n_active > 0) {
    const BandLayout bl = build_row_bands(corners, t->win_len, 2 * t->ops->stream_tpw());
    p->n_band_items = (int)bl.items.size();
    p->band_frame_rows = bl.frame_rows;
    if (cudaMalloc(&p->band_items_dev, sizeof(BandItem) * bl.items.size()) != cudaSuccess) return destroy_fail("band items");
    if (cudaMemcpy(p->band_items_dev, bl.items.data(), sizeof(BandItem) * bl.items.size(), cudaMemcpyHostToDevice) != cudaSuccess) return upload_fail();
    if (cudaMalloc(&p->patch_row_dev, sizeof(int) * bl.patch_row.size()) != cudaSuccess) return destroy_fail("band rows of the patches");
    if (cudaMemcpy(p->patch_row_dev, bl.patch_row.data(), sizeof(int) * bl.patch_row.size(), cudaMemcpyHostToDevice) != cudaSuccess) return upload_fail();
  }
  p->k1 = embedded ? K1Kernel::plain : K1Kernel::bulk;       // the plain K1 honours ApplyGeom::win_len
  p->overlap = default_overlap(p);
  const size_t cs = 2 * real_size(t->dtype);
  p->band_offset = (size_t)max_batch * p->n_active * P * (P / 2) * cs;
  p->workspace_bytes = p->band_offset + (size_t)max_batch * p->band_frame_rows * (P / 2) * cs;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { rpsf_plan_destroy(p); return fail(RPSF_E_CUDA, "plan upload failed: %s", cudaGetErrorString(e)); }
  *out = p;
  return RPSF_OK;
}

// CSR preimages of the np.pad index map of one axis of length n, restricted to the box positions [b0, b0 + nb) (frame
// coordinates): offsets [n + 1] then box indices, ascending per pixel
std::vector<int> fold_table(int n, int b0, int nb, int pad_mode) {
  std::vector<std::vector<int>> pre(n);
  for (int k = 0; k < nb; ++k) {
    const int src = pad_index(b0 + k, n, pad_mode);
    if (src >= 0) pre[src].push_back(k);
  }
  std::vector<int> csr(1, 0);
  for (const auto& v : pre) csr.push_back(csr.back() + (int)v.size());
  for (const auto& v : pre) csr.insert(csr.end(), v.begin(), v.end());
  return csr;
}
}  // namespace

extern "C" {

int rpsf_plan_create(rpsf_plan** out, rpsf_transform* t, int H, int W, int pad_mode, int row_begin, int row_end,
                     int max_batch) {
  if (out && t) REFUSE_IN_CAPTURE("rpsf_plan_create");
  return plan_build(out, t, H, W, pad_mode, row_begin, row_end, max_batch, nullptr);
}

int rpsf_plan_create_stack(rpsf_plan** out, rpsf_stack* st, int H, int W, int pad_mode, int max_batch) {
  if (!out || !st) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  REFUSE_IN_CAPTURE("rpsf_plan_create_stack");
  if (pad_mode == RPSF_PAD_MATERIALIZED) return fail(RPSF_E_UNSUPPORTED, "a stack plan needs a pad mode with an index map");
  if (max_batch < 1) return fail(RPSF_E_INVALID_ARGUMENT, "max_batch must be >= 1");
  // the overlap-add runs once over n_kernels * batch spectra: a grid dimension
  if ((long long)max_batch * st->m > 65535)
    return fail(RPSF_E_INVALID_ARGUMENT, "kernels x max_batch = %lld exceeds 65535", (long long)max_batch * st->m);
  // built for n_kernels * max_batch frames, so that the overlap-add's work split fits the batch it runs
  if (int rc = plan_build(out, st->t, H, W, pad_mode, 0, H, max_batch * st->m, nullptr)) return rc;
  rpsf_plan* p = *out;
  rpsf_transform* t = st->t;
  const size_t cs = 2 * real_size(t->dtype);
  p->max_batch = max_batch;            // frames per call: the row bands and the saturation scratch
  p->stack = st;
  p->band_offset = (size_t)st->m * max_batch * p->n_active * t->P * (t->P / 2) * cs;
  p->workspace_bytes = p->band_offset + (size_t)max_batch * p->band_frame_rows * (t->P / 2) * cs;
  return RPSF_OK;
}

int rpsf_plan_create_adjoint(rpsf_plan** out, rpsf_transform* t, int H, int W, int pad_mode, int max_batch) {
  if (!out || !t) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (H <= 0 || W <= 0) return fail(RPSF_E_INCORRECT_SHAPE, "frame shape must be positive, got (%d, %d)", H, W);
  if (pad_mode < 0 || pad_mode >= RPSF_PAD_MATERIALIZED)
    return fail(RPSF_E_UNSUPPORTED, "the transpose needs a pad mode with an index map (0..4), got %d", pad_mode);
  if (max_batch < 1) return fail(RPSF_E_INVALID_ARGUMENT, "max_batch must be >= 1");
  REFUSE_IN_CAPTURE("rpsf_plan_create_adjoint");
  if (int rc = check_corners(t, H, W)) return rc;
  // the box: bounding box of the footprints of the patches that touch the frame (a 1 x 1 box when none does)
  const int L = t->win_len;
  int y0 = INT_MAX, x0 = INT_MAX, y1 = INT_MIN, x1 = INT_MIN;
  for (const int2& c : t->corners) {
    if (std::max(c.x, 0) >= std::min(c.x + L, H) || std::max(c.y, 0) >= std::min(c.y + L, W)) continue;
    y0 = std::min(y0, c.x); x0 = std::min(x0, c.y); y1 = std::max(y1, c.x + L); x1 = std::max(x1, c.y + L);
  }
  if (y0 == INT_MAX) { y0 = 0; x0 = 0; y1 = 1; x1 = 1; }
  const int Hb = y1 - y0, Wb = x1 - x0;
  const AdjointBox box{y0, x0, H, W};
  rpsf_plan* p = nullptr;
  // the box holds every patch it serves whole, so the index map is never consulted there; constant is the cheapest
  if (int rc = plan_build(&p, t, Hb, Wb, RPSF_PAD_CONSTANT, 0, Hb, max_batch, &box)) return rc;
  DeviceGuard guard(t->device);
  p->adjoint = true;
  p->frame_H = H; p->frame_W = W; p->box_y0 = y0; p->box_x0 = x0;
  p->frame_pad_mode = pad_mode;
  const size_t rs = real_size(t->dtype), align = 16 / rs;
  p->box_pitch = (long long)((Wb + align - 1) / align * align);
  const size_t box_bytes = (size_t)max_batch * Hb * p->box_pitch * rs;
  const std::vector<int> rows = fold_table(H, y0, Hb, pad_mode), cols = fold_table(W, x0, Wb, pad_mode);
  const int pad = 2 * t->P;
  const std::vector<int> prows = fold_table(H, -pad, H + 2 * pad, pad_mode), pcols = fold_table(W, -pad, W + 2 * pad, pad_mode);
  auto bail = [&](const char* what) {
    const cudaError_t e = cudaGetLastError();
    rpsf_plan_destroy(p);
    return fail(RPSF_E_CUDA, "adjoint plan: %s failed: %s", what, cudaGetErrorString(e));
  };
  if (cudaMalloc(&p->box_in, box_bytes) != cudaSuccess || cudaMalloc(&p->box_out, box_bytes) != cudaSuccess)
    return bail("box buffers");
  if (cudaMemset(p->box_in, 0, box_bytes) != cudaSuccess) return bail("zeroing the box");     // margins stay zero
  if (cudaMalloc(&p->fold_rows, sizeof(int) * rows.size()) != cudaSuccess ||
      cudaMalloc(&p->fold_cols, sizeof(int) * cols.size()) != cudaSuccess)
    return bail("fold tables");
  if (cudaMemcpy(p->fold_rows, rows.data(), sizeof(int) * rows.size(), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(p->fold_cols, cols.data(), sizeof(int) * cols.size(), cudaMemcpyHostToDevice) != cudaSuccess)
    return bail("fold table upload");
  if (cudaMalloc(&p->fold_prows, sizeof(int) * prows.size()) != cudaSuccess ||
      cudaMalloc(&p->fold_pcols, sizeof(int) * pcols.size()) != cudaSuccess)
    return bail("padded fold tables");
  if (cudaMemcpy(p->fold_prows, prows.data(), sizeof(int) * prows.size(), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(p->fold_pcols, pcols.data(), sizeof(int) * pcols.size(), cudaMemcpyHostToDevice) != cudaSuccess)
    return bail("padded fold table upload");
  if (!t->kconj_main && t->n_kept > 0) {
    const size_t cs = 2 * rs;
    if (cudaMalloc(&t->kconj_main, (size_t)t->n_kept * t->P * (t->P / 2) * cs) != cudaSuccess ||
        cudaMalloc(&t->kconj_nyq, (size_t)t->n_kept * t->P * cs) != cudaSuccess) {
      cudaFree(t->kconj_main); cudaFree(t->kconj_nyq); t->kconj_main = t->kconj_nyq = nullptr;
      return bail("conjugated transfer kernel");
    }
    if (t->has_kernel) {
      // kmain may still be written on another stream by rpsf_transform_set_kernel: order by the device
      if (cudaDeviceSynchronize() != cudaSuccess) return bail("synchronise before conjugating");
      if (int rc = refresh_conj_kernel(t, nullptr)) { rpsf_plan_destroy(p); return rc; }
      if (cudaDeviceSynchronize() != cudaSuccess) return bail("conjugating the transfer kernel");
    }
  }
  *out = p;
  return RPSF_OK;
}

int rpsf_plan_destroy(rpsf_plan* p) {
  if (!p) return RPSF_OK;
  DeviceGuard guard(p->tr->device);
  for (cudaStream_t s : {p->s_in, p->s_comp, p->s_out})
    if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
  for (int i = 0; i < rpsf_plan::HOST_SLOTS; ++i) {
    if (p->ev_in[i]) cudaEventDestroy(p->ev_in[i]);
    if (p->ev_comp[i]) cudaEventDestroy(p->ev_comp[i]);
    if (p->ev_out[i]) cudaEventDestroy(p->ev_out[i]);
    cudaFree(p->d_in_raw[i]); cudaFree(p->d_in[i]); cudaFree(p->d_out[i]); cudaFree(p->d_out_conv[i]);
    if (p->h_stage[i]) cudaFreeHost(p->h_stage[i]);
  }
  cudaFree(p->active_dev); cudaFree(p->corners_dev); cudaFree(p->workspace);
  cudaFree(p->band_items_dev); cudaFree(p->patch_row_dev);
  cudaFree(p->tiles_dev); cudaFree(p->groups_dev); cudaFree(p->gitems_dev);
  cudaFree(p->stasks_dev); cudaFree(p->scodes_dev);
  cudaFree(p->sat_pf); cudaFree(p->sat_mask[0]); cudaFree(p->sat_mask[1]); cudaFree(p->sat_list);
  cudaFree(p->sat_rows); cudaFree(p->sat_flags);
  cudaFree(p->box_in); cudaFree(p->box_out); cudaFree(p->fold_rows); cudaFree(p->fold_cols);
  cudaFree(p->fold_prows); cudaFree(p->fold_pcols); cudaFree(p->mask_out); cudaFree(p->mask_count);
  for (int* d : p->items_dev) cudaFree(d);
  for (cudaEvent_t e : p->events) cudaEventDestroy(e);
  delete p;
  return RPSF_OK;
}

int rpsf_plan_set_overlap_mode(rpsf_plan* p, int mode) {
  if (!p) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (p->tr->win_len != p->tr->P) return RPSF_OK;             // embedded patch sizes only have the colour-phase kernel
  if (mode == 1) p->overlap = Overlap::phases;
  else if (mode == 2) p->overlap = p->gather ? Overlap::gather : Overlap::phases;
  else p->overlap = default_overlap(p);
  return RPSF_OK;
}

int rpsf_plan_set_gather_mode(rpsf_plan* p, int mode) {
  if (!p) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (p->tr->win_len != p->tr->P) return RPSF_OK;             // embedded patch sizes only have the plain gather kernel
  p->k1 = mode == 1 ? K1Kernel::plain : K1Kernel::bulk;
  return RPSF_OK;
}

int rpsf_plan_info(const rpsf_plan* p, int64_t info[9]) {
  if (!p || !info) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  info[0] = p->n_active; info[1] = p->tr->n_colours; info[2] = (int64_t)p->workspace_bytes;
  info[3] = p->img_lo; info[4] = p->img_hi; info[5] = p->colour0_covers ? 1 : 0;
  info[6] = (int64_t)p->overlap; info[7] = p->teams;
  info[8] = p->overlap == Overlap::stream ? p->stream_chunks : 0;
  return RPSF_OK;
}

static RowBands row_bands(const rpsf_plan* p) {
  return RowBands{p->band_items_dev, p->patch_row_dev, p->n_band_items, p->band_frame_rows};
}
static void* band_buffer(const rpsf_plan* p) { return (char*)p->workspace + p->band_offset; }

static int ensure_workspace(rpsf_plan* p) {
  if (p->workspace || p->workspace_bytes == 0) return RPSF_OK;
  if (t_capturing) return refuse_capture("the first call of a plan (its spectrum workspace)");
  DeviceGuard guard(p->tr->device);
  if (cudaMalloc(&p->workspace, p->workspace_bytes) != cudaSuccess) {
    cudaGetLastError();
    return fail(RPSF_E_CUDA, "out of device memory for the spectrum workspace (%zu bytes)", p->workspace_bytes);
  }
  return RPSF_OK;
}

int rpsf_plan_workspace(const rpsf_plan* p, void** ptr, int64_t* bytes) {
  if (!p || !ptr || !bytes) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (int rc = ensure_workspace(const_cast<rpsf_plan*>(p))) return rc;
  *ptr = p->workspace; *bytes = (int64_t)p->workspace_bytes;
  return RPSF_OK;
}

int rpsf_plan_column_info(const rpsf_plan* p, int64_t info[2]) {
  if (!p || !info) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  info[0] = 0; info[1] = 0;       // there is one column pass, and it needs no workspace of its own
  return RPSF_OK;
}

int rpsf_upload(void** device_ptr, const void* src_host, int64_t bytes, int device) {
  if (!device_ptr || bytes < 0 || (bytes > 0 && !src_host)) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  REFUSE_IN_CAPTURE("rpsf_upload");
  DeviceGuard guard(device);
  *device_ptr = nullptr;
  if (bytes == 0) return RPSF_OK;
  CU(cudaMalloc(device_ptr, (size_t)bytes));
  cudaError_t e = cudaMemcpy(*device_ptr, src_host, (size_t)bytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    cudaFree(*device_ptr); *device_ptr = nullptr;
    return fail(RPSF_E_CUDA, "upload failed: %s", cudaGetErrorString(e));
  }
  return RPSF_OK;
}

int rpsf_device_free(void* device_ptr, int device) {
  if (!device_ptr) return RPSF_OK;
  REFUSE_IN_CAPTURE("rpsf_device_free");
  DeviceGuard guard(device);
  CU(cudaDeviceSynchronize());
  CU(cudaFree(device_ptr));
  return RPSF_OK;
}

int rpsf_copy_to_host(void* dst, const void* src, int64_t bytes, int device) {
  if (bytes < 0 || (bytes > 0 && (!dst || !src))) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  REFUSE_IN_CAPTURE("rpsf_copy_to_host");
  DeviceGuard guard(device);
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost));
  return RPSF_OK;
}

int rpsf_plan_set_saturation(rpsf_plan* p, double threshold, int dilation, int neighborhood_width) {
  if (!p) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (threshold != threshold) return fail(RPSF_E_INVALID_ARGUMENT, "saturation threshold is NaN");
  if (neighborhood_width < 0) return fail(RPSF_E_INVALID_ARGUMENT, "neighborhood_width must be >= 0");
  if (p->adjoint && threshold < INFINITY)
    return fail(RPSF_E_UNSUPPORTED, "an adjoint plan has no saturation branch (the mask depends on the image)");
  p->sat_threshold = threshold;
  p->sat_dilation = dilation;
  p->sat_width = neighborhood_width;
  return RPSF_OK;
}

}  // extern "C"

namespace {
// The caller's frames before their conversion to the compute dtype (laid out like the converted ones, with pitches
// of their own): the saturation mask is decided on these, as the reference decides it on float64 values.
struct SatSource {
  const void* ptr;
  int dtype;
  long long pitch, frame_stride;
};

// A caller-given bad-pixel mask (rpsf_apply_masked): uint8, nonzero = masked, pixel (y, x) of frame b at
// ptr + b*frame_stride + y*pitch + x; frame_stride 0 shares one mask across the frames.
struct MaskArg {
  const unsigned char* ptr;
  long long pitch, frame_stride;
};

SatGeom mask_geom(const rpsf_plan* p, int H, int W, int pad_mode) {
  SatGeom sg{};
  const int pad = 2 * p->tr->P;
  sg.H = H; sg.W = W; sg.pad = pad; sg.Hp = H + 2 * pad; sg.Wp = W + 2 * pad;
  sg.half = p->sat_width / 2; sg.row_begin = 0; sg.row_end = H; sg.pad_mode = pad_mode;
  return sg;
}

void launch_mask_ingest(const MaskArg& m, unsigned char* state, const SatGeom& sg, int batch, cudaStream_t s) {
  const dim3 rows_grid((unsigned)std::min((sg.Wp + 255) / 256, 8), (unsigned)sg.Hp, (unsigned)batch);
  mask_ingest<<<rows_grid, 256, 0, s>>>(m.ptr, m.pitch, m.frame_stride, state, sg);
}

// raster-ordered list of the masked pixels of `state`: per-row counts, scan, ordered scatter
int mask_compact(rpsf_plan* p, const unsigned char* state, const SatGeom& sg, int batch, cudaStream_t s) {
  const dim3 warp_rows((unsigned)((sg.Hp + 7) / 8), (unsigned)batch);
  sat_row_count<<<warp_rows, 256, 0, s>>>(state, p->sat_rows, sg.Hp, sg.Wp);
  LAUNCH((int)cudaGetLastError());
  sat_row_scan<<<batch, 1024, 0, s>>>(p->sat_rows, sg.Hp);
  LAUNCH((int)cudaGetLastError());
  sat_row_scatter<<<warp_rows, 256, 0, s>>>(state, p->sat_rows, p->sat_list, sg.Hp, sg.Wp);
  LAUNCH((int)cudaGetLastError());
  return RPSF_OK;
}

// launch sat_pad_mask with the mask decided on `src` when converting its dtype to T can change a comparison with
// the threshold (float64 and 32/64-bit integers into float32), else on the converted image itself.  A 64-bit integer
// rounds to double in the comparison, as it does in the reference's `.astype(float)`.
template <typename T>
int launch_sat_pad_mask(rpsf_plan* p, const void* image, const SatSource* src, const SatGeom& sg, int* any_flag,
                        dim3 grid, cudaStream_t s) {
  auto go = [&](auto tag, const void* ptr, long long pitch, long long stride) {
    using TS = decltype(tag);
    sat_pad_mask<T, TS><<<grid, 256, 0, s>>>((const T*)image, (const TS*)ptr, pitch, stride, (T*)p->sat_pf,
                                             p->sat_mask[0], any_flag, p->sat_threshold, sg);
  };
  const int dt = (src && std::is_same<T, float>::value) ? src->dtype : -1;
  switch (dt) {
    case RPSF_F64: go(double(), src->ptr, src->pitch, src->frame_stride); break;
    case RPSF_I32: go(int32_t(), src->ptr, src->pitch, src->frame_stride); break;
    case RPSF_U32: go(uint32_t(), src->ptr, src->pitch, src->frame_stride); break;
    case RPSF_I64: go((long long)0, src->ptr, src->pitch, src->frame_stride); break;
    default: go(T(), image, sg.img_pitch, sg.img_frame_stride); break;
  }
  return (int)cudaGetLastError();
}

// Saturation pre-fill on the stream: pad + mask, dilate, OR the caller's mask (`mask`, may be null), compact in raster
// order, ordered fill.  With an infinite threshold the threshold mask is empty and only the caller's mask is used.
// On return *filled points at padded pixel (2P, 2P) of frame 0, i.e. at unpadded (0, 0).
template <typename T>
int sat_prefill(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, const SatSource* src,
                int batch, cudaStream_t s, SatGeom* sg_out, const void** filled, const MaskArg* mask = nullptr) {
  rpsf_transform* t = p->tr;
  const int P = t->P, pad = 2 * P;
  SatGeom sg;
  sg.H = p->H; sg.W = p->W; sg.pad = pad; sg.Hp = p->H + 2 * pad; sg.Wp = p->W + 2 * pad;
  sg.half = p->sat_width / 2; sg.row_begin = p->row_begin; sg.row_end = p->row_end;
  sg.img_pitch = img_pitch; sg.img_frame_stride = img_frame_stride;
  sg.out_pitch = 0; sg.out_frame_stride = 0; sg.out_row0 = 0; sg.pad_mode = p->pad_mode;
  const size_t px = (size_t)sg.Hp * sg.Wp, mb = (size_t)p->max_batch;
  if ((long long)px > 0x7fffffffLL) return fail(RPSF_E_UNSUPPORTED, "padded frame too large for the saturation branch");
  if (!p->sat_pf) {
    if (t_capturing) return refuse_capture("the first saturation branch of a plan (its scratch)");
    CU(cudaMalloc(&p->sat_pf, px * sizeof(T) * mb));
    CU(cudaMalloc((void**)&p->sat_mask[0], px * mb));
    CU(cudaMalloc((void**)&p->sat_mask[1], px * mb));
    CU(cudaMalloc((void**)&p->sat_list, px * sizeof(int) * mb));
    CU(cudaMalloc((void**)&p->sat_rows, (size_t)(sg.Hp + 1) * sizeof(int) * mb));
    CU(cudaMalloc((void**)&p->sat_flags, 2 * sizeof(int) * mb));
  }
  CU(cudaMemsetAsync(p->sat_flags, 0, 2 * sizeof(int) * mb, s));
  int* any_flag = p->sat_flags;
  int* tickets = p->sat_flags + mb;
  const dim3 rows_grid((unsigned)std::min((sg.Wp + 255) / 256, 8), (unsigned)sg.Hp, (unsigned)batch);
  LAUNCH(launch_sat_pad_mask<T>(p, image, src, sg, any_flag, rows_grid, s));
  int cur = 0;
  if (mask && p->sat_threshold == INFINITY) {
    // nothing is above the threshold: no dilation
  } else if (p->sat_dilation < 1) {
    sat_dilate<<<rows_grid, 256, 0, s>>>(p->sat_mask[0], p->sat_mask[1], any_flag, sg.Hp, sg.Wp, 1);
    LAUNCH((int)cudaGetLastError());
    cur = 1;
  } else {
    for (int it = 0; it < p->sat_dilation; ++it) {
      sat_dilate<<<rows_grid, 256, 0, s>>>(p->sat_mask[cur], p->sat_mask[cur ^ 1], any_flag, sg.Hp, sg.Wp, 0);
      LAUNCH((int)cudaGetLastError());
      cur ^= 1;
    }
  }
  unsigned char* state = p->sat_mask[cur];
  if (mask) {
    launch_mask_ingest(*mask, state, sg, batch, s);
    LAUNCH((int)cudaGetLastError());
  }
  if (int rc = mask_compact(p, state, sg, batch, s)) return rc;
  // every CTA of the fill must be resident at once only for speed, not for correctness (tickets)
  sat_fill<T><<<dim3((unsigned)t->sm_count * 2, (unsigned)batch), 256, 0, s>>>((T*)p->sat_pf, state, p->sat_list, p->sat_rows, tickets, sg);
  LAUNCH((int)cudaGetLastError());
  *sg_out = sg;
  *filled = (const T*)p->sat_pf + (size_t)pad * sg.Wp + pad;
  return RPSF_OK;
}

template <typename T>
int sat_restore_launch(rpsf_plan* p, const void* image, void* out, int64_t out_pitch, int64_t out_frame_stride,
                       int out_row0, int batch, cudaStream_t s, SatGeom sg) {
  sg.out_pitch = out_pitch; sg.out_frame_stride = out_frame_stride; sg.out_row0 = out_row0;
  sat_restore<T><<<dim3((unsigned)p->tr->sm_count, (unsigned)batch), 256, 0, s>>>((const T*)image, (T*)out, p->sat_list, p->sat_rows, sg);
  LAUNCH((int)cudaGetLastError());
  return RPSF_OK;
}

// `src`: the frames before their conversion to the compute dtype, for the saturation mask (nullptr: `image`)
int apply_stages(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int img_row0,
                 int img_rows, void* out, int64_t out_pitch, int64_t out_frame_stride, int out_row0,
                 int batch, int stages, void* stream_v, const SatSource* src = nullptr, const MaskArg* mask = nullptr) {
  if (p->stack) return fail(RPSF_E_INVALID_ARGUMENT, "a plan of a transform stack runs through rpsf_apply_stack only");
  if (p->row_end == p->row_begin && stages >= 3) return RPSF_OK;      // an empty band (more ranks than half-patch rows): nothing to write
  if (!image || !out) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  rpsf_transform* t = p->tr;
  if (!t->has_kernel) return fail(RPSF_E_NO_KERNEL, "transfer kernel not loaded (call rpsf_transform_set_kernel)");
  if (batch < 1 || batch > p->max_batch)
    return fail(RPSF_E_INVALID_ARGUMENT, "batch %d outside [1, max_batch=%d]", batch, p->max_batch);
  if (p->pad_mode == PAD_NONE && (img_row0 != 0 || img_rows != p->H))
    return fail(RPSF_E_INVALID_ARGUMENT, "a materialised pad needs the whole frame: img_row0 = 0, img_rows = height");
  if (p->pad_mode != PAD_NONE && p->n_active > 0 && (img_row0 > p->img_lo || img_row0 + img_rows < p->img_hi))
    return fail(RPSF_E_INVALID_ARGUMENT, "resident rows [%d,%d) do not cover the rows this plan reads [%d,%d)",
                img_row0, img_row0 + img_rows, p->img_lo, p->img_hi);
  if (out_row0 > p->row_begin) return fail(RPSF_E_INVALID_ARGUMENT, "out_row0 %d is past row_begin %d", out_row0, p->row_begin);
  if (img_pitch < p->W || out_pitch < p->W) return fail(RPSF_E_INCORRECT_SHAPE, "row pitch smaller than frame width");
  DeviceGuard guard(t->device);
  cudaStream_t s = (cudaStream_t)stream_v;
  ApplyGeom g;
  g.H = p->H; g.W = p->W; g.img_row0 = img_row0; g.img_rows = img_rows; g.img_pitch = img_pitch;
  g.img_frame_stride = img_frame_stride; g.out_row0 = out_row0; g.row_begin = p->row_begin; g.row_end = p->row_end;
  g.out_pitch = out_pitch; g.out_frame_stride = out_frame_stride; g.n_active = p->n_active; g.pad_mode = p->pad_mode;
  g.win_len = t->win_len;
  const size_t rs = real_size(t->dtype);
  const int band = p->row_end - p->row_begin;
  const bool use_stream = p->overlap == Overlap::stream;
  const bool use_gather = p->overlap == Overlap::gather;
  const bool need_zero = !((p->colour0_covers || use_gather || use_stream) && stages >= 3);
  cudaEvent_t* ev = nullptr;
  if (p->timing && stages >= 3 && p->n_active > 0) {
    if (t_capturing) return refuse_capture("a plan with stage timing");
    if (p->events_used + 4 > p->events.size()) {
      for (int i = 0; i < 4; ++i) { cudaEvent_t e; CU(cudaEventCreate(&e)); p->events.push_back(e); }
    }
    ev = &p->events[p->events_used];
    p->events_used += 4;
    CU(cudaEventRecord(ev[0], s));
  }
  if (need_zero && band > 0 && stages >= 3) {
    for (int b = 0; b < batch; ++b) {
      char* dst = (char*)out + ((size_t)b * out_frame_stride + (size_t)(p->row_begin - out_row0) * out_pitch) * rs;
      CU(cudaMemset2DAsync(dst, (size_t)out_pitch * rs, 0, (size_t)p->W * rs, band, s));
    }
  }
  // a caller's mask fills the frame before K1 at every stage count (the kernel gradient's X is K1 of the filled frame)
  const bool sat = (p->sat_threshold < INFINITY && stages >= 3) || mask;
  if (p->n_active == 0 && !sat) return RPSF_OK;
  SatGeom sg;
  const void* k1_image = image;
  ApplyGeom g1 = g;
  if (sat) {
    if (img_row0 != 0 || img_rows < p->H)
      return fail(RPSF_E_UNSUPPORTED, "the saturation branch needs the whole frame resident (rows [0,%d))", p->H);
    int rc = t->dtype == RPSF_F32 ? sat_prefill<float>(p, image, img_pitch, img_frame_stride, src, batch, s, &sg, &k1_image, mask)
                                  : sat_prefill<double>(p, image, img_pitch, img_frame_stride, src, batch, s, &sg, &k1_image, mask);
    if (rc) return rc;
    g1.img_row0 = 0; g1.img_rows = sg.Hp; g1.img_pitch = sg.Wp; g1.img_frame_stride = (long long)sg.Hp * sg.Wp;
    g1.pad_mode = PAD_NONE;
  }
  auto restore = [&]() -> int {
    if (!sat || stages < 3) return RPSF_OK;
    return t->dtype == RPSF_F32
               ? sat_restore_launch<float>(p, image, out, out_pitch, out_frame_stride, out_row0, batch, s, sg)
               : sat_restore_launch<double>(p, image, out, out_pitch, out_frame_stride, out_row0, batch, s, sg);
  };
  if (p->n_active == 0) return restore();
  if (int rc = ensure_workspace(p)) return rc;
  const RowBands rb = row_bands(p);
  // the streaming K1 packs a band-buffer row index and a 2-bit kind into 32 bits
  if (p->k1 == K1Kernel::bulk && (long long)batch * p->band_frame_rows < (1LL << 30)) {
    // bulk (1-D TMA) row copies need 16-byte aligned rows; the kernel still checks each band's column offset
    const size_t rsz = real_size(t->dtype);
    const int bulk_ok = ((reinterpret_cast<uintptr_t>(k1_image) & 15) == 0 && ((size_t)g1.img_pitch * rsz) % 16 == 0 &&
                         ((size_t)g1.img_frame_stride * rsz) % 16 == 0) ? 1 : 0;
    LAUNCH(t->ops->k1s(t->dtype, k1_image, band_buffer(p), rb, t->tw, t->win, g1, batch, bulk_ok, t->sm_count, s));
  } else {
    LAUNCH(t->ops->k1(t->dtype, k1_image, band_buffer(p), rb, t->tw, t->win, g1, batch, s));
  }
  if (ev) CU(cudaEventRecord(ev[1], s));
  if (stages < 2) return RPSF_OK;
  LAUNCH(t->ops->k2(t->dtype, band_buffer(p), rb, p->workspace, p->adjoint ? t->kconj_main : t->kmain,
                    p->adjoint ? t->kconj_nyq : t->knyq, p->active_dev, t->tw, t->win, g, batch, t->sm_count, s));
  if (ev) CU(cudaEventRecord(ev[2], s));
  if (stages < 3) return RPSF_OK;
  if (!p->mirrors.empty() && (!use_stream || sat))
    return fail(RPSF_E_UNSUPPORTED, "output mirrors need the streaming overlap-add of a covering, without the saturation branch");
  if (use_stream) {
    OutMirrors mir{};
    mir.n = (int)p->mirrors.size();
    for (int d = 0; d < mir.n; ++d) {
      mir.delta[d] = (long long)((char*)p->mirrors[d] - (char*)out);
      if (mir.delta[d] & 15) return fail(RPSF_E_INVALID_ARGUMENT, "mirror %d is not 16-byte congruent with out", d);
    }
    LAUNCH(t->ops->k3s(t->dtype, p->workspace, out, p->stasks_dev, p->scodes_dev, p->n_warp_items, t->tw, t->win, g, batch,
                       t->sm_count, mir.n ? &mir : nullptr, s));
    if (ev) CU(cudaEventRecord(ev[3], s));
    return restore();
  }
  if (use_gather) {
    LAUNCH(t->ops->k3g(t->dtype, p->workspace, out, p->tiles_dev, p->n_tiles, p->groups_dev, p->gitems_dev, t->tw,
                       t->win, p->teams, p->seg_w, g, batch, s));
    if (ev) CU(cudaEventRecord(ev[3], s));
    return restore();
  }
  for (size_t c = 0; c < p->items_dev.size(); ++c) {
    if (p->n_items[c] == 0) continue;
    const int store_only = (c == 0 && p->colour0_covers) ? 1 : 0;
    LAUNCH(t->ops->k3(t->dtype, p->workspace, out, p->corners_dev, p->items_dev[c], p->n_items[c], t->tw, t->win,
                      store_only, g, batch, s));
  }
  if (ev) CU(cudaEventRecord(ev[3], s));
  return restore();
}

// whether a stack plan runs k2_stack: from two kernels on (with one it has no forward transform to share, and was
// measured 9 % slower than K2 in float32), not at embedded patch sizes (their pruned column pass), nor where the stage
// ring of the pipelined column pass does not fit (ops->k2s_ok), nor when rpsf_plan_set_stack_mode forced the per-kernel K2
bool stack_fused(const rpsf_plan* p) {
  const rpsf_transform* t = p->tr;
  return p->stack_mode == 0 && p->stack->m >= 2 && t->win_len == t->P && t->ops->k2s_ok(t->dtype);
}

// rpsf_apply_stack: the saturation / mask fill and K1 once for the `batch` frames, K2 once per kernel from the shared row
// bands into that kernel's spectra, and one overlap-add over all n_kernels * batch spectra.  Each kernel's output is
// what apply_stages computes for it alone: the same kernels run on the same data, and none of them depends on where
// its frame sits in the batch.
int apply_stack(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, void* out,
                int64_t out_pitch, int64_t out_frame_stride, int batch, cudaStream_t s, const SatSource* src,
                const MaskArg* mask) {
  rpsf_transform* t = p->tr;
  const rpsf_stack* st = p->stack;
  const int M = st->m;
  for (int m = 0; m < M; ++m)
    if (!st->loaded[m]) return fail(RPSF_E_NO_KERNEL, "transfer kernel %d of the stack not loaded (call rpsf_stack_set_kernel)", m);
  if (batch < 1 || batch > p->max_batch)
    return fail(RPSF_E_INVALID_ARGUMENT, "batch %d outside [1, max_batch=%d]", batch, p->max_batch);
  if (img_pitch < p->W || out_pitch < p->W) return fail(RPSF_E_INCORRECT_SHAPE, "row pitch smaller than frame width");
  DeviceGuard guard(t->device);
  ApplyGeom g;
  g.H = p->H; g.W = p->W; g.img_row0 = 0; g.img_rows = p->H; g.img_pitch = img_pitch;
  g.img_frame_stride = img_frame_stride; g.out_row0 = 0; g.row_begin = 0; g.row_end = p->H;
  g.out_pitch = out_pitch; g.out_frame_stride = out_frame_stride; g.n_active = p->n_active; g.pad_mode = p->pad_mode;
  g.win_len = t->win_len;
  const size_t rs = real_size(t->dtype), cs = 2 * rs;
  const int frames = M * batch;                 // output frame m * batch + b is kernel m applied to frame b
  const bool use_stream = p->overlap == Overlap::stream;
  const bool use_gather = p->overlap == Overlap::gather;
  if (!(p->colour0_covers || use_gather || use_stream))
    for (int j = 0; j < frames; ++j)
      CU(cudaMemset2DAsync((char*)out + (size_t)j * out_frame_stride * rs, (size_t)out_pitch * rs, 0, (size_t)p->W * rs,
                           p->H, s));
  const bool sat = p->sat_threshold < INFINITY || mask;
  if (p->n_active == 0 && !sat) return RPSF_OK;
  SatGeom sg;
  const void* k1_image = image;
  ApplyGeom g1 = g;
  if (sat) {
    int rc = t->dtype == RPSF_F32 ? sat_prefill<float>(p, image, img_pitch, img_frame_stride, src, batch, s, &sg, &k1_image, mask)
                                  : sat_prefill<double>(p, image, img_pitch, img_frame_stride, src, batch, s, &sg, &k1_image, mask);
    if (rc) return rc;
    g1.img_row0 = 0; g1.img_rows = sg.Hp; g1.img_pitch = sg.Wp; g1.img_frame_stride = (long long)sg.Hp * sg.Wp;
    g1.pad_mode = PAD_NONE;
  }
  auto restore = [&]() -> int {
    if (!sat) return RPSF_OK;
    for (int m = 0; m < M; ++m) {
      void* om = (char*)out + (size_t)m * batch * out_frame_stride * rs;
      int rc = t->dtype == RPSF_F32 ? sat_restore_launch<float>(p, image, om, out_pitch, out_frame_stride, 0, batch, s, sg)
                                    : sat_restore_launch<double>(p, image, om, out_pitch, out_frame_stride, 0, batch, s, sg);
      if (rc) return rc;
    }
    return RPSF_OK;
  };
  if (p->n_active == 0) return restore();
  if (int rc = ensure_workspace(p)) return rc;
  const RowBands rb = row_bands(p);
  if (p->k1 == K1Kernel::bulk && (long long)batch * p->band_frame_rows < (1LL << 30)) {
    const int bulk_ok = ((reinterpret_cast<uintptr_t>(k1_image) & 15) == 0 && ((size_t)g1.img_pitch * rs) % 16 == 0 &&
                         ((size_t)g1.img_frame_stride * rs) % 16 == 0) ? 1 : 0;
    LAUNCH(t->ops->k1s(t->dtype, k1_image, band_buffer(p), rb, t->tw, t->win, g1, batch, bulk_ok, t->sm_count, s));
  } else {
    LAUNCH(t->ops->k1(t->dtype, k1_image, band_buffer(p), rb, t->tw, t->win, g1, batch, s));
  }
  const size_t spec_frame = (size_t)p->n_active * t->P * (t->P / 2) * cs;
  if (stack_fused(p)) {
    // one forward column FFT per tile and frame, then the multiply and inverse FFT of every kernel (k2_stack)
    LAUNCH(t->ops->k2s(t->dtype, band_buffer(p), rb, p->workspace, (long long)((size_t)batch * spec_frame / cs), t->kmain,
                       (long long)(st->main_bytes / cs), t->knyq, (long long)(st->nyq_bytes / cs), M, p->active_dev, t->tw,
                       t->win, g, batch, t->sm_count, s));
  } else {
    // per-kernel column pass: the existing K2 once per kernel, on the shared row bands
    for (int m = 0; m < M; ++m)
      LAUNCH(t->ops->k2(t->dtype, band_buffer(p), rb, (char*)p->workspace + (size_t)m * batch * spec_frame,
                        (char*)t->kmain + st->main_bytes * m, (char*)t->knyq + st->nyq_bytes * m, p->active_dev, t->tw,
                        t->win, g, batch, t->sm_count, s));
  }
  if (use_stream) {
    LAUNCH(t->ops->k3s(t->dtype, p->workspace, out, p->stasks_dev, p->scodes_dev, p->n_warp_items, t->tw, t->win, g,
                       frames, t->sm_count, nullptr, s));
  } else if (use_gather) {
    LAUNCH(t->ops->k3g(t->dtype, p->workspace, out, p->tiles_dev, p->n_tiles, p->groups_dev, p->gitems_dev, t->tw,
                       t->win, p->teams, p->seg_w, g, frames, s));
  } else {
    for (size_t c = 0; c < p->items_dev.size(); ++c) {
      if (p->n_items[c] == 0) continue;
      const int store_only = (c == 0 && p->colour0_covers) ? 1 : 0;
      LAUNCH(t->ops->k3(t->dtype, p->workspace, out, p->corners_dev, p->items_dev[c], p->n_items[c], t->tw, t->win,
                        store_only, g, frames, s));
    }
  }
  return restore();
}

// y (whole frames) -> interior of the zero-bordered box of an adjoint plan (the margins stay zero)
template <typename T>
int adjoint_copy(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int batch, cudaStream_t s) {
  const int H = p->frame_H, W = p->frame_W;
  const long long box_stride = (long long)p->H * p->box_pitch;
  // the part of the frame inside the box; the rest of y meets no patch
  const int r0 = std::max(0, p->box_y0), r1 = std::min(H, p->box_y0 + p->H);
  const int c0 = std::max(0, p->box_x0), c1 = std::min(W, p->box_x0 + p->W);
  if (r1 > r0 && c1 > c0) {
    const dim3 grid((unsigned)((c1 - c0 + 255) / 256), (unsigned)std::min(r1 - r0, 1024), (unsigned)batch);
    adjoint_copy_in<T><<<grid, 256, 0, s>>>((const T*)image + (long long)r0 * img_pitch + c0, img_pitch, img_frame_stride,
                                            r1 - r0, c1 - c0,
                                            (T*)p->box_in + (long long)(r0 - p->box_y0) * p->box_pitch + (c0 - p->box_x0),
                                            p->box_pitch, box_stride);
    LAUNCH((int)cudaGetLastError());
  }
  return RPSF_OK;
}

// Aᵀ y: y (whole frames) -> interior of the zero-bordered box, the forward kernels on the box with conj(Kh), fold
template <typename T>
int apply_adjoint(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int img_row0,
                  int img_rows, void* out, int64_t out_pitch, int64_t out_frame_stride, int out_row0, int batch,
                  cudaStream_t s) {
  rpsf_transform* t = p->tr;
  if (!image || !out) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (!t->has_kernel) return fail(RPSF_E_NO_KERNEL, "transfer kernel not loaded (call rpsf_transform_set_kernel)");
  if (batch < 1 || batch > p->max_batch)
    return fail(RPSF_E_INVALID_ARGUMENT, "batch %d outside [1, max_batch=%d]", batch, p->max_batch);
  if (img_row0 != 0 || img_rows != p->frame_H || out_row0 != 0)
    return fail(RPSF_E_INVALID_ARGUMENT, "an adjoint plan takes and writes whole frames (row0 = 0, rows = %d)", p->frame_H);
  if (img_pitch < p->frame_W || out_pitch < p->frame_W) return fail(RPSF_E_INCORRECT_SHAPE, "row pitch smaller than frame width");
  DeviceGuard guard(t->device);
  const int H = p->frame_H, W = p->frame_W;
  const long long box_stride = (long long)p->H * p->box_pitch;
  if (int rc = adjoint_copy<T>(p, image, img_pitch, img_frame_stride, batch, s)) return rc;
  if (int rc = apply_stages(p, p->box_in, p->box_pitch, box_stride, 0, p->H, p->box_out, p->box_pitch, box_stride, 0,
                            batch, 3, s))
    return rc;
  const int* rows = p->fold_rows;
  const int* cols = p->fold_cols;
  const dim3 grid((unsigned)((W + 255) / 256), (unsigned)std::min(H, 1024), (unsigned)batch);
  fold_pad_adjoint<T><<<grid, 256, 0, s>>>((const T*)p->box_out, p->box_pitch, box_stride, rows, rows + H + 1, cols,
                                           cols + W + 1, (T*)out, out_pitch, out_frame_stride, H, W);
  LAUNCH((int)cudaGetLastError());
  return RPSF_OK;
}

// (1 - M) y (whole frames) -> interior of the zero-bordered box of an adjoint plan
template <typename T>
int adjoint_copy_masked(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, const MaskArg& m,
                        int batch, cudaStream_t s) {
  const int H = p->frame_H, W = p->frame_W;
  const long long box_stride = (long long)p->H * p->box_pitch;
  const int r0 = std::max(0, p->box_y0), r1 = std::min(H, p->box_y0 + p->H);
  const int c0 = std::max(0, p->box_x0), c1 = std::min(W, p->box_x0 + p->W);
  if (r1 > r0 && c1 > c0) {
    const dim3 grid((unsigned)((c1 - c0 + 255) / 256), (unsigned)std::min(r1 - r0, 1024), (unsigned)batch);
    mask_copy_in<T><<<grid, 256, 0, s>>>((const T*)image + (long long)r0 * img_pitch + c0, img_pitch, img_frame_stride,
                                         m.ptr + (long long)r0 * m.pitch + c0, m.pitch, m.frame_stride, r1 - r0, c1 - c0,
                                         (T*)p->box_in + (long long)(r0 - p->box_y0) * p->box_pitch + (c0 - p->box_x0),
                                         p->box_pitch, box_stride);
    LAUNCH((int)cudaGetLastError());
  }
  return RPSF_OK;
}

// L_Mᵀ y = padᵀ(pad(M) g_ext + (1 - pad(M)) Fᵀ v), v = the patch path's transpose of (1 - M) y on the padded frame:
// masked copy into the box, the three kernels with conj(Kh), the box onto the padded frame, the fill's structure from
// the mask alone (ingest, raster list, counts), the transposed fill, the gather and combine, the fold over the padded frame
template <typename T>
int apply_adjoint_masked(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int img_row0,
                         int img_rows, void* out, int64_t out_pitch, int64_t out_frame_stride, int out_row0, int batch,
                         const MaskArg& m, cudaStream_t s) {
  rpsf_transform* t = p->tr;
  if (!image || !out) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (!t->has_kernel) return fail(RPSF_E_NO_KERNEL, "transfer kernel not loaded (call rpsf_transform_set_kernel)");
  if (batch < 1 || batch > p->max_batch)
    return fail(RPSF_E_INVALID_ARGUMENT, "batch %d outside [1, max_batch=%d]", batch, p->max_batch);
  if (img_row0 != 0 || img_rows != p->frame_H || out_row0 != 0)
    return fail(RPSF_E_INVALID_ARGUMENT, "an adjoint plan takes and writes whole frames (row0 = 0, rows = %d)", p->frame_H);
  if (img_pitch < p->frame_W || out_pitch < p->frame_W) return fail(RPSF_E_INCORRECT_SHAPE, "row pitch smaller than frame width");
  DeviceGuard guard(t->device);
  const int H = p->frame_H, W = p->frame_W;
  const SatGeom sg = mask_geom(p, H, W, p->frame_pad_mode);
  const size_t px = (size_t)sg.Hp * sg.Wp, mb = (size_t)p->max_batch;
  if ((long long)px > 0x7fffffffLL) return fail(RPSF_E_UNSUPPORTED, "padded frame too large for the masked transpose");
  if (p->box_y0 < -sg.pad || p->box_x0 < -sg.pad || p->box_y0 + p->H > H + sg.pad || p->box_x0 + p->W > W + sg.pad)
    return fail(RPSF_E_UNSUPPORTED, "the patch footprints reach past the padded frame");
  if (!p->mask_count) {
    if (t_capturing) return refuse_capture("the first masked transpose of a plan (its scratch)");
    CU(cudaMalloc(&p->sat_pf, px * sizeof(T) * mb));
    CU(cudaMalloc(&p->mask_out, px * sizeof(T) * mb));
    CU(cudaMalloc((void**)&p->sat_mask[0], px * mb));
    CU(cudaMalloc((void**)&p->sat_list, px * sizeof(int) * mb));
    CU(cudaMalloc((void**)&p->sat_rows, (size_t)(sg.Hp + 1) * sizeof(int) * mb));
    CU(cudaMalloc((void**)&p->sat_flags, 2 * sizeof(int) * mb));
    CU(cudaMalloc((void**)&p->mask_count, px * sizeof(int) * mb));
  }
  const long long box_stride = (long long)p->H * p->box_pitch;
  if (int rc = adjoint_copy_masked<T>(p, image, img_pitch, img_frame_stride, m, batch, s)) return rc;
  if (int rc = apply_stages(p, p->box_in, p->box_pitch, box_stride, 0, p->H, p->box_out, p->box_pitch, box_stride, 0,
                            batch, 3, s))
    return rc;
  const dim3 rows_grid((unsigned)std::min((sg.Wp + 255) / 256, 8), (unsigned)sg.Hp, (unsigned)batch);
  T* u = (T*)p->sat_pf;
  unsigned char* state = p->sat_mask[0];
  box_to_padded<T><<<rows_grid, 256, 0, s>>>((const T*)p->box_out, p->box_pitch, box_stride, p->box_y0, p->box_x0, p->H,
                                             p->W, u, sg);
  LAUNCH((int)cudaGetLastError());
  CU(cudaMemsetAsync(state, 0, px * batch, s));
  CU(cudaMemsetAsync(p->sat_flags, 0, 2 * sizeof(int) * mb, s));
  launch_mask_ingest(m, state, sg, batch, s);
  LAUNCH((int)cudaGetLastError());
  if (int rc = mask_compact(p, state, sg, batch, s)) return rc;
  const dim3 fill_grid((unsigned)t->sm_count * 2, (unsigned)batch);
  sat_fill_count<<<fill_grid, 256, 0, s>>>(state, p->sat_list, p->sat_rows, p->sat_flags, p->mask_count, sg);
  LAUNCH((int)cudaGetLastError());
  sat_fill_adjoint<T><<<fill_grid, 256, 0, s>>>(u, state, p->sat_list, p->sat_rows, p->sat_flags + mb, p->mask_count, sg);
  LAUNCH((int)cudaGetLastError());
  mask_gather_adjoint<T><<<rows_grid, 256, 0, s>>>(u, state, (const T*)image, img_pitch, img_frame_stride,
                                                   (T*)p->mask_out, sg);
  LAUNCH((int)cudaGetLastError());
  const dim3 grid((unsigned)((W + 255) / 256), (unsigned)std::min(H, 1024), (unsigned)batch);
  fold_pad_adjoint<T><<<grid, 256, 0, s>>>((const T*)p->mask_out, sg.Wp, (long long)px, p->fold_prows,
                                           p->fold_prows + H + 1, p->fold_pcols, p->fold_pcols + W + 1, (T*)out,
                                           out_pitch, out_frame_stride, H, W);
  LAUNCH((int)cudaGetLastError());
  return RPSF_OK;
}
}  // namespace

extern "C" {

int rpsf_apply_stages(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int img_row0,
                      int img_rows, void* out, int64_t out_pitch, int64_t out_frame_stride, int out_row0,
                      int batch, int stages, void* stream) {
  if (!p) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (p->adjoint) return fail(RPSF_E_UNSUPPORTED, "an adjoint plan runs whole (rpsf_apply)");
  return ordered(p->tr, (cudaStream_t)stream, [&]() -> int {
    return apply_stages(p, image, img_pitch, img_frame_stride, img_row0, img_rows, out, out_pitch, out_frame_stride,
                        out_row0, batch, stages, stream);
  });
}

// `mask` (may be null): X is K1 of the frame filled under the caller's mask, G that of (1 - M) grad
static int kernel_gradient(rpsf_plan* ap, rpsf_plan* fp, const void* image, int64_t img_pitch, int64_t img_frame_stride,
                           const void* grad, int64_t grad_pitch, int64_t grad_frame_stride, int batch, void* kernel_grad,
                           void* stream, const MaskArg* mask) {
  if (!ap || !fp || !image || !grad || !kernel_grad) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (!ap->adjoint || fp->adjoint)
    return fail(RPSF_E_INVALID_ARGUMENT, "rpsf_kernel_gradient takes an adjoint plan, then a forward plan");
  rpsf_transform* t = fp->tr;
  if (ap->tr != t) return fail(RPSF_E_INVALID_ARGUMENT, "the two plans belong to different transforms");
  if (fp->H != ap->frame_H || fp->W != ap->frame_W)
    return fail(RPSF_E_INVALID_ARGUMENT, "the plans are for frames of (%d, %d) and (%d, %d)", fp->H, fp->W, ap->frame_H,
                ap->frame_W);
  if (t->win_len != t->P)
    return fail(RPSF_E_UNSUPPORTED, "patch size %d runs embedded in %d; its kernel gradient is not implemented", t->win_len,
                t->P);
  if (t->n_kept < t->n) return fail(RPSF_E_UNSUPPORTED, "a sharded transform holds only some patches' kernels");
  if (fp->sat_threshold < INFINITY)
    return fail(RPSF_E_UNSUPPORTED, "the kernel gradient has no saturation branch (set an infinite threshold)");
  if (fp->pad_mode == PAD_NONE) return fail(RPSF_E_UNSUPPORTED, "the materialised pad has no index map");
  if (fp->row_begin != 0 || fp->row_end != fp->H)
    return fail(RPSF_E_UNSUPPORTED, "the forward plan owns rows [%d, %d), not the whole frame", fp->row_begin, fp->row_end);
  if (fp->pad_mode != ap->frame_pad_mode)
    return fail(RPSF_E_INVALID_ARGUMENT, "the plans use pad modes %d and %d", fp->pad_mode, ap->frame_pad_mode);
  if (batch < 1 || batch > fp->max_batch || batch > ap->max_batch)
    return fail(RPSF_E_INVALID_ARGUMENT, "batch %d outside [1, %d]", batch, std::min(fp->max_batch, ap->max_batch));
  if (img_pitch < fp->W || grad_pitch < fp->W) return fail(RPSF_E_INCORRECT_SHAPE, "row pitch smaller than frame width");
  // both plans take the patches that touch the frame, sorted by corner: kgrad pairs their workspaces slot by slot
  if (fp->active_host != ap->active_host)
    return fail(RPSF_E_INVALID_ARGUMENT, "the forward and adjoint plans list different active patches");
  cudaStream_t s = (cudaStream_t)stream;
  return ordered(t, s, [&]() -> int {
    const int P = t->P;
    // per-stage events of the forward plan (bench only): K1(x) | copy + K1(g) | zeroing + kgrad
    cudaEvent_t* ev = nullptr;
    if (fp->timing && fp->n_active > 0) {
      if (t_capturing) return refuse_capture("a plan with stage timing");
      if (fp->events_used + 4 > fp->events.size()) {
        for (int i = 0; i < 4; ++i) { cudaEvent_t e; CU(cudaEventCreate(&e)); fp->events.push_back(e); }
      }
      ev = &fp->events[fp->events_used];
      fp->events_used += 4;
      CU(cudaEventRecord(ev[0], s));
    }
    // 1. X: K1 of the forward plan (stages = 1 writes nothing to `out`)
    if (int rc = apply_stages(fp, image, img_pitch, img_frame_stride, 0, fp->H, kernel_grad, fp->W, 0, 0, batch, 1, s,
                              nullptr, mask))
      return rc;
    if (ev) CU(cudaEventRecord(ev[1], s));
    // 2-3. G: the gradient into the adjoint plan's zero-bordered box, K1 there
    const long long box_stride = (long long)ap->H * ap->box_pitch;
    if (mask) {
      if (int rc = (t->dtype == RPSF_F32 ? adjoint_copy_masked<float> : adjoint_copy_masked<double>)(
              ap, grad, grad_pitch, grad_frame_stride, *mask, batch, s))
        return rc;
    } else if (int rc = (t->dtype == RPSF_F32 ? adjoint_copy<float> : adjoint_copy<double>)(ap, grad, grad_pitch,
                                                                                              grad_frame_stride, batch, s)) {
      return rc;
    }
    if (int rc = apply_stages(ap, ap->box_in, ap->box_pitch, box_stride, 0, ap->H, ap->box_out, ap->box_pitch, box_stride, 0,
                              batch, 1, s))
      return rc;
    if (ev) CU(cudaEventRecord(ev[2], s));
    // 4. patches that do not touch the frame: an exact zero (neither map reads them)
    const size_t slot_bytes = (size_t)P * P * 2 * real_size(t->dtype);
    std::vector<char> touched(t->n, 0);           // the active list is in corner order: zero runs of untouched indices
    for (int i : fp->active_host) touched[i] = 1;
    for (int i = 0; i < t->n;) {
      if (touched[i]) { ++i; continue; }
      int j = i;
      while (j < t->n && !touched[j]) ++j;
      CU(cudaMemsetAsync((char*)kernel_grad + (size_t)i * slot_bytes, 0, (size_t)(j - i) * slot_bytes, s));
      i = j;
    }
    // 5. conj(X) G / P^2, summed over the batch
    if (fp->n_active > 0)
      LAUNCH(t->ops->kgrad(t->dtype, band_buffer(fp), row_bands(fp), band_buffer(ap), row_bands(ap), kernel_grad,
                           fp->active_dev, t->tw, t->win, fp->n_active, batch, s));
    if (ev) CU(cudaEventRecord(ev[3], s));
    return RPSF_OK;
  });
}

int rpsf_kernel_gradient(rpsf_plan* ap, rpsf_plan* fp, const void* image, int64_t img_pitch, int64_t img_frame_stride,
                         const void* grad, int64_t grad_pitch, int64_t grad_frame_stride, int batch, void* kernel_grad,
                         void* stream) {
  return kernel_gradient(ap, fp, image, img_pitch, img_frame_stride, grad, grad_pitch, grad_frame_stride, batch, kernel_grad,
                         stream, nullptr);
}

int rpsf_kernel_gradient_masked(rpsf_plan* ap, rpsf_plan* fp, const void* image, int64_t img_pitch,
                                int64_t img_frame_stride, const void* grad, int64_t grad_pitch, int64_t grad_frame_stride,
                                int batch, void* kernel_grad, const void* mask, int64_t mask_pitch,
                                int64_t mask_frame_stride, void* stream) {
  if (!mask) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (fp && mask_pitch < fp->W) return fail(RPSF_E_INCORRECT_SHAPE, "mask row pitch smaller than frame width");
  const MaskArg m{(const unsigned char*)mask, mask_pitch, mask_frame_stride};
  return kernel_gradient(ap, fp, image, img_pitch, img_frame_stride, grad, grad_pitch, grad_frame_stride, batch, kernel_grad,
                         stream, &m);
}

int rpsf_plan_enable_timing(rpsf_plan* p, int enabled) {
  if (!p) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  p->timing = enabled != 0;
  return RPSF_OK;
}

int rpsf_plan_read_timing(rpsf_plan* p, double ms[3], int* calls) {
  if (!p || !ms || !calls) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  REFUSE_IN_CAPTURE("rpsf_plan_read_timing");
  DeviceGuard guard(p->tr->device);
  ms[0] = ms[1] = ms[2] = 0.0;
  *calls = 0;
  for (size_t i = 0; i + 4 <= p->events_used; i += 4) {
    CU(cudaEventSynchronize(p->events[i + 3]));
    for (int k = 0; k < 3; ++k) {
      float t = 0.f;
      CU(cudaEventElapsedTime(&t, p->events[i + k], p->events[i + k + 1]));
      ms[k] += t;
    }
    ++*calls;
  }
  p->events_used = 0;
  return RPSF_OK;
}

int rpsf_apply(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int img_row0,
               int img_rows, void* out, int64_t out_pitch, int64_t out_frame_stride, int out_row0, int batch,
               void* stream) {
  if (!p) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  return ordered(p->tr, (cudaStream_t)stream, [&]() -> int {
    if (p->adjoint)
      return (p->tr->dtype == RPSF_F32 ? apply_adjoint<float> : apply_adjoint<double>)(
          p, image, img_pitch, img_frame_stride, img_row0, img_rows, out, out_pitch, out_frame_stride, out_row0, batch,
          (cudaStream_t)stream);
    return apply_stages(p, image, img_pitch, img_frame_stride, img_row0, img_rows, out, out_pitch,
                             out_frame_stride, out_row0, batch, 3, stream);
  });
}

int rpsf_apply_masked(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int img_row0,
                      int img_rows, void* out, int64_t out_pitch, int64_t out_frame_stride, int out_row0, int batch,
                      const void* src, int src_dtype, int64_t src_pitch, int64_t src_frame_stride, const void* mask,
                      int64_t mask_pitch, int64_t mask_frame_stride, void* stream) {
  if (!p || !mask) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  const int W = p->adjoint ? p->frame_W : p->W;
  if (mask_pitch < W) return fail(RPSF_E_INCORRECT_SHAPE, "mask row pitch smaller than frame width");
  if (p->pad_mode == PAD_NONE) return fail(RPSF_E_UNSUPPORTED, "a mask needs a pad mode with an index map (0..4)");
  if (p->adjoint && src) return fail(RPSF_E_UNSUPPORTED, "an adjoint plan has no saturation branch (src)");
  if (src && !elem_size(src_dtype)) return fail(RPSF_E_UNSUPPORTED, "unsupported source dtype code %d", src_dtype);
  if (src && src_pitch < p->W) return fail(RPSF_E_INCORRECT_SHAPE, "source row pitch smaller than frame width");
  const MaskArg m{(const unsigned char*)mask, mask_pitch, mask_frame_stride};
  const SatSource source{src, src_dtype, src_pitch, src_frame_stride};
  return ordered(p->tr, (cudaStream_t)stream, [&]() -> int {
    if (p->adjoint)
      return (p->tr->dtype == RPSF_F32 ? apply_adjoint_masked<float> : apply_adjoint_masked<double>)(
          p, image, img_pitch, img_frame_stride, img_row0, img_rows, out, out_pitch, out_frame_stride, out_row0, batch, m,
          (cudaStream_t)stream);
    if (img_row0 != 0 || img_rows < p->H)
      return fail(RPSF_E_UNSUPPORTED, "a mask needs the whole frame resident (rows [0,%d))", p->H);
    return apply_stages(p, image, img_pitch, img_frame_stride, img_row0, img_rows, out, out_pitch, out_frame_stride,
                        out_row0, batch, 3, stream, src ? &source : nullptr, &m);
  });
}

int rpsf_apply_source(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, int img_row0,
                      int img_rows, void* out, int64_t out_pitch, int64_t out_frame_stride, int out_row0, int batch,
                      const void* src, int src_dtype, int64_t src_pitch, int64_t src_frame_stride, void* stream) {
  if (!p) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (p->adjoint) return fail(RPSF_E_UNSUPPORTED, "an adjoint plan has no saturation branch (rpsf_apply)");
  if (!src) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (!elem_size(src_dtype)) return fail(RPSF_E_UNSUPPORTED, "unsupported source dtype code %d", src_dtype);
  if (src_pitch < p->W) return fail(RPSF_E_INCORRECT_SHAPE, "source row pitch smaller than frame width");
  const SatSource source{src, src_dtype, src_pitch, src_frame_stride};
  return ordered(p->tr, (cudaStream_t)stream, [&]() -> int {
    return apply_stages(p, image, img_pitch, img_frame_stride, img_row0, img_rows, out, out_pitch, out_frame_stride,
                        out_row0, batch, 3, stream, &source);
  });
}

int rpsf_plan_set_stack_mode(rpsf_plan* p, int mode) {
  if (!p || !p->stack) return fail(RPSF_E_INVALID_ARGUMENT, "not a plan of a transform stack");
  if (mode != 0 && mode != 1) return fail(RPSF_E_INVALID_ARGUMENT, "stack mode must be 0 or 1, got %d", mode);
  p->stack_mode = mode;
  return RPSF_OK;
}

int rpsf_plan_stack_info(const rpsf_plan* p, int* fused) {
  if (!p || !p->stack || !fused) return fail(RPSF_E_INVALID_ARGUMENT, "null argument or not a plan of a transform stack");
  *fused = stack_fused(p) ? 1 : 0;
  return RPSF_OK;
}

int rpsf_apply_stack(rpsf_plan* p, const void* image, int64_t img_pitch, int64_t img_frame_stride, void* out,
                     int64_t out_pitch, int64_t out_frame_stride, int n_kernels, int batch, const void* src, int src_dtype,
                     int64_t src_pitch, int64_t src_frame_stride, const void* mask, int64_t mask_pitch,
                     int64_t mask_frame_stride, void* stream) {
  if (!p || !image || !out) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (!p->stack) return fail(RPSF_E_INVALID_ARGUMENT, "not a plan of a transform stack (rpsf_plan_create_stack)");
  if (n_kernels != p->stack->m)
    return fail(RPSF_E_INVALID_ARGUMENT, "%d kernels given, the plan's stack has %d", n_kernels, p->stack->m);
  if (mask && mask_pitch < p->W) return fail(RPSF_E_INCORRECT_SHAPE, "mask row pitch smaller than frame width");
  if (src && !elem_size(src_dtype)) return fail(RPSF_E_UNSUPPORTED, "unsupported source dtype code %d", src_dtype);
  if (src && src_pitch < p->W) return fail(RPSF_E_INCORRECT_SHAPE, "source row pitch smaller than frame width");
  const MaskArg m{(const unsigned char*)mask, mask_pitch, mask_frame_stride};
  const SatSource source{src, src_dtype, src_pitch, src_frame_stride};
  return ordered(p->tr, (cudaStream_t)stream, [&]() -> int {
    return apply_stack(p, image, img_pitch, img_frame_stride, out, out_pitch, out_frame_stride, batch,
                       (cudaStream_t)stream, src ? &source : nullptr, mask ? &m : nullptr);
  });
}


int rpsf_convert(const void* src, int sdt, int64_t sp, void* dst, int ddt, int64_t dp, int rows, int cols,
                 int device, void* stream) {
  if (!src || !dst) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (rows <= 0 || cols <= 0) return RPSF_OK;
  DeviceGuard guard(device);
  int rc = ddt == RPSF_F32   ? convert_to<float>(src, sdt, sp, dst, dp, rows, cols, (cudaStream_t)stream)
           : ddt == RPSF_F64 ? convert_to<double>(src, sdt, sp, dst, dp, rows, cols, (cudaStream_t)stream)
                             : -1;
  if (rc) return fail(RPSF_E_UNSUPPORTED, "unsupported conversion %d -> %d", sdt, ddt);
  LAUNCH((int)cudaGetLastError());
  return RPSF_OK;
}

}  // extern "C"

namespace {
// A numpy array is pageable memory.  cudaMemcpyAsync from pageable memory is staged by the driver through its own
// bounce buffer on ONE thread (about 12 GB/s on this pool's hosts against 55 GB/s from pinned memory), and it blocks
// the calling thread meanwhile.  Here the staging is done by a few host threads into the plan's own pinned buffers,
// chunk by chunk, while the DMA and the kernels of the previous chunks run.
bool is_pageable_host(const void* ptr) {
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess) { cudaGetLastError(); return true; }
  return attr.type == cudaMemoryTypeUnregistered;
}
int host_copy_threads() {
  // measured on a 16-core host: 4 threads 8.5 ms per 8 frames, 8 threads 9.2, 16 threads 10.1 —
  // the copy competes with the DMA for the host memory system, more threads only add contention
  const unsigned hw = std::thread::hardware_concurrency();
  return (int)std::max(1u, std::min(4u, hw / 2));
}
// The staged bytes are read next by the DMA engine, never by this CPU: write them with non-temporal stores so the
// destination lines are not first read into the cache (a third of a plain copy's memory traffic, and the host memory
// system — shared with the DMA both ways — is what bounds the staging).
void stream_copy(char* dst, const char* src, size_t bytes) {
#if defined(__SSE2__)
  size_t head = (16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15;
  if (head > bytes) head = bytes;
  memcpy(dst, src, head);
  dst += head; src += head; bytes -= head;
  const size_t blocks = bytes / 64;
  for (size_t i = 0; i < blocks; ++i) {
    const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 0);
    const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 1);
    const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 2);
    const __m128i d = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 3);
    _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 0, a);
    _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 1, b);
    _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 2, c);
    _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 3, d);
    src += 64; dst += 64;
  }
  _mm_sfence();
  memcpy(dst, src, bytes - blocks * 64);
#else
  memcpy(dst, src, bytes);
#endif
}
// A call that fits one chunk has no earlier chunk to hide its staging behind: it is staged in pieces, the DMA of a
// piece under the staging of the next.  Measured (one 2048^2 frame): float32 1.58 ms through the driver's own pageable
// path, 1.37 staged whole, 1.26 in 4 MB pieces (2 MB: slower); uint16 1.20 / 1.11 / 1.05.  Several chunks are staged
// whole (6.7 ms per 8 frames; in 4 MB pieces 7.3).  A single chunk below 4 MB keeps the driver's path.
size_t stage_piece_bytes(bool single_chunk) { return single_chunk ? (size_t)4 << 20 : ~(size_t)0; }
bool stage_single_chunk(size_t chunk_bytes) { return chunk_bytes >= ((size_t)4 << 20); }
void parallel_copy(void* dst, const void* src, size_t bytes, int threads) {
  const size_t grain = (size_t)1 << 20;
  const int n = (int)std::min<size_t>((size_t)threads, std::max<size_t>(bytes / grain, 1));
  if (n <= 1) { stream_copy((char*)dst, (const char*)src, bytes); return; }
  std::vector<std::thread> pool;
  const size_t per = ((bytes + n - 1) / n + 63) / 64 * 64;
  for (int i = 1; i < n; ++i) {
    const size_t b = std::min(bytes, per * i), e = std::min(bytes, per * (i + 1));
    if (e > b) pool.emplace_back([=]() { stream_copy((char*)dst + b, (const char*)src + b, e - b); });
  }
  stream_copy((char*)dst, (const char*)src, std::min(bytes, per));
  for (auto& t : pool) t.join();
}
}  // namespace

extern "C" {

int rpsf_apply_host(rpsf_plan* p, const void* image, int image_dtype, void* out, int out_dtype, int batch) {
  if (!p) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (p->adjoint) return fail(RPSF_E_UNSUPPORTED, "an adjoint plan takes device pointers (rpsf_apply)");
  if (batch < 1) return fail(RPSF_E_INVALID_ARGUMENT, "batch must be >= 1");
  if (p->row_end == p->row_begin) return RPSF_OK;                      // empty band: no bytes to produce
  if (!image || !out) return fail(RPSF_E_INVALID_ARGUMENT, "null argument");
  if (out_dtype != RPSF_F32 && out_dtype != RPSF_F64) return fail(RPSF_E_UNSUPPORTED, "output dtype must be f32 or f64");
  REFUSE_IN_CAPTURE("rpsf_apply_host");
  const size_t isz = elem_size(image_dtype);
  if (!isz) return fail(RPSF_E_UNSUPPORTED, "unsupported image dtype code %d", image_dtype);
  rpsf_transform* t = p->tr;
  DeviceGuard guard(t->device);
  constexpr int R = rpsf_plan::HOST_SLOTS;
  const int H = p->H, W = p->W, band = p->row_end - p->row_begin;
  const size_t rs = real_size(t->dtype), os = real_size(out_dtype);
  const size_t frame_px = (size_t)H * W, band_px = (size_t)band * W;
  const size_t band_alloc = std::max<size_t>(band_px, 1);
  const int mb = p->max_batch;                       // frames per chunk
  const bool conv_in = image_dtype != t->dtype;
  const bool conv_out = out_dtype != t->dtype;
  if (!p->s_in) {
    CU(cudaStreamCreateWithFlags(&p->s_in, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&p->s_comp, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&p->s_out, cudaStreamNonBlocking));
    for (int i = 0; i < R; ++i) {
      CU(cudaEventCreateWithFlags(&p->ev_in[i], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&p->ev_comp[i], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&p->ev_out[i], cudaEventDisableTiming));
    }
  }
  // a single chunk needs one slot; allocate the ring lazily as far as this call uses it
  const int n_chunks = (batch + mb - 1) / mb;
  const int slots = std::min(R, n_chunks);
  for (int i = 0; i < slots; ++i) {
    if (!p->d_in[i]) CU(cudaMalloc(&p->d_in[i], frame_px * rs * mb));
    if (!p->d_out[i]) CU(cudaMalloc(&p->d_out[i], band_alloc * rs * mb));
  }
  if (conv_in && p->d_in_raw_bytes < frame_px * isz * mb) {
    for (int i = 0; i < R; ++i) { cudaFree(p->d_in_raw[i]); p->d_in_raw[i] = nullptr; }
    p->d_in_raw_bytes = frame_px * isz * mb;
  }
  if (conv_out && p->d_out_conv_bytes < band_alloc * os * mb) {
    for (int i = 0; i < R; ++i) { cudaFree(p->d_out_conv[i]); p->d_out_conv[i] = nullptr; }
    p->d_out_conv_bytes = band_alloc * os * mb;
  }
  for (int i = 0; i < slots; ++i) {
    if (conv_in && !p->d_in_raw[i]) CU(cudaMalloc(&p->d_in_raw[i], p->d_in_raw_bytes));
    if (conv_out && !p->d_out_conv[i]) CU(cudaMalloc(&p->d_out_conv[i], p->d_out_conv_bytes));
  }
  const bool stage = (n_chunks >= 2 || stage_single_chunk(frame_px * isz * (size_t)batch)) && is_pageable_host(image);
  const int copy_threads = stage ? host_copy_threads() : 1;
  if (stage && p->h_stage_bytes < frame_px * isz * mb) {
    for (int i = 0; i < R; ++i) { if (p->h_stage[i]) cudaFreeHost(p->h_stage[i]); p->h_stage[i] = nullptr; }
    p->h_stage_bytes = frame_px * isz * mb;
  }
  for (int i = 0; i < slots && stage; ++i)
    if (!p->h_stage[i]) CU(cudaHostAlloc(&p->h_stage[i], p->h_stage_bytes, cudaHostAllocDefault));
  // the kernels run on s_comp, ordered with the transform's calls on other streams (a kernel layout on the caller's
  // stream, device calls sharing this plan's workspace)
  OrderedCall order{t, p->s_comp};
  int rc = order.begin();
  for (int ci = 0; ci < n_chunks && rc == RPSF_OK; ++ci) {
    const int b0 = ci * mb, nb = std::min(mb, batch - b0), k = ci % R;
    const char* src = (const char*)image + (size_t)b0 * frame_px * isz;
    char* dst = (char*)out + (size_t)b0 * band_px * os;
    // upload: the slot's previous occupant must have been consumed by its kernels
    if (ci >= R) CU(cudaStreamWaitEvent(p->s_in, p->ev_comp[k], 0));
    char* d_dst = (char*)(conv_in ? p->d_in_raw[k] : p->d_in[k]);
    const size_t chunk_bytes = frame_px * isz * nb;
    if (!stage) {
      CU(cudaMemcpyAsync(d_dst, src, chunk_bytes, cudaMemcpyHostToDevice, p->s_in));
    } else {
      if (ci >= R) CU(cudaEventSynchronize(p->ev_in[k]));        // the staging slot's previous DMA has read it
      // piece by piece, so that the DMA of a piece runs under the staging of the next one (and under the DMA and
      // kernels of earlier chunks)
      const size_t piece = stage_piece_bytes(n_chunks == 1);
      for (size_t off = 0; off < chunk_bytes; off += std::min(piece, chunk_bytes)) {
        const size_t nbytes = std::min(piece, chunk_bytes - off);
        parallel_copy((char*)p->h_stage[k] + off, src + off, nbytes, copy_threads);
        CU(cudaMemcpyAsync(d_dst + off, (char*)p->h_stage[k] + off, nbytes, cudaMemcpyHostToDevice, p->s_in));
      }
    }
    CU(cudaEventRecord(p->ev_in[k], p->s_in));
    // kernels: need this chunk's upload, and the slot's previous download to be done with d_out
    CU(cudaStreamWaitEvent(p->s_comp, p->ev_in[k], 0));
    if (ci >= R) CU(cudaStreamWaitEvent(p->s_comp, p->ev_out[k], 0));
    if (conv_in) {
      int e = t->dtype == RPSF_F32
                  ? convert_to<float>(p->d_in_raw[k], image_dtype, W, p->d_in[k], W, H * nb, W, p->s_comp)
                  : convert_to<double>(p->d_in_raw[k], image_dtype, W, p->d_in[k], W, H * nb, W, p->s_comp);
      if (e) return fail(RPSF_E_UNSUPPORTED, "unsupported image dtype code %d", image_dtype);
      LAUNCH((int)cudaGetLastError());
    }
    const SatSource raw{p->d_in_raw[k], image_dtype, W, (long long)frame_px};
    rc = apply_stages(p, p->d_in[k], W, (int64_t)frame_px, 0, H, p->d_out[k], W, (int64_t)band_px, p->row_begin, nb, 3,
                      p->s_comp, conv_in ? &raw : nullptr);
    if (rc) break;
    if (band_px == 0) { CU(cudaEventRecord(p->ev_comp[k], p->s_comp)); continue; }
    if (conv_out) {
      int e = out_dtype == RPSF_F32
                  ? convert_to<float>(p->d_out[k], t->dtype, W, p->d_out_conv[k], W, band * nb, W, p->s_comp)
                  : convert_to<double>(p->d_out[k], t->dtype, W, p->d_out_conv[k], W, band * nb, W, p->s_comp);
      if (e) return fail(RPSF_E_UNSUPPORTED, "unsupported output conversion");
      LAUNCH((int)cudaGetLastError());
    }
    CU(cudaEventRecord(p->ev_comp[k], p->s_comp));
    // download
    CU(cudaStreamWaitEvent(p->s_out, p->ev_comp[k], 0));
    CU(cudaMemcpyAsync(dst, conv_out ? p->d_out_conv[k] : p->d_out[k], band_px * os * nb, cudaMemcpyDeviceToHost,
                       p->s_out));
    CU(cudaEventRecord(p->ev_out[k], p->s_out));
  }
  rc = order.end(rc);
  // drain all three streams even on error so no copy is in flight when the caller's buffers go away
  cudaError_t e1 = cudaStreamSynchronize(p->s_in), e2 = cudaStreamSynchronize(p->s_comp),
              e3 = cudaStreamSynchronize(p->s_out);
  if (rc) return rc;
  for (cudaError_t e : {e1, e2, e3})
    if (e != cudaSuccess) return fail(RPSF_E_CUDA, "host apply failed: %s", cudaGetErrorString(e));
  return RPSF_OK;
}

}  // extern "C"
