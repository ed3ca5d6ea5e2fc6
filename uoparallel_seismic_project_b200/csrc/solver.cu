// solver.cu -- host side of the C ABI (include/sweeptt.h): device float-box pool, star
// tables, the device-resident convergence loop, the multi-start dispatcher.
//
// Replaces the host orchestration of cudaRun (cuda/cudasweep-tt-multistart.cu:227-410) and
// the serial convergence loop (serial_new/sweep-tt-multistart.c:150-170).  Differences by
// design: no per-sweep host round trip (CUDA-graph WHILE node, or K rounds per poll), all
// sources relaxed concurrently from one work list, sources sharded over GPUs instead of the
// reference's star splitting.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <limits>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "../../include/sweeptt.h"
#include "kernels.h"
#include "pullstar.h"
#include "quiescence.h"

using namespace sweeptt;

static constexpr int MAX_GROUPS = 8;
static constexpr int STATE_SLOTS = 1 + 512;  // slot 0: the whole-context view; 1..: one per slice of the solve plan

// ---------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------
static thread_local std::string g_err;
namespace sweeptt {
// records the message for sweeptt_last_error() and returns 0 (= failure in this ABI)
int set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return 0;
}
}  // namespace sweeptt
#define fail sweeptt::set_error
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) return fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

extern "C" const char* sweeptt_last_error(void) { return g_err.c_str(); }
extern "C" const char* sweeptt_version(void) { return "sweeptt-b200 0.1 (sm_100a)"; }

extern "C" int sweeptt_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

extern "C" int sweeptt_device_info(int device, char* name, int name_len, int* sm_count, int* clock_khz,
                                   size_t* smem_optin) {
  cudaDeviceProp p;
  CK(cudaGetDeviceProperties(&p, device));
  if (name && name_len > 0) snprintf(name, name_len, "%s", p.name);
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (clock_khz) {
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device);
    *clock_khz = khz;
  }
  if (smem_optin) *smem_optin = p.sharedMemPerBlockOptin;
  return 1;
}

extern "C" void sweeptt_star_fill_distances(struct FS* fs, int starsize, float delta) {
  // serial_new/sweep-tt-multistart.c:122,127: sqrt in double on an int, stored to float, times delta
  for (int l = 0; l < starsize; ++l) {
    float d = (float)std::sqrt((double)(fs[l].i * fs[l].i + fs[l].j * fs[l].j + fs[l].k * fs[l].k));
    fs[l].d = delta * d;
  }
}

extern "C" int sweeptt_build_pull_star(const struct FS* fs, int starsize, int star_used, int32_t* ijk_out,
                                       float* half_d_out, int32_t* guard_out, int capacity) {
  if (!fs || starsize <= 0) return -1;
  PullStar ps = build_pull_star(fs, starsize, star_used);
  const int n = (int)ps.all.size();
  if (capacity < n && (ijk_out || half_d_out || guard_out)) return -1;
  for (int l = 0; l < n; ++l) {
    if (ijk_out) { ijk_out[3 * l] = ps.all[l].i; ijk_out[3 * l + 1] = ps.all[l].j; ijk_out[3 * l + 2] = ps.all[l].k; }
    if (half_d_out) half_d_out[l] = ps.all[l].hd;
    if (guard_out) guard_out[l] = ps.all[l].guarded;
  }
  return n;
}

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  });
  return fn;
}

struct sweeptt_ctx {
  sweeptt_opts opts{};
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr;

  BoxGeom g{};
  bool have_model = false, have_star = false, have_sources = false;
  float* d_slow = nullptr;
  float* d_tt = nullptr;
  int tt_cap = 0;  // boxes allocated in the pool
  int nsrc = 0;
  std::vector<int> src_xyz;
  int* d_src = nullptr;
  int src_cap = 0;
  SolveState* d_state = nullptr;
  SolveState* h_state = nullptr;  // pinned mirror
  unsigned* d_worklist = nullptr;
  unsigned* d_key = nullptr;   // per-tile activation keys
  unsigned* d_tmax = nullptr;  // per-tile upper bound of the largest travel time (downwind filter)
  unsigned* d_busy = nullptr;  // per-tile "on a list / being relaxed" flags (single-launch scheduling)
  unsigned* d_keysnap = nullptr;  // key snapshot of the device-side list builder
  float min_slowness = 0.f;    // exact minimum of the model (device reduction); < 0: negative/NaN values present
  float max_slowness = 0.f;    // largest finite slowness of the model (domain guard, ready())
  float pos_slowness = std::numeric_limits<float>::infinity();  // smallest positive slowness (+INF: none)
  float bucket = -1.f;         // bucket width in travel-time units (<0: relax every dirty tile each round)
  double mean_slowness = 0;
  size_t tiles_cap = 0;  // nsrc*ntiles the lists/flags were sized for
  unsigned long long* d_tile_pulls = nullptr;
  int pulls_sig[7] = {0, 0, 0, 0, 0, 0, -1};  // geometry + star generation d_tile_pulls was built for
  int star_gen = 0;                           // bumped by every sweeptt_set_star
  unsigned long long* d_viol = nullptr;
  // ray tracer (sweeptt_trace_rays): pull table, receivers and a grow-only output buffer
  std::vector<RayPull> ray_pull;
  RayPull* d_ray_pull = nullptr;
  size_t ray_pull_cap = 0;
  int ray_sig[6] = {-1, -1, -1, -1, -1, -1};  // star generation, axis permutation and padded pitches of the table
  std::vector<int> rec_xyz;
  int* d_rec = nullptr;
  size_t rec_cap = 0;
  unsigned char* d_ray_out = nullptr;
  size_t ray_out_cap = 0;
  // tomography operators (sweeptt_ray_project / sweeptt_ray_backproject): grow-only padded perturbation box, int64
  // accumulator box and per-warp path records
  float* d_pert = nullptr;
  size_t pert_cap = 0;
  long long* d_acc = nullptr;
  size_t acc_cap = 0;
  unsigned short* d_path = nullptr;
  size_t path_cap = 0;
  float* d_stage = nullptr;  // dense staging box for pad/unpad
  size_t stage_floats = 0;
  // event location (sweeptt_locate_events / sweeptt_misfit_box): grow-only buffer of the picks, keys and results
  unsigned char* d_loc = nullptr;
  size_t loc_cap = 0;
  size_t pool_bytes = 0;

  std::vector<FS> fs;
  PullStar star;
  StarDev* d_star = nullptr;
  int nstar = 0;
  long long pulls_per_round = 0;

  int kernel_used = 0;
  TiledLaunch tl{};
  CUtensorMap tm_slow{}, tm_tt{};
  bool maps_valid = false;
  int consts_rxy = -1;  // variant the host image of the __constant__ tables was built for
  std::vector<ColumnDev> img_cols;
  std::vector<float> img_hd;
  std::vector<ExtraDev> img_extra;
  std::vector<unsigned> img_pdesc;
  int consts_nx = -1;   // ... and the grid's x extent (the column tables of the first / last tile along x depend on it)
  uint64_t img_sig = 0;
  std::vector<int> pat_begin;  // column ranges per k-pattern (stock-star kernels)
  std::vector<unsigned short> psplit;  // per pattern group: first column of every fine part (kernels.cu c_psplit)
  std::vector<PullColumn> dev_columns;  // pattern-sorted, even-padded columns as uploaded

  cudaGraphExec_t graph_exec = nullptr;
  bool graph_valid = false;

  // Solve plan: the sources are cut into WAVES that run one after the other; a wave is either ONE slice solved by
  // a single persistent launch (all its activation keys fit the CTA's shared memory: the best scheduler), or G
  // slices ("source groups") that run as G independent WHILE graphs on G streams -- one group's relaxation CTAs
  // fill the SMs that another group's round has already drained.  Every slice works on its own part of the work
  // lists / keys / boxes and has its own SolveState slot, so a whole solve is enqueued without a host decision
  // and finished sources can leave for the host while later waves are still being relaxed (sweeptt_solve).
  struct Slice {
    int wave = 0;
    int s0 = 0, ns = 0;
    int slot = 1;                   // SolveState slot
    int lane = 0;                   // stream: 0 = the context's own, g >= 1 = aux_streams[g-1]
    bool persistent = false;
    int grid = 0;                   // persistent launch: CTAs (0 = the whole device)
    cudaGraphExec_t graph = nullptr;
    CUtensorMap tm_tt{};
  };
  std::vector<Slice> plan;
  int plan_waves = 0;
  bool plan_valid = false;
  std::vector<cudaStream_t> aux_streams;
  std::vector<cudaEvent_t> aux_done;
  cudaEvent_t ev_fork = nullptr;

  // host <-> device staging of sweeptt_solve: finished boxes are un-padded into a ring of dense boxes on the solve
  // stream and copied out by the copy stream while the next wave is being relaxed
  cudaStream_t copy_stream = nullptr;
  float* d_out_ring = nullptr;
  float* h_out_ring = nullptr;  // page-locked twin of the ring: stop-over for results that go to PAGEABLE caller boxes
  size_t out_ring_boxes = 0, out_ring_box_floats = 0;
  std::vector<cudaEvent_t> ring_unpadded, ring_copied;

  std::vector<cudaEvent_t> prof_events;
  bool allow_outside_sources = false;  // (internal) accept start points outside the model
  int max_inner = 1;                   // in-tile passes per tile visit
  int force_window_axis = -1;          // forced caller axis of the kernel's register-window (z) axis
  int force_x_axis = -1;               // one grid over several devices: caller axis that becomes kernel x (block axis)
  bool external_boxes = false;         // d_tt belongs to a SharedBox (one grid over several devices); d_slow is ours
  int slow_pb = 0;                     // one grid over several devices: planes per block of the local slowness copy
  long long slow_planes = 0;           // ... and its total number of planes
  // one grid over several devices (see RelaxArgs): this context's part of the job
  int mp_nparts = 0, mp_part = 0;
  unsigned char* d_tx_owner = nullptr;  // [ntx] owner of every tile column along x
  int* d_tx_slow0 = nullptr;            // [ntx] first local slowness plane of every owned tile's staged box
  unsigned* mp_key[MAX_PARTS] = {};
  unsigned* mp_tmax[MAX_PARTS] = {};
  unsigned* mp_kmin[MAX_PARTS] = {};
};

// The __constant__ star tables are per-device module state shared by every context on that device.  A compute
// call holds a LEASE on them for its whole duration: contexts whose tables are identical (slab contexts, the
// cached contexts of sweeptt_solve) share the lease, a context with a different star waits until the device's
// tables are unused, then replaces them.  So two host threads driving different stars on one device serialise
// instead of overwriting each other's tables (include/sweeptt.h, "Threading").
namespace {
struct ConstTables {
  std::mutex mu;
  std::condition_variable cv;
  uint64_t sig = 0;
  bool loaded = false;
  int users = 0;
};
ConstTables& const_tables(int device) {
  static std::mutex mu;
  static std::map<int, ConstTables*> all;
  std::lock_guard<std::mutex> lk(mu);
  auto it = all.find(device);
  if (it == all.end()) it = all.emplace(device, new ConstTables()).first;
  return *it->second;
}
struct ConstLease {
  ConstTables* t = nullptr;
  ConstLease() = default;
  ConstLease(const ConstLease&) = delete;
  ConstLease& operator=(const ConstLease&) = delete;
  void release() {
    if (!t) return;
    {
      std::lock_guard<std::mutex> lk(t->mu);
      --t->users;
    }
    t->cv.notify_all();
    t = nullptr;
  }
  ~ConstLease() { release(); }
};
}  // namespace

static void invalidate_graph(sweeptt_ctx* c) {
  if (c->graph_exec) cudaGraphExecDestroy(c->graph_exec);
  c->graph_exec = nullptr;
  c->graph_valid = false;
  for (auto& sl : c->plan) {
    if (sl.graph) cudaGraphExecDestroy(sl.graph);
    sl.graph = nullptr;
  }
  c->plan.clear();
  c->plan_valid = false;
}

static int dev_alloc(sweeptt_ctx* c, void** p, size_t bytes) {
  CK(cudaMalloc(p, bytes));
  c->pool_bytes += bytes;
  return 1;
}
static void dev_free(sweeptt_ctx* c, void* p, size_t bytes) {
  if (p) {
    cudaFree(p);
    c->pool_bytes -= std::min(bytes, c->pool_bytes);
  }
}

extern "C" sweeptt_ctx* sweeptt_create(const sweeptt_opts* opts) {
  int ndev = sweeptt_device_count();
  if (ndev <= 0) {
    fail("no CUDA device available: the sweep has no CPU fallback");
    return nullptr;
  }
  auto* c = new sweeptt_ctx();
  if (opts) std::memcpy(&c->opts, opts, std::min<size_t>(sizeof(sweeptt_opts), opts->struct_size > 0 ? opts->struct_size : sizeof(sweeptt_opts)));
  int dev = c->opts.device;
  if (dev < 0) cudaGetDevice(&dev);
  if (dev >= ndev) {
    fail("device %d out of range (have %d)", dev, ndev);
    delete c;
    return nullptr;
  }
  c->device = dev;
  cudaDeviceProp prop;
  if (cudaSetDevice(dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
    fail("cannot select device %d", dev);
    delete c;
    return nullptr;
  }
  if (prop.major < 10) {
    fail("device %d (%s) is sm_%d%d; this library ships sm_100a kernels only", dev, prop.name, prop.major, prop.minor);
    delete c;
    return nullptr;
  }
  bool ok = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) == cudaSuccess;
  c->own_stream = true;
  ok = ok && cudaEventCreate(&c->ev0) == cudaSuccess && cudaEventCreate(&c->ev1) == cudaSuccess &&
       cudaEventCreate(&c->ev2) == cudaSuccess && cudaEventCreate(&c->ev3) == cudaSuccess;
  ok = ok && cudaMalloc(&c->d_state, sizeof(SolveState) * STATE_SLOTS) == cudaSuccess &&
       cudaMallocHost(&c->h_state, sizeof(SolveState) * STATE_SLOTS) == cudaSuccess &&
       cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) == cudaSuccess &&
       cudaMalloc(&c->d_viol, 32) == cudaSuccess;
  if (!ok) {
    fail("context setup failed on device %d: %s", dev, cudaGetErrorString(cudaGetLastError()));
    sweeptt_destroy(c);
    return nullptr;
  }
  return c;
}

extern "C" void sweeptt_destroy(sweeptt_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  invalidate_graph(c);
  for (auto st : c->aux_streams) cudaStreamDestroy(st);
  for (auto e : c->aux_done) cudaEventDestroy(e);
  if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
  for (auto e : c->ring_unpadded) cudaEventDestroy(e);
  for (auto e : c->ring_copied) cudaEventDestroy(e);
  cudaFree(c->d_out_ring);
  if (c->h_out_ring) cudaFreeHost(c->h_out_ring);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  for (auto e : c->prof_events) cudaEventDestroy(e);
  cudaFree(c->d_slow);
  cudaFree(c->d_tx_owner); cudaFree(c->d_tx_slow0);
  if (!c->external_boxes) cudaFree(c->d_tt);
  cudaFree(c->d_src); cudaFree(c->d_state);
  cudaFree(c->d_worklist); cudaFree(c->d_key); cudaFree(c->d_tmax); cudaFree(c->d_busy); cudaFree(c->d_keysnap); cudaFree(c->d_tile_pulls); cudaFree(c->d_viol);
  cudaFree(c->d_stage); cudaFree(c->d_star);
  cudaFree(c->d_ray_pull); cudaFree(c->d_rec); cudaFree(c->d_ray_out);
  cudaFree(c->d_pert); cudaFree(c->d_acc); cudaFree(c->d_path);
  cudaFree(c->d_loc);
  if (c->h_state) cudaFreeHost(c->h_state);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->ev2) cudaEventDestroy(c->ev2);
  if (c->ev3) cudaEventDestroy(c->ev3);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

extern "C" int sweeptt_set_stream(sweeptt_ctx* c, void* cuda_stream) {
  if (!c) return fail("null context");
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  c->stream = static_cast<cudaStream_t>(cuda_stream);
  c->own_stream = false;
  invalidate_graph(c);
  return 1;
}

static int ensure_stage(sweeptt_ctx* c, size_t floats) {
  if (c->stage_floats >= floats) return 1;
  dev_free(c, c->d_stage, c->stage_floats * 4);
  c->d_stage = nullptr; c->stage_floats = 0;
  if (!dev_alloc(c, (void**)&c->d_stage, floats * 4)) return 0;
  c->stage_floats = floats;
  return 1;
}

static int build_tile_pulls(sweeptt_ctx* c);
static int build_maps(sweeptt_ctx* c);
static int encode_tt_map(sweeptt_ctx* c, float* base, int nboxes, CUtensorMap* out);
static int choose_kernel(sweeptt_ctx* c);

// Kernel geometry of an nx x ny x nz (caller order) model: axis order, padded dims, tiles.
static int compute_geometry(sweeptt_ctx* c, int nx, int ny, int nz, BoxGeom* out) {
  BoxGeom g{};
  {
    // Axis order of the kernel: any permutation of the caller's axes gives the same field (the star is
    // permuted with it); the kernel's granularity is 4 nodes along its x (a tile's 4-wide units are
    // skipped individually), TY along y and TZ along z, so the order that wastes the fewest lanes in
    // partly filled edge tiles wins (241x241x51: the 51 axis becomes kernel x, 52/51 instead of 56/51).
    // Ties keep the caller's order.  SWEEPTT_WINDOW_AXIS=a forces caller axis a to be the window axis.
    const int n[3] = {nx, ny, nz};
    static const int perms[6][3] = {{0, 1, 2}, {1, 0, 2}, {0, 2, 1}, {2, 0, 1}, {1, 2, 0}, {2, 1, 0}};
    const int gran[3] = {4, TY, TZ};
    int pick = -1;
    double best = -1;
    int forced = -1;
    if (const char* e = getenv("SWEEPTT_WINDOW_AXIS")) forced = std::max(0, std::min(2, atoi(e)));
    if (c->force_window_axis >= 0) forced = c->force_window_axis;
    if (c->force_x_axis >= 0 && forced == c->force_x_axis) forced = -1;  // (cannot be both)
    for (int pi = 0; pi < 6; ++pi) {
      if (forced >= 0 && perms[pi][2] != forced) continue;
      if (c->force_x_axis >= 0 && perms[pi][0] != c->force_x_axis) continue;
      double eff = 1.0;
      for (int q = 0; q < 3; ++q) {
        const int len = n[perms[pi][q]];
        eff *= (double)len / (double)(((len + gran[q] - 1) / gran[q]) * gran[q]);
      }
      if (pick < 0 || eff > best * 1.02) { best = eff; pick = pi; }  // a permutation must pay for its transposing copies
    }
    for (int q = 0; q < 3; ++q) g.perm[q] = perms[pick][q];
    if (getenv("SWEEPTT_DEBUG"))
      fprintf(stderr, "sweeptt: %d x %d x %d, kernel axes = caller axes (%d,%d,%d), lane efficiency %.3f\n", nx, ny, nz,
              g.perm[0], g.perm[1], g.perm[2], best);
    const long long ds[3] = {(long long)ny * nz, (long long)nz, 1};
    for (int k = 0; k < 3; ++k) g.dstride[k] = ds[g.perm[k]];
    g.nx = n[g.perm[0]]; g.ny = n[g.perm[1]]; g.nz = n[g.perm[2]];
    nx = g.nx; ny = g.ny; nz = g.nz;  // from here on: kernel axis order
  }
  g.ntx = (nx + TX - 1) / TX; g.nty = (ny + TY - 1) / TY; g.ntz = (nz + TZ - 1) / TZ;
  g.px = AX + g.ntx * TX + RXY_MAX;
  g.py = AY + g.nty * TY + RXY_MAX;
  g.pz = AZ + g.ntz * TZ + ZHALO + 4;  // +4: the staged row is SZD = TZ+2*ZHALO+4 floats long
  g.sx = (long long)g.py * g.pz;
  g.vol = (long long)g.px * g.sx;
  if ((long long)g.ntx * g.nty * g.ntz > 0x7fffffffLL) return fail("grid too large for 32-bit tile ids");
  *out = g;
  return 1;
}

// Halo variant of the tiled kernel that holds the star (0: the star does not fit the tiled kernel).
static int tiled_rxy(const PullStar& s) {
  const bool fits = s.fits_tiled() && (int)s.columns.size() + MAX_PATTERNS + 2 <= MAX_COLUMNS &&
                    (int)s.col_hd.size() <= MAX_COL_HD && (int)s.extra.size() <= MAX_EXTRA;
  return fits ? tiled_variant_for_radius(std::max(s.rx, s.ry)) : 0;
}

// A star built in kernel axis order and checked, not yet part of the context: every refusal of a star happens in
// build_star, before set_star or set_model changes anything.
struct StarBuild {
  std::vector<FS> fs;  // the caller's entries, caller axis order
  PullStar ps;         // the pull star in kernel axis order
};

static int build_star(const sweeptt_ctx* c, const FS* fs, int starsize, const int* perm, const char* who, StarBuild* out) {
  out->fs.assign(fs, fs + starsize);  // (fs may alias c->fs)
  std::vector<FS> pf(out->fs);
  if (perm)
    for (auto& e : pf) {
      const int o[3] = {e.i, e.j, e.k};
      e.i = o[perm[0]]; e.j = o[perm[1]]; e.k = o[perm[2]];
    }
  const PullStar& ps = out->ps = build_pull_star(pf.data(), starsize, c->opts.star_used);
  if (ps.bad_d >= 0) {
    const FS& e = out->fs[ps.bad_d];
    return fail("%s: entry %d (%d,%d,%d) has distance d = %g; every used entry needs a finite d >= 0 (a negative d "
                "gives travel times that are not bounded below)", who, ps.bad_d, e.i, e.j, e.k, (double)e.d);
  }
  if (ps.all.empty()) return fail("%s: the star has no usable offsets", who);
  if (c->opts.kernel == SWEEPTT_KERNEL_TILED && tiled_rxy(ps) == 0)
    return fail("%s: the tiled kernel holds |i|,|j| <= %d, |k| <= %d and <= %d guarded offsets; this star needs "
                "(%d,%d,%d) / %d in kernel axis order", who, RXY_MAX, KHALO, MAX_EXTRA, ps.rx, ps.ry, ps.rz,
                (int)ps.extra.size());
  return 1;
}

// Makes a built star the context's star (fails only on a CUDA error).
static int commit_star(sweeptt_ctx* c, StarBuild& b) {
  std::vector<StarDev> sd(b.ps.all.size());
  for (size_t l = 0; l < sd.size(); ++l) {
    const PullOffset& p = b.ps.all[l];
    sd[l] = StarDev{p.i, p.j, p.k, p.hd, p.guarded};
  }
  CK(cudaStreamSynchronize(c->stream));
  cudaFree(c->d_star);
  c->d_star = nullptr;
  c->have_star = false;
  CK(cudaMalloc(&c->d_star, sd.size() * sizeof(StarDev)));
  CK(cudaMemcpy(c->d_star, sd.data(), sd.size() * sizeof(StarDev), cudaMemcpyHostToDevice));
  c->fs.swap(b.fs);
  c->star = std::move(b.ps);
  c->nstar = (int)sd.size();
  c->have_star = true;
  c->star_gen += 1;
  c->consts_rxy = -1;
  invalidate_graph(c);
  if (!choose_kernel(c)) return 0;
  if (c->have_model && !build_tile_pulls(c)) return 0;
  return 1;
}

extern "C" int sweeptt_set_model(sweeptt_ctx* c, const float* slowness, int nx, int ny, int nz) {
  if (!c || !slowness) return fail("sweeptt_set_model: null argument");
  if (nx <= 0 || ny <= 0 || nz <= 0) return fail("sweeptt_set_model: bad dimensions %d x %d x %d", nx, ny, nz);
  CK(cudaSetDevice(c->device));
  BoxGeom g{};
  if (!compute_geometry(c, nx, ny, nz, &g)) return 0;
  nx = g.nx; ny = g.ny; nz = g.nz;  // from here on: kernel axis order
  const bool same = c->have_model && c->g.px == g.px && c->g.py == g.py && c->g.pz == g.pz;
  const bool perm_changed = !c->have_model || std::memcmp(c->g.perm, g.perm, sizeof g.perm) != 0;
  // check the model, and the star in the model's kernel axis order (the star tables are kept in that order), before
  // anything of the context changes: a refused model leaves the previous model, star and sources
  const bool rebuild_star = c->have_star && perm_changed;
  StarBuild sb;
  if (rebuild_star && !build_star(c, c->fs.data(), (int)c->fs.size(), g.perm, "sweeptt_set_model", &sb)) return 0;
  const size_t dense = (size_t)nx * ny * nz;
  if (!ensure_stage(c, dense)) return 0;
  unsigned r[8];
  {
    // exact minimum of the model: lower bound of every edge delay for the downwind filter; the largest finite and
    // the smallest positive value bound the domain (ready()); the mean of the finite values only scales the
    // activation bucket (scheduling, never the arithmetic).  One device pass instead of a host loop.
    CK(cudaMemcpyAsync(c->d_stage, slowness, dense * 4, cudaMemcpyHostToDevice, c->stream));
    CK(launch_min_slowness(c->d_stage, (long long)dense, reinterpret_cast<unsigned*>(c->d_viol), c->stream));
    CK(cudaMemcpyAsync(r, c->d_viol, sizeof r, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (r[1])
      return fail("sweeptt_set_model: the model holds negative or NaN slowness values (travel times would not be "
                  "bounded below; the reference itself never converges on such input)");
  }
  if (!same) {
    dev_free(c, c->d_slow, (size_t)c->g.vol * 4);
    c->d_slow = nullptr;
    dev_free(c, c->d_tt, (size_t)c->g.vol * 4 * c->tt_cap);
    c->d_tt = nullptr; c->tt_cap = 0; c->have_sources = false;
    c->have_model = false;
    c->maps_valid = false;
    invalidate_graph(c);
    if (!dev_alloc(c, (void**)&c->d_slow, (size_t)g.vol * 4)) return 0;
  }
  c->g = g;
  CK(launch_fill(c->d_slow, g.vol, std::numeric_limits<float>::infinity(), c->stream));
  CK(launch_pad_box(c->d_stage, c->d_slow, g, c->stream));
  {
    float vmin;
    std::memcpy(&vmin, &r[0], 4);
    c->min_slowness = !std::isfinite(vmin) ? -1.f : vmin;
    std::memcpy(&c->max_slowness, &r[6], 4);
    std::memcpy(&c->pos_slowness, &r[7], 4);
    double sum;
    unsigned long long cnt;
    std::memcpy(&sum, &r[2], 8);
    std::memcpy(&cnt, &r[4], 8);
    c->mean_slowness = cnt ? sum / (double)cnt : 0.0;
    invalidate_graph(c);
  }
  c->have_model = true;
  if (perm_changed) c->have_sources = false;
  if (rebuild_star) return commit_star(c, sb);
  if (c->have_star && !build_tile_pulls(c)) return 0;
  return 1;
}

static int build_tile_pulls(sweeptt_ctx* c) {
  // per tile position: in-bounds pulls of one visit.  Memoised on the per-axis clipping
  // class so only O(5^3) distinct products are evaluated.
  const BoxGeom& g = c->g;
  // (a repeated sweeptt_solve on the same geometry and star keeps its table: the cudaFree/cudaMalloc pair below
  //  costs more than the upload of a 241x241x51 model)
  const int sig[7] = {g.nx, g.ny, g.nz, g.perm[0], g.perm[1], g.perm[2], c->star_gen};
  if (c->d_tile_pulls && std::memcmp(sig, c->pulls_sig, sizeof sig) == 0) return 1;
  auto axis_classes = [&](int nt, int T, int n, int r, std::vector<int>& cls, std::vector<std::pair<int, int>>& rep) {
    cls.resize(nt);
    std::map<std::vector<int>, int> seen;
    for (int t = 0; t < nt; ++t) {
      const int lo = t * T, hi = std::min(n, lo + T);
      std::vector<int> sig;
      for (int o = -r; o <= r; ++o) sig.push_back(std::max(0, std::min(hi, n - o) - std::max(lo, -o)));
      auto it = seen.find(sig);
      if (it == seen.end()) {
        it = seen.emplace(sig, (int)rep.size()).first;
        rep.push_back({lo, hi});
      }
      cls[t] = it->second;
    }
  };
  std::vector<int> cx, cy, cz;
  std::vector<std::pair<int, int>> rx, ry, rz;
  axis_classes(g.ntx, TX, g.nx, c->star.rx, cx, rx);
  axis_classes(g.nty, TY, g.ny, c->star.ry, cy, ry);
  axis_classes(g.ntz, TZ, g.nz, c->star.rz, cz, rz);
  std::map<std::tuple<int, int, int>, unsigned long long> memo;
  std::vector<unsigned long long> table((size_t)g.ntx * g.nty * g.ntz);
  for (int tx = 0; tx < g.ntx; ++tx)
    for (int ty = 0; ty < g.nty; ++ty)
      for (int tz = 0; tz < g.ntz; ++tz) {
        auto key = std::make_tuple(cx[tx], cy[ty], cz[tz]);
        auto it = memo.find(key);
        if (it == memo.end()) {
          const auto& X = rx[cx[tx]]; const auto& Y = ry[cy[ty]]; const auto& Z = rz[cz[tz]];
          it = memo.emplace(key, (unsigned long long)count_pulls(c->star, g.nx, g.ny, g.nz, X.first, X.second, Y.first,
                                                                  Y.second, Z.first, Z.second)).first;
        }
        table[((size_t)tx * g.nty + ty) * g.ntz + tz] = it->second;
      }
  c->pulls_per_round = count_pulls(c->star, g.nx, g.ny, g.nz, 0, g.nx, 0, g.ny, 0, g.nz);
  CK(cudaStreamSynchronize(c->stream));
  cudaFree(c->d_tile_pulls);
  c->d_tile_pulls = nullptr;
  CK(cudaMalloc(&c->d_tile_pulls, table.size() * 8));
  CK(cudaMemcpy(c->d_tile_pulls, table.data(), table.size() * 8, cudaMemcpyHostToDevice));
  std::memcpy(c->pulls_sig, sig, sizeof sig);
  return 1;
}

extern "C" int sweeptt_set_star(sweeptt_ctx* c, const struct FS* fs, int starsize) {
  if (!c || !fs) return fail("sweeptt_set_star: null argument");
  if (starsize < 2) return fail("sweeptt_set_star: a forward star needs at least 2 entries (the last one is unused)");
  CK(cudaSetDevice(c->device));
  // kernel axis order: identity until a model has been set (set_model re-builds the star when the order changes)
  StarBuild b;
  if (!build_star(c, fs, starsize, c->have_model ? c->g.perm : nullptr, "sweeptt_set_star", &b)) return 0;
  return commit_star(c, b);
}

static int choose_kernel(sweeptt_ctx* c) {
  const int want = c->opts.kernel;
  int rxy = tiled_rxy(c->star);
  if (want == SWEEPTT_KERNEL_SIMPLE || (want == SWEEPTT_KERNEL_AUTO && rxy == 0)) {
    c->kernel_used = SWEEPTT_KERNEL_SIMPLE;
    return 1;
  }
  // group the columns by k-pattern (ascending mask): the stock-star kernels run one unrolled
  // code block per pattern over a contiguous column range
  std::stable_sort(c->star.columns.begin(), c->star.columns.end(),
                   [](const PullColumn& a, const PullColumn& b) { return a.kmask < b.kmask; });
  std::vector<uint32_t> masks;
  c->pat_begin.clear();
  for (size_t i = 0; i < c->star.columns.size(); ++i)
    if (i == 0 || c->star.columns[i].kmask != c->star.columns[i - 1].kmask) {
      masks.push_back(c->star.columns[i].kmask);
      c->pat_begin.push_back((int)i);
    }
  c->pat_begin.push_back((int)c->star.columns.size());
  c->dev_columns = c->star.columns;
  int stock = 0;
  if ((int)masks.size() <= MAX_PATTERNS && !getenv("SWEEPTT_GENERIC"))
    stock = tiled_stock_star_for(masks.data(), (int)masks.size(), rxy);
  const char* force = getenv("SWEEPTT_FORCE_RXY");  // testing: run a small star in a wider halo variant
  if (force && atoi(force) >= rxy) { rxy = tiled_variant_for_radius(atoi(force)); stock = 0; }
  CK(tiled_prepare(rxy, stock, c->device, &c->tl));
  if (!stock) {
    // generic kernel (it reads every column's mask at run time): the column groups are plain chunks of the list
    const int nw = c->tl.nw;
    const int ncols = (int)c->dev_columns.size();
    std::vector<int> gbeg;
    const int per = std::max(nw, (ncols + MAX_PATTERNS - 1) / MAX_PATTERNS);
    for (int i = 0; i < ncols; i += per) gbeg.push_back(i);
    gbeg.push_back(ncols);
    c->pat_begin = gbeg;
  }
  c->kernel_used = SWEEPTT_KERNEL_TILED;
  c->maps_valid = false;
  c->consts_rxy = -1;
  return 1;
}

// Host image of the context's __constant__ tables (rebuilt after set_star / a kernel change) and its content hash.
static int build_const_image(sweeptt_ctx* c) {
  if (c->consts_rxy == c->tl.rxy && c->consts_nx == c->g.nx) return 1;
  int sxd, syd, szd;
  tiled_variant_dims(c->tl.rxy, &sxd, &syd, &szd);
  {
    // Share the star's columns out between the compute warps (kernels.cu, c_pdesc).  Column groups: the
    // k-pattern groups for a stock-star kernel (one unrolled code block each), else plain chunks of the
    // column list.  Every warp walks ALL groups in the same order and runs a contiguous piece of each, so
    // the pieces of a group are just cut points.  Per tile position along x (interior / first / last tile):
    // three layouts -- a tile with one live unit spreads it over all nw warps (table 0); with two live units
    // each gets nw/2 warps (tables 1 and 2) -- times two sets of head starts (round-based / single-launch
    // kernels; cost units, 1 unit = one k offset of one column): the unit owners finish the tile (min cells,
    // pin, stores), the feeder warp drives the TMA ring, the finisher warp wakes the neighbours and keeps the
    // books.  At the first and last tile along x only the columns that can reach a node INSIDE the grid from
    // some in-grid lane of the unit are shared out (columns are sorted by i within a group, so they stay a
    // contiguous sub-range); the others would only evaluate pulls across the box boundary.
    const int nw = c->tl.nw;
    const std::vector<int>& gbeg = c->pat_begin;
    const int ngroups = (int)gbeg.size() - 1;
    double bias[2][3];
    std::memcpy(bias, kDefaultBias, sizeof bias);
    if (const char* e = getenv("SWEEPTT_BIAS"))
      sscanf(e, "%lf,%lf,%lf,%lf,%lf,%lf", &bias[0][0], &bias[0][1], &bias[0][2], &bias[1][0], &bias[1][1], &bias[1][2]);
    std::vector<uint32_t> kmasks(c->dev_columns.size());
    for (size_t i = 0; i < kmasks.size(); ++i) kmasks[i] = c->dev_columns[i].kmask;
    double col_overhead = 1.5;  // window loads + set-up of a column, in units of one k offset
    if (const char* e = getenv("SWEEPTT_COLCOST")) col_overhead = atof(e);
    const bool clip = !getenv("SWEEPTT_NO_XCLIP");
    c->psplit.assign((size_t)NXCLASS * 6 * MAX_PATTERNS * (MAX_WARPS + 1), 0);
    for (int xc = 0; xc < NXCLASS; ++xc) {
      GroupRange ur[2];
      const int tx = xc == 0 ? -1 : xc == 1 ? 0 : c->g.ntx - 1;
      for (int u = 0; u < 2; ++u) {
        // i range of unit u's columns that connect an in-grid lane with an in-grid node
        int imin = -RXY_MAX - 1, imax = RXY_MAX + 1;
        if (clip && tx >= 0) {
          const int xlo = tx * TX + 4 * u, xhi = std::min(xlo + 3, c->g.nx - 1);
          if (xlo <= xhi) { imin = -xhi; imax = c->g.nx - 1 - xlo; }
        }
        ur[u].first.resize(ngroups); ur[u].end.resize(ngroups);
        for (int g = 0; g < ngroups; ++g) {
          int f = gbeg[g], e = gbeg[g + 1];
          bool sorted = true;  // (columns of a group come in (i,j) order; anything else keeps the whole group)
          for (int col = gbeg[g] + 1; col < gbeg[g + 1]; ++col) sorted = sorted && c->dev_columns[col - 1].i <= c->dev_columns[col].i;
          if (sorted) {
            while (f < e && c->dev_columns[f].i < imin) ++f;
            while (e > f && c->dev_columns[e - 1].i > imax) --e;
          }
          ur[u].first[g] = f; ur[u].end[g] = e;
        }
      }
      std::vector<unsigned short> ps;
      std::vector<double> loads;
      split_columns(kmasks, gbeg, nw, MAX_PATTERNS, MAX_WARPS, bias, &ps, &loads, col_overhead, ur);
      std::copy(ps.begin(), ps.end(), c->psplit.begin() + (size_t)xc * 6 * MAX_PATTERNS * (MAX_WARPS + 1));
      if (getenv("SWEEPTT_DEBUG"))
        for (int table = 0; table < 6; ++table) {
          const int parts = table % 3 == 0 ? nw : nw / 2;
          fprintf(stderr, "sweeptt: column split x-class %d table %d loads:", xc, table);
          for (int pt = 0; pt < parts; ++pt) fprintf(stderr, " %.1f", loads[(size_t)table * MAX_WARPS + pt]);
          fprintf(stderr, "\n");
        }
    }
  }
  // columns in upload order (pattern-sorted, even-padded); half-distances re-packed in the same
  // order so that a pattern group's hd values are contiguous; two spare entries at the end
  std::vector<ColumnDev>& cols = c->img_cols;
  std::vector<float>& hd_packed = c->img_hd;
  cols.assign(c->dev_columns.size() + 2, ColumnDev{});
  hd_packed.clear();
  for (size_t i = 0; i < c->dev_columns.size(); ++i) {
    const PullColumn& pc = c->dev_columns[i];
    ColumnDev d;
    d.soff = pc.i * syd * szd + pc.j * szd;
    d.kmask = pc.kmask;
    d.hd_begin = (int)hd_packed.size();
    d.gmask = 0;
    int nk = 0;
    for (int b = 0; b <= 2 * ZHALO; ++b)
      if (pc.kmask & (1u << b)) {
        hd_packed.push_back(c->star.col_hd[pc.hd_begin + nk++]);
        for (int k = 0; k < KZ; ++k) d.gmask |= 1u << ((k + b) / 4);
      }
    cols[i] = d;
  }
  cols[cols.size() - 2] = cols[cols.size() - 1] = cols[c->dev_columns.size() - 1];
  if ((int)hd_packed.size() > MAX_COL_HD || (int)cols.size() > MAX_COLUMNS)
    return fail("star tables exceed the __constant__ budget (%zu half-distances, %zu columns)", hd_packed.size(), cols.size());
  std::vector<ExtraDev>& ex = c->img_extra;
  ex.assign(c->star.extra.size(), ExtraDev{});
  for (size_t i = 0; i < ex.size(); ++i) {
    const PullOffset& p = c->star.extra[i];
    ex[i] = ExtraDev{p.i, p.j, p.k, p.i * syd * szd + p.j * szd + p.k, p.hd, p.guarded, 0, 0};
  }
  // per (table, group, part): the part's piece of the group + where its half-distances start (kernels.cu c_pdesc)
  std::vector<unsigned>& pdesc = c->img_pdesc;
  pdesc.assign((size_t)NXCLASS * 6 * MAX_PATTERNS * MAX_WARPS, 0u);
  for (int table = 0; table < NXCLASS * 6; ++table)
    for (int g = 0; g + 1 < (int)c->pat_begin.size() && g < MAX_PATTERNS; ++g)
      for (int pt = 0; pt < MAX_WARPS; ++pt) {
        const unsigned short* row = &c->psplit[((size_t)table * MAX_PATTERNS + g) * (MAX_WARPS + 1)];
        const unsigned lo = row[pt], hi = row[pt + 1];
        pdesc[((size_t)table * MAX_PATTERNS + g) * MAX_WARPS + pt] =
            lo | (hi << 9) | ((lo < hi ? (unsigned)cols[lo].hd_begin : 0u) << 18);
      }
  uint64_t sig = 1469598103934665603ull;
  auto mix = [&sig](const void* p, size_t n) {
    const unsigned char* b = static_cast<const unsigned char*>(p);
    for (size_t i = 0; i < n; ++i) { sig ^= b[i]; sig *= 1099511628211ull; }
  };
  mix(cols.data(), cols.size() * sizeof(ColumnDev));
  mix(hd_packed.data(), hd_packed.size() * sizeof(float));
  mix(ex.data(), ex.size() * sizeof(ExtraDev));
  mix(pdesc.data(), pdesc.size() * sizeof(unsigned));
  c->img_sig = sig | 1ull;
  c->consts_rxy = c->tl.rxy;
  c->consts_nx = c->g.nx;
  return 1;
}

// Takes the lease on the device's __constant__ tables for this context's star (uploading them if others are there).
static int upload_constants(sweeptt_ctx* c, ConstLease* lease) {
  if (!build_const_image(c)) return 0;
  if (lease->t) return 1;  // (already held by this call)
  ConstTables& t = const_tables(c->device);
  std::unique_lock<std::mutex> lk(t.mu);
  t.cv.wait(lk, [&] { return t.users == 0 || (t.loaded && t.sig == c->img_sig); });
  if (!(t.loaded && t.sig == c->img_sig)) {
    // nobody holds the old tables; their last kernels were synchronised by the calls that launched them, but a
    // caller-provided stream may still be draining
    CK(cudaDeviceSynchronize());
    t.loaded = false;
    CK(upload_star_constants(c->img_cols.data(), (int)c->img_cols.size(), c->img_hd.data(), (int)c->img_hd.size(),
                             c->img_extra.data(), (int)c->img_extra.size(), c->img_pdesc.data(), (int)c->img_pdesc.size(),
                             c->stream));
    CK(cudaStreamSynchronize(c->stream));
    t.sig = c->img_sig;
    t.loaded = true;
  }
  ++t.users;
  lease->t = &t;
  return 1;
}

static int build_maps(sweeptt_ctx* c) {
  if (c->maps_valid) return 1;
  auto enc = get_encode_fn();
  if (!enc) return fail("cuTensorMapEncodeTiled not available from this driver");
  const BoxGeom& g = c->g;
  int sxd, syd, szd;
  tiled_variant_dims(c->tl.rxy, &sxd, &syd, &szd);
  {
    cuuint64_t dims[3] = {(cuuint64_t)g.pz, (cuuint64_t)g.py, (cuuint64_t)(c->slow_pb ? c->slow_planes : g.px)};
    cuuint64_t strides[2] = {(cuuint64_t)g.pz * 4, (cuuint64_t)g.sx * 4};
    cuuint32_t box[3] = {(cuuint32_t)szd, (cuuint32_t)syd, (cuuint32_t)sxd};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = enc(&c->tm_slow, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, c->d_slow, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(slowness) failed: %d", (int)r);
  }
  if (!encode_tt_map(c, c->d_tt, std::max(1, c->tt_cap), &c->tm_tt)) return 0;
  c->maps_valid = true;
  invalidate_graph(c);
  return 1;
}

static int encode_tt_map(sweeptt_ctx* c, float* base, int nboxes, CUtensorMap* out) {
  auto enc = get_encode_fn();
  if (!enc) return fail("cuTensorMapEncodeTiled not available from this driver");
  const BoxGeom& g = c->g;
  int sxd, syd, szd;
  tiled_variant_dims(c->tl.rxy, &sxd, &syd, &szd);
  cuuint64_t dims[4] = {(cuuint64_t)g.pz, (cuuint64_t)g.py, (cuuint64_t)g.px, (cuuint64_t)nboxes};
  cuuint64_t strides[3] = {(cuuint64_t)g.pz * 4, (cuuint64_t)g.sx * 4, (cuuint64_t)g.vol * 4};
  cuuint32_t box[4] = {(cuuint32_t)szd, (cuuint32_t)syd, (cuuint32_t)sxd, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(travel times) failed: %d", (int)r);
  return 1;
}

extern "C" int sweeptt_set_sources(sweeptt_ctx* c, const struct START* starts, int numstart) {
  if (!c || !starts) return fail("sweeptt_set_sources: null argument");
  if (!c->have_model) return fail("sweeptt_set_sources: set the model first");
  if (numstart <= 0) return fail("sweeptt_set_sources: need at least one start point");
  CK(cudaSetDevice(c->device));
  const BoxGeom& g = c->g;
  int on[3];  // caller-order dims
  on[g.perm[0]] = g.nx; on[g.perm[1]] = g.ny; on[g.perm[2]] = g.nz;
  for (int s = 0; s < numstart && !c->allow_outside_sources; ++s)
    if (starts[s].i < 0 || starts[s].i >= on[0] || starts[s].j < 0 || starts[s].j >= on[1] || starts[s].k < 0 ||
        starts[s].k >= on[2])
      return fail("start point %d (%d,%d,%d) is outside the %d x %d x %d model", s, starts[s].i, starts[s].j,
                  starts[s].k, on[0], on[1], on[2]);
  CK(cudaStreamSynchronize(c->stream));
  if (numstart > c->tt_cap) {  // grow the pool
    dev_free(c, c->d_tt, (size_t)g.vol * 4 * c->tt_cap);
    c->d_tt = nullptr; c->tt_cap = 0;
    if (!dev_alloc(c, (void**)&c->d_tt, (size_t)g.vol * 4 * numstart)) return 0;
    c->tt_cap = numstart;
    c->maps_valid = false;
    invalidate_graph(c);
  }
  if (numstart > c->src_cap) {
    cudaFree(c->d_src);
    c->d_src = nullptr;
    CK(cudaMalloc(&c->d_src, sizeof(int) * 3 * numstart));
    c->src_cap = numstart;
    invalidate_graph(c);
  }
  const size_t ntiles = (size_t)g.ntx * g.nty * g.ntz;
  if (ntiles * numstart > 0xfffffff0ull) return fail("too many tiles (%zu x %d sources) for 32-bit work-list entries", ntiles, numstart);
  if (ntiles * numstart > c->tiles_cap) {
    dev_free(c, c->d_worklist, c->tiles_cap * 16);
    dev_free(c, c->d_key, (c->tiles_cap + 4) * 4);
    dev_free(c, c->d_tmax, (c->tiles_cap + 4) * 4);
    dev_free(c, c->d_busy, (c->tiles_cap + 4) * 4);
    dev_free(c, c->d_keysnap, (c->tiles_cap + 4) * 4);
    c->d_worklist = nullptr; c->d_key = nullptr; c->d_tmax = nullptr; c->d_busy = nullptr; c->d_keysnap = nullptr;
    c->tiles_cap = ntiles * numstart;
    if (!dev_alloc(c, (void**)&c->d_worklist, c->tiles_cap * 16)) return 0;
    if (!dev_alloc(c, (void**)&c->d_key, (c->tiles_cap + 4) * 4)) return 0;
    if (!dev_alloc(c, (void**)&c->d_tmax, (c->tiles_cap + 4) * 4)) return 0;
    if (!dev_alloc(c, (void**)&c->d_busy, (c->tiles_cap + 4) * 4)) return 0;
    if (!dev_alloc(c, (void**)&c->d_keysnap, (c->tiles_cap + 4) * 4)) return 0;
    invalidate_graph(c);
  }
  if (numstart != c->nsrc) invalidate_graph(c);
  c->nsrc = numstart;
  c->src_xyz.resize(3 * numstart);
  for (int s = 0; s < numstart; ++s) {
    const int o[3] = {starts[s].i, starts[s].j, starts[s].k};
    for (int q = 0; q < 3; ++q) c->src_xyz[3 * s + q] = o[g.perm[q]];
  }
  CK(cudaMemcpy(c->d_src, c->src_xyz.data(), sizeof(int) * 3 * numstart, cudaMemcpyHostToDevice));
  c->have_sources = true;
  return 1;
}

static RelaxArgs make_args(sweeptt_ctx* c) {
  RelaxArgs a{};
  a.g = c->g;
  a.slow = c->d_slow;
  a.tt = c->d_tt;
  a.nsrc = c->nsrc;
  a.src_xyz = c->d_src;
  a.st = c->d_state;
  a.worklist = c->d_worklist;
  a.cap = (unsigned)((size_t)c->nsrc * c->g.ntx * c->g.nty * c->g.ntz);
  a.key = c->d_key;
  a.busy = c->d_busy;
  a.keysnap = c->d_keysnap;
  {
    // downwind filter (kernels.cu): needs non-negative slowness; dmin = fl(hd_min * fl(vmin + vmin)) bounds
    // every fl(hd * fl(v_n + v_m)) from below because rounding is monotone
    static const bool off = getenv("SWEEPTT_NO_TMAX") != nullptr;
    a.tmax = (!off && c->min_slowness >= 0.f) ? c->d_tmax : nullptr;
    float hdmin = std::numeric_limits<float>::infinity();
    for (const auto& p : c->star.all) hdmin = std::min(hdmin, p.hd);
    const float two_v = c->min_slowness + c->min_slowness;
    a.dmin = (a.tmax && std::isfinite(hdmin) && hdmin > 0.f) ? hdmin * two_v : 0.f;
  }
  a.bucket = c->bucket;
  a.bin_scale = c->bucket > 0.f ? 32.0f / c->bucket : 0.f;
  a.tile_pulls = c->d_tile_pulls;
  a.ncols = (int)c->dev_columns.size();
  a.nextra = (int)c->star.extra.size();
  a.neg_zero = -0.0f;
  a.max_inner = c->max_inner;
  a.nparts = c->mp_nparts; a.part = c->mp_part;
  a.tx_owner = c->d_tx_owner; a.tx_slow0 = c->d_tx_slow0;
  a.slow_pb = c->slow_pb;
  {
    static const double slack = getenv("SWEEPTT_FRONT_SLACK") ? atof(getenv("SWEEPTT_FRONT_SLACK")) : 1.0;  // in buckets
    a.front_slack = c->bucket > 0.f ? (float)(slack * c->bucket) : 0.f;
  }
  static const bool own_front = getenv("SWEEPTT_NO_GLOBAL_KMIN") != nullptr;  // (experiment: every part follows its own front)
  for (int q = 0; q < MAX_PARTS; ++q) {
    a.part_key[q] = c->mp_key[q];
    a.part_tmax[q] = a.tmax ? c->mp_tmax[q] : nullptr;
    a.part_kmin[q] = own_front ? c->mp_kmin[c->mp_part] : c->mp_kmin[q];
  }
  for (size_t i = 0; i < c->pat_begin.size() && i <= (size_t)MAX_PATTERNS; ++i) a.pat_begin[i] = c->pat_begin[i];
  a.npat = (int)c->pat_begin.size() - 1;
  {
    double look = 16.0;  // in tiles per persistent CTA (measured on config 2: 0 -> 14.1 ms, 1.5 -> 13.8, 2.5 -> 13.4, 4 -> 12.9, 8 -> 12.9;
                         // a wave of 8 sources: 4 -> 27.6 ms, 8 -> 25.0, 16 -> 24.3, 32 -> 24.4)
    if (const char* e = getenv("SWEEPTT_LOOKAHEAD")) look = atof(e);
    a.lookahead = (unsigned)std::max(0.0, look * c->tl.grid_persistent);
    double frac = 0.4;  // (0.9 -> 14.8 ms, 0.6 -> 13.1, 0.4 -> 12.9, 0.1 -> 13.2)
    if (const char* e = getenv("SWEEPTT_TRIGGER_FRAC")) frac = atof(e);
    a.trig_q8 = (unsigned)std::min(255.0, std::max(0.0, frac * 256.0));
  }
  return a;
}

// The kernels evaluate an edge delay as fl(hd * fl(v_n + v_m)) with hd = fl(0.5f * d), the reference as
// fl(fl(d * fl(v_n + v_m)) / 2.0).  The two agree for every edge of the model and star when (DESIGN §1)
//   fl(dmax * fl(vmax + vmax)) is finite    (else the reference's product overflows where the kernels' does not),
//   every positive d is >= 2^-125            (else hd = 0.5f * d rounds),
//   fl(dpos * vpos) >= 2^-125                (else the reference's halving rounds a second time, in the subnormals),
// with dmax / dpos the largest / smallest positive d of the star's edges and vmax / vpos the largest finite /
// smallest positive slowness (every fl(v_n + v_m) that is not 0 is >= vpos).  A model and star outside are refused.
static int check_domain(const sweeptt_ctx* c) {
  const float lo = std::ldexp(1.f, -125);
  const PullStar& s = c->star;
  if (s.dpos < lo)
    return fail("star distance d = %g is below 2^-125: 0.5f * d would round, the kernels' delays would differ from "
                "the reference's d * (v_n + v_m) / 2.0", (double)s.dpos);
  const float two_v = c->max_slowness + c->max_slowness;
  if (std::isinf(s.dmax * two_v))
    return fail("slowness %g with star distance %g: d * (v + v) = inf overflows float (the largest slowness must keep "
                "dmax * 2 vmax <= FLT_MAX), the kernels' delays would differ from the reference's d * (v_n + v_m) / 2.0",
                (double)c->max_slowness, (double)s.dmax);
  if (s.dpos * c->pos_slowness < lo)
    return fail("slowness %g with star distance %g: d * v = %g is below 2^-125 (the smallest positive slowness must keep "
                "dpos * vpos >= 2^-125), the kernels' delays would differ from the reference's d * (v_n + v_m) / 2.0",
                (double)c->pos_slowness, (double)s.dpos, (double)(s.dpos * c->pos_slowness));
  return 1;
}

static int ready(sweeptt_ctx* c, ConstLease* lease) {
  if (!c) return fail("null context");
  if (!c->have_model || !c->have_star || !c->have_sources) return fail("context needs a model, a star and start points first");
  if (!check_domain(c)) return 0;
  CK(cudaSetDevice(c->device));
  if (c->kernel_used == SWEEPTT_KERNEL_TILED) {
    if (!build_maps(c)) return 0;
    if (!upload_constants(c, lease)) return 0;
    // activation bucket = factor x (delay of the longest star edge in a medium of mean slowness)
    double factor = 2.0;  // measured on config 2: 1 -> 21.9 ms, 2 -> 21.2 ms, 4 -> 21.4 ms, off -> 50 ms
    if (const char* e = getenv("SWEEPTT_BUCKET")) factor = atof(e);
    float hdmax = 0.f;
    for (const auto& p : c->star.all) hdmax = std::max(hdmax, p.hd);
    {
      // in-tile passes per visit: pays when the star radius is small next to the 8x8x8 tile (measured on the
      // 241x241x51 box: 3-FS 5.1 -> 2.8 ms with 4 passes, 5-FS 9.3 -> 8.6 ms with 2, 818-FS 12.9 -> 13.6 ms)
      int mi = c->tl.rxy <= 2 ? 4 : c->tl.rxy <= 4 ? 2 : 1;
      if (const char* e = getenv("SWEEPTT_INNER")) mi = std::max(1, atoi(e));
      if (mi != c->max_inner) { c->max_inner = mi; invalidate_graph(c); }
    }
    const float b = (factor > 0 && c->mean_slowness > 0) ? (float)(factor * 2.0 * hdmax * c->mean_slowness) : -1.f;
    if (b != c->bucket) { c->bucket = b; invalidate_graph(c); }
  }
  return 1;
}

extern "C" int sweeptt_reset(sweeptt_ctx* c) {
  ConstLease lease;
  if (!ready(c, &lease)) return 0;
  CK(launch_reset(make_args(c), c->opts.max_rounds, c->stream));
  return 1;
}

static int read_state(sweeptt_ctx* c) {
  CK(cudaMemcpyAsync(c->h_state, c->d_state, sizeof(SolveState), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 1;
}

// CUDA graph: WHILE(cond) { relax; compact -> sets cond }  -- the whole convergence loop is
// one graph launch; the host is not consulted between rounds.
static int encode_tt_map(sweeptt_ctx* c, float* base, int nboxes, CUtensorMap* out);

static int build_while_graph(sweeptt_ctx* c, const RelaxArgs& a, const CUtensorMap& tm_tt, cudaStream_t stream,
                             cudaGraphExec_t* exec) {
  cudaGraph_t graph = nullptr;
  CK(cudaGraphCreate(&graph, 0));
  cudaGraphConditionalHandle handle;
  cudaError_t e = cudaGraphConditionalHandleCreate(&handle, graph, 1, cudaGraphCondAssignDefault);
  if (e != cudaSuccess) { cudaGraphDestroy(graph); return fail("cudaGraphConditionalHandleCreate: %s", cudaGetErrorString(e)); }
  cudaGraphNodeParams np = {cudaGraphNodeTypeConditional};
  np.conditional.handle = handle;
  np.conditional.type = cudaGraphCondTypeWhile;
  np.conditional.size = 1;
  cudaGraphNode_t node;
  e = cudaGraphAddNode(&node, graph, nullptr, 0, &np);
  if (e != cudaSuccess) { cudaGraphDestroy(graph); return fail("cudaGraphAddNode(conditional): %s", cudaGetErrorString(e)); }
  cudaGraph_t body = np.conditional.phGraph_out[0];
  e = cudaStreamBeginCaptureToGraph(stream, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed);
  if (e != cudaSuccess) { cudaGraphDestroy(graph); return fail("cudaStreamBeginCaptureToGraph: %s", cudaGetErrorString(e)); }
  int ok = 1;
  if (c->kernel_used == SWEEPTT_KERNEL_TILED) {
    ok = launch_relax_tiled(c->tl, c->tm_slow, tm_tt, a, stream) == cudaSuccess &&
         launch_compact(a, (unsigned long long)handle, stream) == cudaSuccess;
  } else {
    ok = launch_relax_simple(a, c->d_star, c->nstar, (unsigned long long)c->pulls_per_round * a.nsrc, stream) == cudaSuccess &&
         launch_advance_simple(a.st, (unsigned long long)handle, stream) == cudaSuccess;
  }
  cudaGraph_t dummy = nullptr;
  e = cudaStreamEndCapture(stream, &dummy);
  if (!ok || e != cudaSuccess) { cudaGraphDestroy(graph); return fail("capturing the relaxation loop failed: %s", cudaGetErrorString(e)); }
  e = cudaGraphInstantiate(exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e != cudaSuccess) { *exec = nullptr; return fail("cudaGraphInstantiate: %s", cudaGetErrorString(e)); }
  return 1;
}

// CUDA graph: WHILE(cond) { relax; compact -> sets cond }  -- the whole convergence loop is
// one graph launch; the host is not consulted between rounds.
static int build_graph(sweeptt_ctx* c) {
  if (c->graph_valid) return 1;
  if (c->graph_exec) cudaGraphExecDestroy(c->graph_exec);
  c->graph_exec = nullptr;
  if (!build_while_graph(c, make_args(c), c->tm_tt, c->stream, &c->graph_exec)) return 0;
  c->graph_valid = true;
  return 1;
}

// the part of the context that a slice of the solve plan works on
static RelaxArgs slice_args(sweeptt_ctx* c, const sweeptt_ctx::Slice& sl) {
  RelaxArgs a = make_args(c);
  const size_t ntiles = (size_t)c->g.ntx * c->g.nty * c->g.ntz;
  a.tt = c->d_tt + (size_t)sl.s0 * c->g.vol;
  a.nsrc = sl.ns;
  a.src_xyz = c->d_src + 3 * sl.s0;
  a.st = c->d_state + sl.slot;
  a.cap = (unsigned)(ntiles * sl.ns);
  a.worklist = c->d_worklist + 4 * ntiles * sl.s0;  // each slice owns 4*cap consecutive entries
  a.key = c->d_key + ntiles * sl.s0;
  a.busy = c->d_busy + ntiles * sl.s0;
  a.keysnap = c->d_keysnap + ntiles * sl.s0;
  if (a.tmax) a.tmax = c->d_tmax + ntiles * sl.s0;
  return a;
}

static int env_loop(const sweeptt_ctx* c) {
  int loop = c->opts.loop;
  if (const char* env = getenv("SWEEPTT_LOOP")) {
    if (!strcmp(env, "graph")) loop = SWEEPTT_LOOP_GRAPH;
    if (!strcmp(env, "batched")) loop = SWEEPTT_LOOP_BATCHED;
  }
  return loop;
}

// How many sources ONE persistent launch can take (0: the single-launch scheduler is not used).
static int persistent_capacity(sweeptt_ctx* c) {
  if (c->kernel_used != SWEEPTT_KERNEL_TILED || c->opts.max_rounds > 0) return 0;
  // the 3-FS kernel (three 4-warp CTAs per SM, tiles of a few hundred nanoseconds) spends its time in list
  // switches: measured 4.6 ms against 2.8 ms for the graph of rounds (config 1) -- unless asked for explicitly
  if (c->tl.nw < MAX_WARPS && !getenv("SWEEPTT_PERSIST")) return 0;
  if (const char* e = getenv("SWEEPTT_PERSIST")) { if (atoi(e) == 0) return 0; }
  if (env_loop(c) == SWEEPTT_LOOP_BATCHED) return 0;
  // One CTA builds every list.  While all keys fit its idle TMA ring (53 Ki keys for 818-FS: 8 sources on a
  // 241x241x51 box) a build takes a few microseconds and hides behind the early-build lookahead; with a
  // snapshot in global memory it does not (measured: 16 sources 65 ms against 50 ms for the graph of rounds).
  // More sources than that run as consecutive waves of persistent launches (build_plan).
  size_t max_keys = tiled_persistent_max_keys(c->tl.rxy);
  if (const char* e = getenv("SWEEPTT_PERSIST_MAX_KEYS")) max_keys = (size_t)atoll(e);
  const size_t ntiles = (size_t)c->g.ntx * c->g.nty * c->g.ntz;
  return (int)std::min<size_t>(max_keys / ntiles, 1u << 20);
}

// Cut the sources into waves and slices (sweeptt_ctx::Slice) and prepare each slice's tensor map / graph.
static int build_plan(sweeptt_ctx* c) {
  if (c->plan_valid) return 1;
  invalidate_graph(c);
  const int cap = persistent_capacity(c);
  int wave_size = 0;  // sources per wave
  bool persistent = false;
  if (cap >= 1) {
    // balanced waves of at most `cap` sources, e.g. 111 sources -> 14 waves of 8 (the last one 7)
    const int nwaves = (c->nsrc + cap - 1) / cap;
    wave_size = (c->nsrc + nwaves - 1) / nwaves;
    persistent = true;
  }
  if (const char* e = getenv("SWEEPTT_WAVE")) {  // 0: every source in ONE wave of graph groups (the round-1 scheme)
    const int w = atoi(e);
    if (w <= 0) { wave_size = c->nsrc; persistent = cap >= c->nsrc; }
    else { wave_size = std::min(w, c->nsrc); persistent = cap >= wave_size; }
  }
  if (wave_size <= 0) wave_size = c->nsrc;
  int want_groups = 2;
  if (const char* env = getenv("SWEEPTT_GROUPS")) want_groups = atoi(env);
  want_groups = std::max(1, std::min(want_groups, MAX_GROUPS));
  // Persistent waves may run K at a time, each on 1/K of the SMs (its own stream): a wave's start and end expose
  // fewer ready tiles than there are SMs (the front is small), and the time lost there shrinks with the SMs per wave.
  // (measured on config 3: 111 sources on 1 stream 345.6 / 348.7 ms, 2 streams 338.2 / 346.9 ms, 4 streams 381.7 ms --
  //  but the SMs are split statically, so the stream that runs dry first idles its half: 28 sources in waves of
  //  8+8+8+4 over 2 streams 94.0 ms against 87.2 ms on one.  One stream unless asked for.)
  int kstreams = 1;
  if (const char* e = getenv("SWEEPTT_WAVE_STREAMS")) kstreams = std::max(1, std::min(atoi(e), MAX_GROUPS));
  const int nwaves_total = (c->nsrc + wave_size - 1) / wave_size;
  if (!persistent || nwaves_total < 2 * kstreams) kstreams = 1;
  if (c->opts.profile_kernels) kstreams = 1;  // per-launch event timing: one launch at a time, on the whole device
  // Wave sizes.  Persistent waves of 4 or more sources run at the same rate (measured: 4 sources 0.549 of the roof,
  // 8: 0.549, 7+7: 0.556; ONE source 0.49), and the device->host copies of the LAST wave cannot hide behind any
  // solve, so the last wave is kept small (4 sources) and the others share the rest evenly.
  std::vector<int> sizes;
  if (persistent && c->nsrc > wave_size && c->nsrc >= 8 && !getenv("SWEEPTT_WAVE")) {
    const int last = std::min(4, wave_size);  // (a wave never exceeds what one launch holds)
    const int rest = c->nsrc - last;
    const int nw = (rest + wave_size - 1) / wave_size;
    for (int w = 0; w < nw; ++w) sizes.push_back((int)((long long)rest * (w + 1) / nw - (long long)rest * w / nw));
    sizes.push_back(last);
  } else {
    for (int s0 = 0; s0 < c->nsrc; s0 += wave_size) sizes.push_back(std::min(wave_size, c->nsrc - s0));
  }
  int slot = 1, wave = 0;
  for (int s0 = 0; wave < (int)sizes.size(); s0 += sizes[wave], ++wave) {
    const int ns = sizes[wave];
    const int parts = persistent ? 1 : std::min(want_groups, ns);
    for (int g = 0; g < parts; ++g) {
      sweeptt_ctx::Slice sl;
      sl.wave = persistent ? wave / kstreams : wave;  // (slices of one "wave" are enqueued together)
      sl.s0 = s0 + (int)((long long)ns * g / parts);
      sl.ns = s0 + (int)((long long)ns * (g + 1) / parts) - sl.s0;
      sl.slot = slot++;
      sl.lane = persistent ? wave % kstreams : g;
      sl.grid = (persistent && kstreams > 1) ? std::max(1, c->tl.grid_persistent / kstreams) : 0;
      sl.persistent = persistent;
      if (slot > STATE_SLOTS) return fail("too many slices in the solve plan (%d sources in waves of %d)", c->nsrc, wave_size);
      c->plan.push_back(sl);
    }
  }
  c->plan_waves = persistent ? (wave + kstreams - 1) / kstreams : wave;
  int lanes = 1;
  for (const auto& sl : c->plan) lanes = std::max(lanes, sl.lane + 1);
  while ((int)c->aux_streams.size() < lanes - 1) {
    cudaStream_t st;
    cudaEvent_t ev;
    CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    c->aux_streams.push_back(st);
    c->aux_done.push_back(ev);
  }
  for (auto& sl : c->plan) {
    if (c->kernel_used == SWEEPTT_KERNEL_TILED && !encode_tt_map(c, c->d_tt + (size_t)sl.s0 * c->g.vol, sl.ns, &sl.tm_tt)) return 0;
    if (!sl.persistent) {
      cudaStream_t st = sl.lane ? c->aux_streams[sl.lane - 1] : c->stream;
      if (!build_while_graph(c, slice_args(c, sl), sl.tm_tt, st, &sl.graph)) return 0;
    }
  }
  c->plan_valid = true;
  return 1;
}

static void fill_stats(sweeptt_ctx* c, sweeptt_stats* st, int rounds_before, long long launches, long long relax_launches,
                       double relax_ms) {
  if (!st) return;
  const SolveState& h = *c->h_state;
  st->struct_size = sizeof(sweeptt_stats);
  st->rounds = h.round - rounds_before;
  st->kernel_used = c->kernel_used;
  st->devices_used = 1;
  st->kernel_launches = launches;
  st->relax_launches = relax_launches;
  st->tile_visits = (long long)h.tile_visits;
  st->relaxations = (long long)h.pulls;
  st->relax_kernel_ms = relax_ms;
  st->units_run = (long long)h.units_run;
  st->units_changed = (long long)h.units_changed;
}

static int run_rounds(sweeptt_ctx* c, bool to_convergence, int fixed_rounds, int* changed_out, sweeptt_stats* stats) {
  const RelaxArgs a = make_args(c);
  int loop = c->opts.loop;
  if (const char* env = getenv("SWEEPTT_LOOP")) {
    if (!strcmp(env, "graph")) loop = SWEEPTT_LOOP_GRAPH;
    if (!strcmp(env, "batched")) loop = SWEEPTT_LOOP_BATCHED;
  }
  if (loop == SWEEPTT_LOOP_AUTO) loop = SWEEPTT_LOOP_GRAPH;
  const bool profile = c->opts.profile_kernels != 0;
  if (profile || !to_convergence) loop = SWEEPTT_LOOP_BATCHED;
  int rounds_before = 0;
  if (stats || to_convergence) {  // (a fixed batch without statistics needs no look at the state first)
    if (!read_state(c)) return 0;
    rounds_before = c->h_state->round;
  }
  long long launches = 0, relax_launches = 0;
  double relax_ms = 0;

  if (loop == SWEEPTT_LOOP_GRAPH) {
    if (!build_graph(c)) {
      if (c->opts.loop == SWEEPTT_LOOP_GRAPH) return 0;
      loop = SWEEPTT_LOOP_BATCHED;  // AUTO: fall back to polling
    }
  }
  if (loop == SWEEPTT_LOOP_GRAPH) {
    CK(cudaGraphLaunch(c->graph_exec, c->stream));
    if (!read_state(c)) return 0;
    const int r = c->h_state->round - rounds_before;
    launches = (c->kernel_used == SWEEPTT_KERNEL_TILED ? 3LL : 2LL) * r; relax_launches = r;
  } else {
    const int per_poll = to_convergence ? (c->opts.rounds_per_poll > 0 ? c->opts.rounds_per_poll : 8) : fixed_rounds;
    size_t ev_used = 0;
    for (;;) {
      for (int k = 0; k < per_poll; ++k) {
        if (profile) {
          if (c->prof_events.size() < ev_used + 2) {
            cudaEvent_t e0, e1;
            CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
            c->prof_events.push_back(e0); c->prof_events.push_back(e1);
          }
          CK(cudaEventRecord(c->prof_events[ev_used], c->stream));
        }
        if (c->kernel_used == SWEEPTT_KERNEL_TILED) {
          CK(launch_relax_tiled(c->tl, c->tm_slow, c->tm_tt, a, c->stream));
        } else {
          CK(launch_relax_simple(a, c->d_star, c->nstar, (unsigned long long)c->pulls_per_round * c->nsrc, c->stream));
        }
        if (profile) { CK(cudaEventRecord(c->prof_events[ev_used + 1], c->stream)); ev_used += 2; }
        if (c->kernel_used == SWEEPTT_KERNEL_TILED) { CK(launch_compact(a, 0, c->stream)); }
        else { CK(launch_advance_simple(c->d_state, 0, c->stream)); }
        launches += (c->kernel_used == SWEEPTT_KERNEL_TILED ? 3 : 2); relax_launches += 1;
      }
      if (!read_state(c)) return 0;
      if (profile) {
        for (size_t i = 0; i < ev_used; i += 2) {
          float ms = 0;
          CK(cudaEventElapsedTime(&ms, c->prof_events[i], c->prof_events[i + 1]));
          relax_ms += ms;
        }
        ev_used = 0;
      }
      if (!to_convergence) break;
      const SolveState& h = *c->h_state;
      const bool done = (c->kernel_used == SWEEPTT_KERNEL_TILED) ? (h.count[h.parity] == 0)  // nothing left to relax
                                                                  : (h.last_changed_round < h.round);
      if (done) break;
      if (c->opts.max_rounds > 0 && h.round - rounds_before >= c->opts.max_rounds) break;
      if (c->opts.verbose > 0)
        fprintf(stderr, "[sweeptt] round %d: %u tiles queued, %llu pulls so far\n", h.round, h.count[h.parity], h.pulls);
    }
  }
  if (changed_out)
    *changed_out = (c->kernel_used == SWEEPTT_KERNEL_TILED) ? (c->h_state->count[c->h_state->parity] != 0)
                                                            : (c->h_state->last_changed_round == c->h_state->round);
  fill_stats(c, stats, rounds_before, launches, relax_launches, relax_ms);
  return 1;
}

// Runs the solve plan: every wave is enqueued without waiting for the one before it; `after_wave(s0, ns)` (may be
// empty) is called as soon as a wave's work is on the context's stream -- whatever it enqueues there runs when the
// wave's sources have converged (sweeptt_solve un-pads them and sends them to the host while the next wave runs).
static int run_plan(sweeptt_ctx* c, sweeptt_stats* stats, const std::function<int(int, int, cudaStream_t)>& after_wave) {
  if (!build_plan(c)) return 0;
  const bool profile = c->opts.profile_kernels != 0;  // (persistent waves only: run_plan is not used otherwise)
  size_t ev_used = 0;
  CK(cudaEventRecord(c->ev0, c->stream));
  CK(cudaEventRecord(c->ev_fork, c->stream));
  std::vector<char> lane_used(1 + c->aux_streams.size(), 0);
  auto lane_stream = [&](int lane) -> cudaStream_t {
    cudaStream_t st = lane ? c->aux_streams[lane - 1] : c->stream;
    if (lane && !lane_used[lane]) cudaStreamWaitEvent(st, c->ev_fork, 0);
    lane_used[lane] = 1;
    return st;
  };
  size_t i = 0;
  while (i < c->plan.size()) {
    if (c->plan[i].persistent) {
      // a wave = one single-launch solve; waves on different lanes (streams) never wait for each other
      const auto& sl = c->plan[i];
      cudaStream_t st = lane_stream(sl.lane);
      RelaxArgs a = slice_args(c, sl);
      TiledLaunch tl = c->tl;
      // (early list builds: 8 tiles per CTA ahead for a few sources, 16 for a full wave -- measured: 4 sources 12.45
      //  vs 12.70 ms, 8 sources 25.0 vs 24.3 ms)
      if (sl.ns < 6 && !getenv("SWEEPTT_LOOKAHEAD")) a.lookahead /= 2;
      if (sl.grid > 0) {
        a.lookahead = (unsigned)((unsigned long long)a.lookahead * sl.grid / std::max(1, tl.grid_persistent));
        tl.grid_persistent = sl.grid;
      }
      CK(launch_reset(a, c->opts.max_rounds, st));
      CK(launch_persist_begin(a, st));
      if (profile) {
        while (c->prof_events.size() < ev_used + 2) {
          cudaEvent_t e;
          CK(cudaEventCreate(&e));
          c->prof_events.push_back(e);
        }
        CK(cudaEventRecord(c->prof_events[ev_used], st));
      }
      CK(launch_relax_persistent(tl, c->tm_slow, sl.tm_tt, a, st));
      if (profile) { CK(cudaEventRecord(c->prof_events[ev_used + 1], st)); ev_used += 2; }
      CK(launch_persist_check(a, st));  // any key still pending after "done" -> kmin_bits != INF (read below)
      if (after_wave && !after_wave(sl.s0, sl.ns, st)) return 0;
      ++i;
      continue;
    }
    // a wave of source groups: G WHILE graphs side by side, joined on the context's stream
    const int wave = c->plan[i].wave;
    size_t j = i;
    while (j < c->plan.size() && c->plan[j].wave == wave) ++j;
    if (i > 0) {  // (lanes start after whatever the context's stream did before)
      CK(cudaEventRecord(c->ev_fork, c->stream));
      for (size_t k = i; k < j; ++k)
        if (c->plan[k].lane) CK(cudaStreamWaitEvent(c->aux_streams[c->plan[k].lane - 1], c->ev_fork, 0));
    }
    for (size_t k = i; k < j; ++k) {
      const auto& sl = c->plan[k];
      cudaStream_t st = lane_stream(sl.lane);
      CK(launch_reset(slice_args(c, sl), c->opts.max_rounds, st));
      CK(cudaGraphLaunch(sl.graph, st));
      if (sl.lane) CK(cudaEventRecord(c->aux_done[sl.lane - 1], st));
    }
    for (size_t k = i; k < j; ++k)
      if (c->plan[k].lane) CK(cudaStreamWaitEvent(c->stream, c->aux_done[c->plan[k].lane - 1], 0));
    if (after_wave) {
      const int s0 = c->plan[i].s0, s1 = c->plan[j - 1].s0 + c->plan[j - 1].ns;
      if (!after_wave(s0, s1 - s0, c->stream)) return 0;
    }
    i = j;
  }
  // join the lanes of independent persistent waves
  for (size_t lane = 1; lane < lane_used.size(); ++lane)
    if (lane_used[lane] && !c->plan.empty() && c->plan[0].persistent) {
      CK(cudaEventRecord(c->aux_done[lane - 1], c->aux_streams[lane - 1]));
      CK(cudaStreamWaitEvent(c->stream, c->aux_done[lane - 1], 0));
    }
  CK(cudaEventRecord(c->ev1, c->stream));
  const size_t nslots = 1 + c->plan.size();
  CK(cudaMemcpyAsync(c->h_state, c->d_state, sizeof(SolveState) * nslots, cudaMemcpyDeviceToHost, c->stream));
  // the round-based view of the state (sweeptt_step / put_tt) restarts from "nothing pending"
  CK(launch_reset_state_only(c->d_state, c->opts.max_rounds, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  if (stats) {
    std::memset(stats, 0, sizeof *stats);
    stats->struct_size = sizeof *stats;
    stats->kernel_used = c->kernel_used;
    stats->devices_used = 1;
    stats->solve_ms = ms;
    for (size_t e = 0; e < ev_used; e += 2) {
      float k = 0;
      CK(cudaEventElapsedTime(&k, c->prof_events[e], c->prof_events[e + 1]));
      stats->relax_kernel_ms += k;
    }
  }
  int pending = 0;
  for (const auto& sl : c->plan) {
    const SolveState& h = c->h_state[sl.slot];
    if (sl.persistent) {
      // done == 1 alone is not trusted: nothing may be in flight and no activation key may be left
      if (h.done != 1u || h.inflight != 0u || h.kmin_bits != 0x7f800000u)
        return fail("single-launch solve of sources %d..%d stopped without reaching the fixed point (done %u, in flight %u, "
                    "pending key %08x)", sl.s0, sl.s0 + sl.ns - 1, h.done, h.inflight, h.kmin_bits);
    } else {
      pending |= (c->kernel_used == SWEEPTT_KERNEL_TILED) ? (h.count[h.parity] != 0) : (h.last_changed_round == h.round);
    }
    if (stats) {
      const long long per_reset = (c->kernel_used == SWEEPTT_KERNEL_TILED && make_args(c).tmax) ? 5 : 4;  // state, tt, keys, (tmax,) sources
      stats->rounds = std::max(stats->rounds, h.round);
      if (sl.persistent) {
        stats->kernel_launches += per_reset + 3;  // + list 0, the solve itself, the final key scan
        stats->relax_launches += 1;
      } else {
        stats->kernel_launches += (c->kernel_used == SWEEPTT_KERNEL_TILED ? 3LL : 2LL) * h.round + per_reset;
        stats->relax_launches += h.round;
      }
      stats->tile_visits += (long long)h.tile_visits;
      stats->relaxations += (long long)h.pulls;
      stats->units_run += (long long)h.units_run;
      stats->units_changed += (long long)h.units_changed;
    }
  }
  if (pending && c->opts.max_rounds > 0) return fail("not converged after max_rounds = %d rounds", c->opts.max_rounds);
  return 1;
}

// Is the device-resident solve plan usable (else: the host-polled loop over all sources at once)?
static bool plan_usable(sweeptt_ctx* c) {
  const int loop = env_loop(c);
  if (loop == SWEEPTT_LOOP_BATCHED) return false;
  if (c->opts.profile_kernels) {  // per-launch timing: only the single-launch waves can be bracketed from outside
    const int cap = persistent_capacity(c);
    if (cap < 1) return false;
    if (const char* e = getenv("SWEEPTT_WAVE")) { const int w = atoi(e); if (w <= 0 ? cap < c->nsrc : cap < std::min(w, c->nsrc)) return false; }
    return true;
  }
  return true;
}

static int run_locked(sweeptt_ctx* c, sweeptt_stats* stats, const std::function<int(int, int, cudaStream_t)>& after_wave) {
  if (stats) { std::memset(stats, 0, sizeof *stats); }
  if (plan_usable(c)) return run_plan(c, stats, after_wave);
  CK(cudaEventRecord(c->ev0, c->stream));
  CK(launch_reset(make_args(c), c->opts.max_rounds, c->stream));
  int changed = 0;
  if (!run_rounds(c, true, 0, &changed, stats)) return 0;
  CK(cudaEventRecord(c->ev1, c->stream));
  CK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  if (stats) { stats->solve_ms = ms; stats->kernel_launches += 4; }
  if (changed && c->opts.max_rounds > 0) return fail("not converged after max_rounds = %d rounds", c->opts.max_rounds);
  if (after_wave && !after_wave(0, c->nsrc, c->stream)) return 0;
  return 1;
}

extern "C" int sweeptt_run(sweeptt_ctx* c, sweeptt_stats* stats) {
  ConstLease lease;
  if (!ready(c, &lease)) return 0;
  return run_locked(c, stats, nullptr);
}

extern "C" int sweeptt_step(sweeptt_ctx* c, int rounds, int* changed, sweeptt_stats* stats) {
  ConstLease lease;
  if (!ready(c, &lease)) return 0;
  if (rounds < 1) return fail("sweeptt_step: rounds must be >= 1");
  if (stats) std::memset(stats, 0, sizeof *stats);
  CK(cudaEventRecord(c->ev0, c->stream));
  if (!run_rounds(c, false, rounds, changed, stats)) return 0;
  CK(cudaEventRecord(c->ev1, c->stream));
  CK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  if (stats) stats->solve_ms = ms;
  return 1;
}

extern "C" int sweeptt_get_tt(sweeptt_ctx* c, int s, float* out) {
  if (!c || !out) return fail("sweeptt_get_tt: null argument");
  if (!c->have_sources || s < 0 || s >= c->nsrc) return fail("sweeptt_get_tt: source %d out of range", s);
  CK(cudaSetDevice(c->device));
  const size_t dense = (size_t)c->g.nx * c->g.ny * c->g.nz;
  if (!ensure_stage(c, dense)) return 0;
  CK(launch_unpad_box(c->d_tt + (size_t)s * c->g.vol, c->d_stage, c->g, c->stream));
  CK(cudaMemcpyAsync(out, c->d_stage, dense * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 1;
}

extern "C" int sweeptt_put_tt(sweeptt_ctx* c, int s, const float* in) {
  if (!c || !in) return fail("sweeptt_put_tt: null argument");
  ConstLease lease;
  if (!ready(c, &lease)) return 0;
  if (s < 0 || s >= c->nsrc) return fail("sweeptt_put_tt: source %d out of range", s);
  const size_t dense = (size_t)c->g.nx * c->g.ny * c->g.nz;
  // A travel time is +0, positive or +INF.  The scheduling orders times by their bits as unsigned integers, where a
  // set sign bit (-0.0, a negative time, -INF) ranks after +INF, and a NaN time would make the location's misfit NaN.
  for (size_t i = 0; i < dense; ++i) {
    uint32_t b;
    std::memcpy(&b, in + i, 4);
    if (std::isnan(in[i]) || (b >> 31))
      return fail("sweeptt_put_tt: tt[%zu] of source %d is %s (a travel time is +0, positive or +INF)", i, s,
                  std::isnan(in[i]) ? "NaN" : in[i] == 0.f ? "-0.0" : std::isinf(in[i]) ? "-INF" : "negative");
  }
  if (!ensure_stage(c, dense)) return 0;
  CK(cudaMemcpyAsync(c->d_stage, in, dense * 4, cudaMemcpyHostToDevice, c->stream));
  CK(launch_pad_box(c->d_stage, c->d_tt + (size_t)s * c->g.vol, c->g, c->stream));
  // every tile of this source must be looked at again
  // (the pending work list is replaced, so mark every source's tiles, not only this one's)
  const size_t ntiles = (size_t)c->g.ntx * c->g.nty * c->g.ntz;
  CK(cudaMemsetAsync(c->d_key, 0, ntiles * c->nsrc * 4, c->stream));  // key 0.0 = relax now
  {
    const RelaxArgs a = make_args(c);
    if (a.tmax) CK(launch_fill_tmax(a, c->stream));  // the stored bounds no longer hold
  }
  CK(launch_compact(make_args(c), 0, c->stream));  // folds the marks into the next work list
  CK(cudaStreamSynchronize(c->stream));
  return 1;
}

extern "C" int sweeptt_count_violations(sweeptt_ctx* c, int s, long long* violations) {
  ConstLease lease;
  if (!ready(c, &lease)) return 0;
  if (s < 0 || s >= c->nsrc || !violations) return fail("sweeptt_count_violations: bad argument");
  CK(cudaMemsetAsync(c->d_viol, 0, 8, c->stream));
  CK(launch_count_violations(make_args(c), s, c->d_star, c->nstar, c->d_viol, c->stream));
  unsigned long long v = 0;
  CK(cudaMemcpyAsync(&v, c->d_viol, 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  *violations = (long long)v;
  return 1;
}

// Grow-only device buffer counted in pool_bytes.
template <typename T>
static int ensure_dev(sweeptt_ctx* c, T** p, size_t* cap_bytes, size_t bytes) {
  if (*cap_bytes >= bytes) return 1;
  dev_free(c, *p, *cap_bytes);
  *p = nullptr; *cap_bytes = 0;
  if (!dev_alloc(c, (void**)p, bytes)) return 0;
  *cap_bytes = bytes;
  return 1;
}

// Pull table of the ray tracer: the context's pull star (kernel axes) with each entry's padded-box offset and its
// rank in caller-axis lexicographic order, sorted by kernel-axis (i,j,k) so that the lanes of one step read
// neighbouring z addresses.  Rebuilt when the star, the axis permutation or the padded geometry changes.
static int build_ray_pulls(sweeptt_ctx* c) {
  const BoxGeom& g = c->g;
  const int sig[6] = {c->star_gen, g.perm[0], g.perm[1], g.perm[2], g.py, g.pz};
  if (c->d_ray_pull && std::memcmp(sig, c->ray_sig, sizeof sig) == 0) return 1;
  const std::vector<PullOffset>& all = c->star.all;
  const int n = (int)all.size();
  if (n >= RAY_MAX_PULLS) return fail("sweeptt_trace_rays: %d pull offsets, the tracer holds fewer than %d", n, RAY_MAX_PULLS);
  std::vector<std::array<int, 3>> caller(n);
  for (int l = 0; l < n; ++l) {
    const int k[3] = {all[l].i, all[l].j, all[l].k};
    for (int q = 0; q < 3; ++q) caller[l][g.perm[q]] = k[q];
  }
  std::vector<int> by_caller(n);
  for (int l = 0; l < n; ++l) by_caller[l] = l;
  std::sort(by_caller.begin(), by_caller.end(), [&](int a, int b) { return caller[a] < caller[b]; });
  std::vector<int> rank(n);
  for (int p = 0, r = 0; p < n; ++p) {  // equal offsets (same m) share a rank
    if (p > 0 && caller[by_caller[p]] != caller[by_caller[p - 1]]) ++r;
    rank[by_caller[p]] = r;
  }
  std::vector<int> by_kernel(n);
  for (int l = 0; l < n; ++l) by_kernel[l] = l;
  std::stable_sort(by_kernel.begin(), by_kernel.end(), [&](int a, int b) {
    return std::tie(all[a].i, all[a].j, all[a].k) < std::tie(all[b].i, all[b].j, all[b].k);
  });
  c->ray_pull.resize(n);
  for (int p = 0; p < n; ++p) {
    const PullOffset& o = all[by_kernel[p]];
    if (std::abs(o.i) > 32767 || std::abs(o.j) > 32767 || std::abs(o.k) > 32767)
      return fail("sweeptt_trace_rays: star offset (%d,%d,%d) is wider than the tracer's 16-bit offsets", o.i, o.j, o.k);
    const long long off = (long long)o.i * g.sx + (long long)o.j * g.pz + o.k;
    if (off > INT32_MAX || off < INT32_MIN) return fail("sweeptt_trace_rays: star offset (%d,%d,%d) too wide for this box", o.i, o.j, o.k);
    c->ray_pull[p] = RayPull{(short)o.i, (short)o.j, (short)o.k,
                             (unsigned short)(rank[by_kernel[p]] | (o.guarded ? RAY_GUARD_BIT : 0u)), (int)off, o.hd};
  }
  if (!ensure_dev(c, &c->d_ray_pull, &c->ray_pull_cap, (size_t)n * sizeof(RayPull))) return 0;
  CK(cudaMemcpyAsync(c->d_ray_pull, c->ray_pull.data(), (size_t)n * sizeof(RayPull), cudaMemcpyHostToDevice, c->stream));
  std::memcpy(c->ray_sig, sig, sizeof sig);
  return 1;
}

// The source range of a call that reads the context's fields (ray, tomography and location calls).
static int check_source_range(const sweeptt_ctx* c, const char* who, int source_begin, int source_count) {
  if (source_count < 1 || source_begin < 0 || source_begin > c->nsrc - source_count)
    return fail("%s: sources [%d, %d) are not within the context's %d sources", who, source_begin,
                source_begin + source_count, c->nsrc);
  return 1;
}

// Argument checks shared by the ray calls (sweeptt_trace_rays, sweeptt_ray_project, sweeptt_ray_backproject), then
// the receivers range-checked and permuted to kernel axes into c->rec_xyz.
static int check_ray_call(sweeptt_ctx* c, ConstLease* lease, const char* who, int source_begin, int source_count,
                          const struct START* receivers, int nrec, int max_nodes, sweeptt_stats* stats) {
  if (!ready(c, lease)) return 0;
  if (stats) std::memset(stats, 0, sizeof *stats);
  if (!receivers || nrec < 1) return fail("%s: need at least one receiver", who);
  if (!check_source_range(c, who, source_begin, source_count)) return 0;
  if (max_nodes < 1) return fail("%s: max_nodes must be >= 1 (got %d)", who, max_nodes);
  const BoxGeom& g = c->g;
  int on[3];  // caller-order dims
  on[g.perm[0]] = g.nx; on[g.perm[1]] = g.ny; on[g.perm[2]] = g.nz;
  c->rec_xyz.resize(3 * (size_t)nrec);
  for (int r = 0; r < nrec; ++r) {
    const int o[3] = {receivers[r].i, receivers[r].j, receivers[r].k};
    if (o[0] < 0 || o[0] >= on[0] || o[1] < 0 || o[1] >= on[1] || o[2] < 0 || o[2] >= on[2])
      return fail("receiver %d (%d,%d,%d) is outside the %d x %d x %d model", r, o[0], o[1], o[2], on[0], on[1], on[2]);
    for (int q = 0; q < 3; ++q) c->rec_xyz[3 * (size_t)r + q] = o[g.perm[q]];
  }
  return 1;
}

// Pull table and the checked receivers on the device.
static int upload_ray_tables(sweeptt_ctx* c, int nrec) {
  if (!build_ray_pulls(c)) return 0;
  if (!ensure_dev(c, &c->d_rec, &c->rec_cap, 3 * sizeof(int) * (size_t)nrec)) return 0;
  CK(cudaMemcpyAsync(c->d_rec, c->rec_xyz.data(), 3 * sizeof(int) * (size_t)nrec, cudaMemcpyHostToDevice, c->stream));
  return 1;
}

static TraceArgs ray_trace_args(sweeptt_ctx* c, int source_begin, int nrec, long long nrays, int max_nodes) {
  TraceArgs t{};
  t.g = c->g;
  t.slow = c->d_slow;
  t.tt = c->d_tt;
  t.src_xyz = c->d_src;
  t.rec_xyz = c->d_rec;
  t.pull = c->d_ray_pull;
  t.npull = (int)c->ray_pull.size();
  t.source_begin = source_begin;
  t.nrec = nrec;
  t.nrays = nrays;
  t.max_nodes = max_nodes;
  return t;
}

extern "C" int sweeptt_trace_rays(sweeptt_ctx* c, int source_begin, int source_count, const struct START* receivers,
                                  int nrec, int max_nodes, struct START* nodes_out, int32_t* length_out,
                                  int32_t* status_out, float* tt_out, sweeptt_stats* stats) {
  ConstLease lease;
  if (!check_ray_call(c, &lease, "sweeptt_trace_rays", source_begin, source_count, receivers, nrec, max_nodes, stats))
    return 0;
  const long long nrays = (long long)source_count * nrec;
  if (nodes_out && (unsigned long long)nrays > (1ull << 60) / (12ull * (unsigned long long)max_nodes))
    return fail("sweeptt_trace_rays: %lld rays of up to %d nodes do not fit one call", nrays, max_nodes);
  if (!upload_ray_tables(c, nrec)) return 0;
  // output buffer: [evaluation counter | length | status | tt | nodes], every part 16-byte aligned
  auto up16 = [](size_t b) { return (b + 15) / 16 * 16; };
  const size_t per_ray = up16(4 * (size_t)nrays);
  const size_t node_bytes = nodes_out ? (size_t)nrays * max_nodes * sizeof(START) : 0;
  if (!ensure_dev(c, &c->d_ray_out, &c->ray_out_cap, 16 + 3 * per_ray + node_bytes)) return 0;
  TraceArgs t = ray_trace_args(c, source_begin, nrec, nrays, max_nodes);
  t.evals = reinterpret_cast<unsigned long long*>(c->d_ray_out);
  t.length = reinterpret_cast<int*>(c->d_ray_out + 16);
  t.status = reinterpret_cast<int*>(c->d_ray_out + 16 + per_ray);
  t.tt_rec = reinterpret_cast<float*>(c->d_ray_out + 16 + 2 * per_ray);
  t.nodes = nodes_out ? reinterpret_cast<int*>(c->d_ray_out + 16 + 3 * per_ray) : nullptr;
  CK(cudaMemsetAsync(t.evals, 0, 8, c->stream));
  if (t.nodes) CK(cudaMemsetAsync(t.nodes, 0xff, node_bytes, c->stream));  // (-1,-1,-1) past every ray's length
  CK(cudaEventRecord(c->ev0, c->stream));
  CK(launch_trace_rays(t, c->device, c->stream));
  CK(cudaEventRecord(c->ev1, c->stream));
  CK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));

  const auto t_copy = std::chrono::steady_clock::now();
  std::vector<int32_t> len_tmp;
  int32_t* len_host = length_out;
  if (!len_host && nodes_out) { len_tmp.resize(nrays); len_host = len_tmp.data(); }
  unsigned long long evals = 0;
  long long bytes = 8;
  CK(cudaMemcpyAsync(&evals, t.evals, 8, cudaMemcpyDeviceToHost, c->stream));
  if (len_host) { CK(cudaMemcpyAsync(len_host, t.length, 4 * nrays, cudaMemcpyDeviceToHost, c->stream)); bytes += 4 * nrays; }
  if (status_out) { CK(cudaMemcpyAsync(status_out, t.status, 4 * nrays, cudaMemcpyDeviceToHost, c->stream)); bytes += 4 * nrays; }
  if (tt_out) { CK(cudaMemcpyAsync(tt_out, t.tt_rec, 4 * nrays, cudaMemcpyDeviceToHost, c->stream)); bytes += 4 * nrays; }
  CK(cudaStreamSynchronize(c->stream));
  if (nodes_out) {
    // only the first max(length) nodes of every ray's slot travel; the rest of nodes_out is left untouched
    const int lmax = *std::max_element(len_host, len_host + nrays);
    const size_t pitch = (size_t)max_nodes * sizeof(START), width = (size_t)lmax * sizeof(START);
    if (lmax == max_nodes)
      CK(cudaMemcpyAsync(nodes_out, t.nodes, node_bytes, cudaMemcpyDeviceToHost, c->stream));
    else
      CK(cudaMemcpy2DAsync(nodes_out, pitch, t.nodes, pitch, width, (size_t)nrays, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    bytes += (long long)(width * nrays);
  }
  if (stats) {
    stats->struct_size = (int)sizeof *stats;
    stats->solve_ms = ms;
    stats->relaxations = (long long)evals;
    stats->kernel_launches = 1;
    stats->devices_used = 1;
    stats->d2h_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_copy).count();
    stats->d2h_bytes = bytes;
  }
  return 1;
}

// Smallest E with 2*hd_max*W*N <= 2^(E+62), in exact arithmetic (hd_max, W > 0 finite).  With hd_max = Mh*2^(eh-24)
// and W = Mw*2^(ew-24) (Mh, Mw the 24-bit integer significands), the condition is X = Mh*Mw*N <= 2^(E+109-eh-ew).
static int quantum_exponent(float hd_max, float W, long long N) {
  int eh = 0, ew = 0;
  const unsigned long long Mh = (unsigned long long)std::ldexp(std::frexp((double)hd_max, &eh), 24);
  const unsigned long long Mw = (unsigned long long)std::ldexp(std::frexp((double)W, &ew), 24);
  const unsigned __int128 X = (unsigned __int128)(Mh * Mw) * (unsigned long long)N;
  int b = 0;  // bit length: 2^(b-1) <= X < 2^b
  while ((X >> b) != 0) ++b;
  const int k = (X & (X - 1)) == 0 ? b - 1 : b;  // smallest k with X <= 2^k
  return k - 109 + eh + ew;
}

// Shared part of sweeptt_ray_project / sweeptt_ray_backproject after the inputs are on the device: the walk kernel
// (and, for the back-projection, the rounding kernel into c->d_stage), timed with events; then the evaluation
// counter, statuses and lengths copied back.
static int run_ray_walk(sweeptt_ctx* c, bool back, TomoArgs& a, int E, int kernels_before,
                        int32_t* status_out, int32_t* length_out, float* proj_out, sweeptt_stats* stats) {
  const long long nrays = a.t.nrays;
  RayWalkLaunch l{};
  CK(ray_walk_prepare(back, a.t.npull, a.t.max_nodes, nrays, c->device, &l));
  if (!l.path_in_smem) {
    if (!ensure_dev(c, &c->d_path, &c->path_cap, (size_t)l.path_entries * sizeof(unsigned short))) return 0;
    a.path_global = c->d_path;
    a.path_entries = l.path_entries;
  }
  CK(launch_ray_walk(back, l, a, c->stream));
  if (back) CK(launch_grad_finish(a.acc, c->d_stage, c->g, E, c->stream));
  CK(cudaEventRecord(c->ev1, c->stream));
  CK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));

  const auto t_copy = std::chrono::steady_clock::now();
  unsigned long long evals = 0;
  long long bytes = 8;
  CK(cudaMemcpyAsync(&evals, a.t.evals, 8, cudaMemcpyDeviceToHost, c->stream));
  if (length_out) { CK(cudaMemcpyAsync(length_out, a.t.length, 4 * nrays, cudaMemcpyDeviceToHost, c->stream)); bytes += 4 * nrays; }
  if (status_out) { CK(cudaMemcpyAsync(status_out, a.t.status, 4 * nrays, cudaMemcpyDeviceToHost, c->stream)); bytes += 4 * nrays; }
  if (proj_out) { CK(cudaMemcpyAsync(proj_out, a.proj, 4 * nrays, cudaMemcpyDeviceToHost, c->stream)); bytes += 4 * nrays; }
  CK(cudaStreamSynchronize(c->stream));
  if (stats) {
    stats->struct_size = (int)sizeof *stats;
    stats->solve_ms = ms;
    stats->relaxations = (long long)evals;
    stats->kernel_launches = kernels_before + 1 + (back ? 1 : 0);
    stats->devices_used = 1;
    stats->d2h_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_copy).count();
    stats->d2h_bytes += bytes;
  }
  return 1;
}

// Output buffer of the tomography calls: [evaluation counter | length | status | projection or weights], every part
// 16-byte aligned.
static int tomo_args(sweeptt_ctx* c, int source_begin, int nrec, long long nrays, int max_nodes, TomoArgs* a,
                     size_t* per_ray) {
  *per_ray = ((size_t)4 * nrays + 15) / 16 * 16;
  if (!ensure_dev(c, &c->d_ray_out, &c->ray_out_cap, 16 + 3 * *per_ray)) return 0;
  *a = TomoArgs{};
  a->t = ray_trace_args(c, source_begin, nrec, nrays, max_nodes);
  a->t.evals = reinterpret_cast<unsigned long long*>(c->d_ray_out);
  a->t.length = reinterpret_cast<int*>(c->d_ray_out + 16);
  a->t.status = reinterpret_cast<int*>(c->d_ray_out + 16 + *per_ray);
  CK(cudaMemsetAsync(a->t.evals, 0, 8, c->stream));
  return 1;
}

extern "C" int sweeptt_ray_project(sweeptt_ctx* c, int source_begin, int source_count, const struct START* receivers,
                                   int nrec, int max_nodes, const float* perturbation, float* proj_out,
                                   int32_t* status_out, int32_t* length_out, sweeptt_stats* stats) {
  ConstLease lease;
  if (!check_ray_call(c, &lease, "sweeptt_ray_project", source_begin, source_count, receivers, nrec, max_nodes, stats))
    return 0;
  if (!perturbation) return fail("sweeptt_ray_project: null perturbation");
  const long long nrays = (long long)source_count * nrec;
  if (!upload_ray_tables(c, nrec)) return 0;
  const BoxGeom& g = c->g;
  const size_t dense = (size_t)g.nx * g.ny * g.nz;
  if (!ensure_stage(c, dense)) return 0;
  if (!ensure_dev(c, &c->d_pert, &c->pert_cap, (size_t)g.vol * 4)) return 0;
  TomoArgs a;
  size_t per_ray;
  if (!tomo_args(c, source_begin, nrec, nrays, max_nodes, &a, &per_ray)) return 0;
  a.pert = c->d_pert;
  a.proj = reinterpret_cast<float*>(c->d_ray_out + 16 + 2 * per_ray);
  // only nodes on a ray are read, and those are in the box: the apron of d_pert is never looked at
  CK(cudaMemcpyAsync(c->d_stage, perturbation, dense * 4, cudaMemcpyHostToDevice, c->stream));
  CK(cudaEventRecord(c->ev0, c->stream));
  CK(launch_pad_box(c->d_stage, c->d_pert, g, c->stream));
  return run_ray_walk(c, false, a, 0, 1, status_out, length_out, proj_out, stats);
}

extern "C" int sweeptt_ray_backproject(sweeptt_ctx* c, int source_begin, int source_count,
                                       const struct START* receivers, int nrec, int max_nodes, const float* weights,
                                       float* grad_out, int* quantum_exp_out, int32_t* status_out,
                                       sweeptt_stats* stats) {
  ConstLease lease;
  if (!check_ray_call(c, &lease, "sweeptt_ray_backproject", source_begin, source_count, receivers, nrec, max_nodes,
                      stats))
    return 0;
  if (!weights || !grad_out) return fail("sweeptt_ray_backproject: weights and grad_out are required");
  const long long nrays = (long long)source_count * nrec;
  float W = 0.f;
  for (long long q = 0; q < nrays; ++q) {
    if (!std::isfinite(weights[q])) return fail("sweeptt_ray_backproject: weight %lld is not finite", q);
    W = std::max(W, std::fabs(weights[q]));
  }
  if (!upload_ray_tables(c, nrec)) return 0;
  float hd_max = 0.f;
  for (const RayPull& p : c->ray_pull) hd_max = std::max(hd_max, p.hd);
  if (!std::isfinite(hd_max)) return fail("sweeptt_ray_backproject: the star's edge lengths are not finite");
  const int E = (W > 0.f && hd_max > 0.f) ? quantum_exponent(hd_max, W, nrays) : 0;
  const BoxGeom& g = c->g;
  const size_t dense = (size_t)g.nx * g.ny * g.nz;
  if (!ensure_stage(c, dense)) return 0;
  if (!ensure_dev(c, &c->d_acc, &c->acc_cap, (size_t)g.vol * 8)) return 0;
  TomoArgs a;
  size_t per_ray;
  if (!tomo_args(c, source_begin, nrec, nrays, max_nodes, &a, &per_ray)) return 0;
  float* d_w = reinterpret_cast<float*>(c->d_ray_out + 16 + 2 * per_ray);
  a.weights = d_w;
  a.acc = c->d_acc;
  a.scale = std::ldexp(1.0, -E);
  CK(cudaMemcpyAsync(d_w, weights, 4 * nrays, cudaMemcpyHostToDevice, c->stream));
  CK(cudaEventRecord(c->ev0, c->stream));
  CK(cudaMemsetAsync(c->d_acc, 0, (size_t)g.vol * 8, c->stream));
  if (!run_ray_walk(c, true, a, E, 0, status_out, nullptr, nullptr, stats)) return 0;
  const auto t_copy = std::chrono::steady_clock::now();
  CK(cudaMemcpyAsync(grad_out, c->d_stage, dense * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (stats) {
    stats->d2h_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_copy).count();
    stats->d2h_bytes += (long long)(dense * 4);
  }
  if (quantum_exp_out) *quantum_exp_out = E;
  return 1;
}

// ---------------------------------------------------------------------------------------
// ray sets (include/sweeptt.h, sweeptt_rayset_*)
// ---------------------------------------------------------------------------------------
// A snapshot of traced rays: the records of the OK rays as pull-table entries, ray-major in q order (CSR), with the
// pull table, geometry and start indices they are decoded with, and the buffers the two operators need.  Only the
// context's device and stream are borrowed.
struct sweeptt_rayset {
  sweeptt_ctx* ctx = nullptr;
  int device = 0;
  BoxGeom g{};
  int source_count = 0, nrec = 0;
  long long nrays = 0, nentries = 0;
  float hd_max = 0.f;
  std::vector<RayPull> pull;          // the pull table at the freeze
  std::vector<int> rec;               // receivers, caller axes
  std::vector<int64_t> offsets;       // [nrays + 1] over the entries
  std::vector<int32_t> length, status;
  std::vector<float> tt;
  RayPull* d_pull = nullptr;
  long long* d_offsets = nullptr;
  unsigned short* d_entries = nullptr;
  int* d_status = nullptr;
  long long* d_start = nullptr;
  float* d_pert = nullptr;            // padded perturbation box
  long long* d_acc = nullptr;         // padded int64 accumulator box
  float* d_stage = nullptr;           // dense staging box
  float* d_io = nullptr;              // [nrays] projections or weights
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  size_t bytes = 0;
};

static void rayset_free(sweeptt_rayset* r) {
  void* bufs[] = {r->d_pull, r->d_offsets, r->d_entries, r->d_status, r->d_start, r->d_pert, r->d_acc, r->d_stage, r->d_io};
  for (void* b : bufs) cudaFree(b);
  if (r->ev0) cudaEventDestroy(r->ev0);
  if (r->ev1) cudaEventDestroy(r->ev1);
  delete r;
}

static int rayset_alloc(sweeptt_rayset* r, void** p, size_t bytes) {
  if (bytes == 0) return 1;
  CK(cudaMalloc(p, bytes));
  r->bytes += bytes;
  return 1;
}

// Staging of one freeze chunk: at most this many bytes of padded records (the chunk is at least one ray).
static constexpr size_t RAYSET_STAGING_BYTES = size_t(256) << 20;

static int rayset_freeze(sweeptt_ctx* c, int source_begin, int source_count, const struct START* receivers, int nrec,
                         int max_nodes, sweeptt_stats* stats, sweeptt_rayset* r) {
  ConstLease lease;
  if (!check_ray_call(c, &lease, "sweeptt_rayset_freeze", source_begin, source_count, receivers, nrec, max_nodes, stats))
    return 0;
  if (!upload_ray_tables(c, nrec)) return 0;
  const long long nrays = (long long)source_count * nrec;
  const long long chunk = std::max(1LL, std::min<long long>(nrays, (long long)(RAYSET_STAGING_BYTES / (2 * (size_t)max_nodes))));
  if (!ensure_dev(c, &c->d_path, &c->path_cap, (size_t)chunk * max_nodes * sizeof(unsigned short))) return 0;
  // [evaluation counter | length | status | tt | chunk offsets], every part 16-byte aligned
  const size_t per_ray = ((size_t)4 * chunk + 15) / 16 * 16;
  if (!ensure_dev(c, &c->d_ray_out, &c->ray_out_cap, 16 + 3 * per_ray + 8 * (size_t)(chunk + 1))) return 0;
  r->ctx = c;
  r->device = c->device;
  r->g = c->g;
  r->source_count = source_count;
  r->nrec = nrec;
  r->nrays = nrays;
  r->pull = c->ray_pull;
  for (const RayPull& p : r->pull) r->hd_max = std::max(r->hd_max, p.hd);
  r->rec.resize(3 * (size_t)nrec);
  for (int q = 0; q < nrec; ++q) { r->rec[3 * q] = receivers[q].i; r->rec[3 * q + 1] = receivers[q].j; r->rec[3 * q + 2] = receivers[q].k; }
  r->length.resize(nrays); r->status.resize(nrays); r->tt.resize(nrays); r->offsets.assign(nrays + 1, 0);
  CK(cudaEventCreate(&r->ev0));
  CK(cudaEventCreate(&r->ev1));

  TomoArgs a{};
  a.t = ray_trace_args(c, source_begin, nrec, 0, max_nodes);
  a.t.evals = reinterpret_cast<unsigned long long*>(c->d_ray_out);
  a.t.length = reinterpret_cast<int*>(c->d_ray_out + 16);
  a.t.status = reinterpret_cast<int*>(c->d_ray_out + 16 + per_ray);
  a.t.tt_rec = reinterpret_cast<float*>(c->d_ray_out + 16 + 2 * per_ray);
  long long* d_off = reinterpret_cast<long long*>(c->d_ray_out + 16 + 3 * per_ray);
  a.path_global = c->d_path;
  CK(cudaMemsetAsync(a.t.evals, 0, 8, c->stream));
  // each chunk's OK records are packed into a piece of their own; the pieces are joined once the total is known
  struct Pieces {
    std::vector<std::pair<unsigned short*, long long>> v;
    ~Pieces() { for (auto& p : v) cudaFree(p.first); }
  } pieces;
  std::vector<int64_t> rel(chunk + 1);
  double ms_total = 0, d2h_ms = 0;
  long long launches = 0, d2h_bytes = 8;
  for (long long q0 = 0; q0 < nrays; q0 += chunk) {
    const long long nc = std::min(chunk, nrays - q0);
    a.t.nrays = nc;
    a.q_begin = q0;
    a.path_entries = nc * max_nodes;
    CK(cudaEventRecord(r->ev0, c->stream));
    CK(launch_rayset_record(a, c->device, c->stream));
    CK(cudaEventRecord(r->ev1, c->stream));
    const auto t_copy = std::chrono::steady_clock::now();
    CK(cudaMemcpyAsync(r->length.data() + q0, a.t.length, 4 * nc, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(r->status.data() + q0, a.t.status, 4 * nc, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(r->tt.data() + q0, a.t.tt_rec, 4 * nc, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    d2h_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_copy).count();
    d2h_bytes += 12 * nc;
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, r->ev0, r->ev1));
    ms_total += ms;
    ++launches;
    rel[0] = 0;
    for (long long q = 0; q < nc; ++q)
      rel[q + 1] = rel[q] + (r->status[q0 + q] == SWEEPTT_RAY_OK ? r->length[q0 + q] - 1 : 0);
    for (long long q = 0; q < nc; ++q) r->offsets[q0 + q + 1] = r->offsets[q0] + rel[q + 1];
    if (rel[nc] == 0) continue;
    unsigned short* piece = nullptr;
    CK(cudaMalloc(&piece, (size_t)rel[nc] * sizeof(unsigned short)));
    pieces.v.emplace_back(piece, rel[nc]);
    CK(cudaMemcpyAsync(d_off, rel.data(), 8 * (size_t)(nc + 1), cudaMemcpyHostToDevice, c->stream));
    CK(cudaEventRecord(r->ev0, c->stream));
    CK(launch_rayset_compact(c->d_path, max_nodes, d_off, nc, piece, c->stream));
    CK(cudaEventRecord(r->ev1, c->stream));
    CK(cudaEventSynchronize(r->ev1));  // before d_off and the staging slots are reused
    CK(cudaEventElapsedTime(&ms, r->ev0, r->ev1));
    ms_total += ms;
    ++launches;
  }
  r->nentries = r->offsets[nrays];
  unsigned long long evals = 0;
  CK(cudaMemcpyAsync(&evals, a.t.evals, 8, cudaMemcpyDeviceToHost, c->stream));

  const BoxGeom& g = r->g;
  const size_t dense = (size_t)g.nx * g.ny * g.nz;
  if (!rayset_alloc(r, (void**)&r->d_entries, (size_t)r->nentries * sizeof(unsigned short)) ||
      !rayset_alloc(r, (void**)&r->d_offsets, 8 * (size_t)(nrays + 1)) ||
      !rayset_alloc(r, (void**)&r->d_status, 4 * (size_t)nrays) ||
      !rayset_alloc(r, (void**)&r->d_io, 4 * (size_t)nrays) ||
      !rayset_alloc(r, (void**)&r->d_pull, r->pull.size() * sizeof(RayPull)) ||
      !rayset_alloc(r, (void**)&r->d_start, 8 * (size_t)source_count) ||
      !rayset_alloc(r, (void**)&r->d_pert, 4 * (size_t)g.vol) ||
      !rayset_alloc(r, (void**)&r->d_acc, 8 * (size_t)g.vol) ||
      !rayset_alloc(r, (void**)&r->d_stage, 4 * dense))
    return 0;
  long long at = 0;
  for (auto& p : pieces.v) {
    CK(cudaMemcpyAsync(r->d_entries + at, p.first, (size_t)p.second * sizeof(unsigned short), cudaMemcpyDeviceToDevice, c->stream));
    at += p.second;
  }
  std::vector<long long> start(source_count);
  for (int s = 0; s < source_count; ++s) {
    const int* p = &c->src_xyz[3 * (size_t)(source_begin + s)];
    start[s] = ((long long)(p[0] + AX) * g.py + (p[1] + AY)) * g.pz + (p[2] + AZ);
  }
  CK(cudaMemcpyAsync(r->d_offsets, r->offsets.data(), 8 * (size_t)(nrays + 1), cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(r->d_status, r->status.data(), 4 * (size_t)nrays, cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(r->d_pull, r->pull.data(), r->pull.size() * sizeof(RayPull), cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(r->d_start, start.data(), 8 * (size_t)source_count, cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));  // the pieces and the host vectors above are released after this
  if (stats) {
    stats->struct_size = (int)sizeof *stats;
    stats->solve_ms = ms_total;
    stats->relaxations = (long long)evals;
    stats->kernel_launches = launches;
    stats->devices_used = 1;
    stats->d2h_ms = d2h_ms;
    stats->d2h_bytes = d2h_bytes;
  }
  return 1;
}

extern "C" sweeptt_rayset* sweeptt_rayset_freeze(sweeptt_ctx* c, int source_begin, int source_count,
                                                 const struct START* receivers, int nrec, int max_nodes,
                                                 sweeptt_stats* stats) {
  auto* r = new sweeptt_rayset();
  if (!rayset_freeze(c, source_begin, source_count, receivers, nrec, max_nodes, stats, r)) {
    if (c) cudaSetDevice(c->device);
    rayset_free(r);
    return nullptr;
  }
  return r;
}

extern "C" void sweeptt_rayset_destroy(sweeptt_rayset* r) {
  if (!r) return;
  cudaSetDevice(r->device);
  cudaStreamSynchronize(r->ctx->stream);
  rayset_free(r);
}

extern "C" size_t sweeptt_rayset_bytes(const sweeptt_rayset* r) { return r ? r->bytes : 0; }

extern "C" int sweeptt_rayset_table(const sweeptt_rayset* r, int32_t* length_out, int32_t* status_out, float* tt_out) {
  if (!r) return fail("null ray set");
  const size_t n = (size_t)r->nrays;
  if (length_out) std::memcpy(length_out, r->length.data(), 4 * n);
  if (status_out) std::memcpy(status_out, r->status.data(), 4 * n);
  if (tt_out) std::memcpy(tt_out, r->tt.data(), 4 * n);
  return 1;
}

extern "C" int sweeptt_rayset_paths(const sweeptt_rayset* r, int64_t* offsets_out, struct START* nodes_out) {
  if (!r) return fail("null ray set");
  if (offsets_out) {
    offsets_out[0] = 0;
    for (long long q = 0; q < r->nrays; ++q)
      offsets_out[q + 1] = offsets_out[q] + (r->status[q] == SWEEPTT_RAY_OK ? r->length[q] : 0);
  }
  if (!nodes_out) return 1;
  std::vector<unsigned short> e((size_t)r->nentries);
  CK(cudaSetDevice(r->device));
  if (r->nentries) {
    CK(cudaMemcpyAsync(e.data(), r->d_entries, e.size() * sizeof(unsigned short), cudaMemcpyDeviceToHost, r->ctx->stream));
    CK(cudaStreamSynchronize(r->ctx->stream));
  }
  const int* perm = r->g.perm;
  START* out = nodes_out;
  for (long long q = 0; q < r->nrays; ++q) {
    if (r->status[q] != SWEEPTT_RAY_OK) continue;
    int p[3];  // caller axes
    std::memcpy(p, &r->rec[3 * (size_t)(q % r->nrec)], sizeof p);
    *out++ = START{p[0], p[1], p[2]};
    for (int64_t k = r->offsets[q]; k < r->offsets[q + 1]; ++k) {
      const RayPull& o = r->pull[e[(size_t)k]];
      p[perm[0]] += o.i; p[perm[1]] += o.j; p[perm[2]] += o.k;  // kernel axis q is caller axis perm[q]
      *out++ = START{p[0], p[1], p[2]};
    }
  }
  return 1;
}

// Shared part of the two operators once the inputs are on the device: the walk (and the rounding into d_stage),
// timed with events, the stream synchronised.
static int rayset_walk(sweeptt_rayset* r, bool back, RaySetArgs& s, int E, sweeptt_stats* stats) {
  cudaStream_t st = r->ctx->stream;
  CK(launch_rayset_walk(back, s, r->device, st));
  if (back) CK(launch_grad_finish(r->d_acc, r->d_stage, r->g, E, st));
  CK(cudaEventRecord(r->ev1, st));
  CK(cudaEventSynchronize(r->ev1));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, r->ev0, r->ev1));
  if (stats) {
    stats->struct_size = (int)sizeof *stats;
    stats->solve_ms = ms;
    stats->kernel_launches = 2;
    stats->devices_used = 1;
  }
  return 1;
}

static RaySetArgs rayset_args(const sweeptt_rayset* r) {
  RaySetArgs s{};
  s.a.t.g = r->g;
  s.a.t.pull = r->d_pull;
  s.a.t.npull = (int)r->pull.size();
  s.a.t.nrec = r->nrec;
  s.a.t.nrays = r->nrays;
  s.a.t.status = r->d_status;
  s.offsets = r->d_offsets;
  s.entries = r->d_entries;
  s.entries_n = r->nentries;
  s.start_idx = r->d_start;
  return s;
}

extern "C" int sweeptt_rayset_project(sweeptt_rayset* r, const float* perturbation, float* proj_out,
                                      sweeptt_stats* stats) {
  if (!r) return fail("null ray set");
  if (stats) std::memset(stats, 0, sizeof *stats);
  if (!perturbation) return fail("sweeptt_rayset_project: null perturbation");
  CK(cudaSetDevice(r->device));
  cudaStream_t st = r->ctx->stream;
  const size_t dense = (size_t)r->g.nx * r->g.ny * r->g.nz;
  RaySetArgs s = rayset_args(r);
  s.a.pert = r->d_pert;
  s.a.proj = r->d_io;
  // only nodes on a ray are read, and those are in the box: the apron of d_pert is never looked at
  CK(cudaMemcpyAsync(r->d_stage, perturbation, dense * 4, cudaMemcpyHostToDevice, st));
  CK(cudaEventRecord(r->ev0, st));
  CK(launch_pad_box(r->d_stage, r->d_pert, r->g, st));
  if (!rayset_walk(r, false, s, 0, stats)) return 0;
  const auto t_copy = std::chrono::steady_clock::now();
  if (proj_out) {
    CK(cudaMemcpyAsync(proj_out, r->d_io, 4 * (size_t)r->nrays, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  if (stats) {
    stats->d2h_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_copy).count();
    stats->d2h_bytes = proj_out ? 4 * r->nrays : 0;
  }
  return 1;
}

extern "C" int sweeptt_rayset_backproject(sweeptt_rayset* r, const float* weights, float* grad_out,
                                          int* quantum_exp_out, sweeptt_stats* stats) {
  if (!r) return fail("null ray set");
  if (stats) std::memset(stats, 0, sizeof *stats);
  if (!weights || !grad_out) return fail("sweeptt_rayset_backproject: weights and grad_out are required");
  float W = 0.f;
  for (long long q = 0; q < r->nrays; ++q) {
    if (!std::isfinite(weights[q])) return fail("sweeptt_rayset_backproject: weight %lld is not finite", q);
    W = std::max(W, std::fabs(weights[q]));
  }
  if (!std::isfinite(r->hd_max)) return fail("sweeptt_rayset_backproject: the star's edge lengths are not finite");
  const int E = (W > 0.f && r->hd_max > 0.f) ? quantum_exponent(r->hd_max, W, r->nrays) : 0;
  CK(cudaSetDevice(r->device));
  cudaStream_t st = r->ctx->stream;
  const BoxGeom& g = r->g;
  const size_t dense = (size_t)g.nx * g.ny * g.nz;
  RaySetArgs s = rayset_args(r);
  s.a.weights = r->d_io;
  s.a.acc = r->d_acc;
  s.a.scale = std::ldexp(1.0, -E);
  CK(cudaMemcpyAsync(r->d_io, weights, 4 * (size_t)r->nrays, cudaMemcpyHostToDevice, st));
  CK(cudaEventRecord(r->ev0, st));
  CK(cudaMemsetAsync(r->d_acc, 0, (size_t)g.vol * 8, st));
  if (!rayset_walk(r, true, s, E, stats)) return 0;
  const auto t_copy = std::chrono::steady_clock::now();
  CK(cudaMemcpyAsync(grad_out, r->d_stage, dense * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (stats) {
    stats->d2h_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_copy).count();
    stats->d2h_bytes = (long long)(dense * 4);
  }
  if (quantum_exp_out) *quantum_exp_out = E;
  return 1;
}

// ---------------------------------------------------------------------------------------
// LSQR over a ray set (include/sweeptt.h, sweeptt_rayset_lsqr; DESIGN §3.11)
// ---------------------------------------------------------------------------------------
// The vectors stay on the device; the host runs scipy's scalar recurrences (this file is built with
// -ffp-contract=off, so they round exactly as numpy's scalars do) and reads four scalars per iteration.

// CTAs that share the blocks of a first-level reduction (SWEEPTT_LSQR_CTAS; the result does not depend on it).
static int lsqr_ctas() {
  int ctas = 1184;
  if (const char* e = getenv("SWEEPTT_LSQR_CTAS")) ctas = std::max(1, atoi(e));
  return ctas;
}

namespace {

struct LsqrSolve {
  sweeptt_rayset* r = nullptr;
  cudaStream_t st = nullptr;
  LsqrArgs a{};
  void* dev = nullptr;      // the whole float64 workspace, one allocation
  double* host = nullptr;   // page-locked: [0] a sum of squares, [1] the bits of max |W|
  long long D = 0;
  int launches = 0;
  double d2h_ms = 0;
  long long d2h_bytes = 0;

  ~LsqrSolve() {
    if (dev) cudaFree(dev);
    if (host) cudaFreeHost(host);
  }

  // sqrt of the sum of squares the last pass left in part[0]
  int read_norm(double* out) {
    const auto t0 = std::chrono::steady_clock::now();
    CK(cudaMemcpyAsync(host, a.part, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    d2h_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    d2h_bytes += 8;
    *out = std::sqrt(host[0]);
    return 1;
  }

  // G x: pass A (v to float32, padded into the set's box) and pass B (the set's projection into io)
  int project() {
    CK(launch_lsqr_to_f32(a.v, r->d_stage, D, st));
    CK(launch_pad_box(r->d_stage, r->d_pert, r->g, st));
    RaySetArgs s = rayset_args(r);
    s.a.pert = r->d_pert;
    s.a.proj = r->d_io;
    CK(launch_rayset_walk(false, s, r->device, st));
    launches += 3;
    return 1;
  }

  // Pass D (u = inv_beta u; W into io; max |W|) and pass E (the set's back-projection of W into stage with the E
  // that sweeptt_rayset_backproject chooses)
  int backproject(double inv_beta) {
    CK(cudaMemsetAsync(r->d_io, 0, 4 * (size_t)r->nrays, st));
    CK(cudaMemsetAsync(a.wmax, 0, 4, st));
    CK(launch_lsqr_scale_u(a, inv_beta, st));
    const auto t0 = std::chrono::steady_clock::now();
    CK(cudaMemcpyAsync(host + 1, a.wmax, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    d2h_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    d2h_bytes += 4;
    unsigned bits;
    std::memcpy(&bits, host + 1, 4);
    float W;
    std::memcpy(&W, &bits, 4);
    const int E = (W > 0.f && r->hd_max > 0.f) ? quantum_exponent(r->hd_max, W, r->nrays) : 0;
    RaySetArgs s = rayset_args(r);
    s.a.weights = r->d_io;
    s.a.acc = r->d_acc;
    s.a.scale = std::ldexp(1.0, -E);
    CK(cudaMemsetAsync(r->d_acc, 0, (size_t)r->g.vol * 8, st));
    CK(launch_rayset_walk(true, s, r->device, st));
    CK(launch_grad_finish(r->d_acc, r->d_stage, r->g, E, st));
    launches += 3;
    return 1;
  }
};

// scipy's _sym_ortho
void sym_ortho(double a, double b, double* c, double* s, double* rr) {
  auto sign = [](double t) { return t > 0 ? 1.0 : t < 0 ? -1.0 : t; };
  if (b == 0) {
    *c = sign(a); *s = 0; *rr = std::fabs(a);
  } else if (a == 0) {
    *c = 0; *s = sign(b); *rr = std::fabs(b);
  } else if (std::fabs(b) > std::fabs(a)) {
    const double tau = a / b;
    *s = sign(b) / std::sqrt(1 + tau * tau);
    *c = *s * tau;
    *rr = b / *s;
  } else {
    const double tau = b / a;
    *c = sign(a) / std::sqrt(1 + tau * tau);
    *s = *c * tau;
    *rr = a / *c;
  }
}

}  // namespace

extern "C" int sweeptt_rayset_lsqr(sweeptt_rayset* r, const uint8_t* rows, const double* b,
                                   const sweeptt_lsqr_opts* opts, double* x_out, sweeptt_lsqr_info* info,
                                   sweeptt_stats* stats) {
  if (!r) return fail("null ray set");
  if (stats) std::memset(stats, 0, sizeof *stats);
  if (!b || !opts || !x_out) return fail("sweeptt_rayset_lsqr: b, opts and x_out are required");
  if (opts->struct_size != (int)sizeof *opts)
    return fail("sweeptt_rayset_lsqr: opts->struct_size is %d, expected %d", opts->struct_size, (int)sizeof *opts);
  if (info && info->struct_size != (int)sizeof *info)
    return fail("sweeptt_rayset_lsqr: info->struct_size is %d, expected %d", info->struct_size, (int)sizeof *info);
  const double damp = opts->damp, smooth = opts->smooth;
  if (!std::isfinite(damp) || damp < 0) return fail("sweeptt_rayset_lsqr: damp must be finite and >= 0");
  if (!std::isfinite(smooth) || smooth < 0) return fail("sweeptt_rayset_lsqr: smooth must be finite and >= 0");
  if (!(opts->atol >= 0) || !(opts->btol >= 0) || !(opts->conlim >= 0))
    return fail("sweeptt_rayset_lsqr: atol, btol and conlim must be >= 0");
  if (opts->iter_lim < 0) return fail("sweeptt_rayset_lsqr: iter_lim must be >= 0");
  if (!std::isfinite(r->hd_max)) return fail("sweeptt_rayset_lsqr: the star's edge lengths are not finite");
  std::vector<long long> row;
  for (long long q = 0; q < r->nrays; ++q) {
    const bool sel = rows ? rows[q] != 0 : r->status[q] == SWEEPTT_RAY_OK;
    if (!sel) continue;
    if (r->status[q] != SWEEPTT_RAY_OK) return fail("sweeptt_rayset_lsqr: rows selects ray %lld, which is not OK", q);
    row.push_back(q);
  }
  const long long m = (long long)row.size();
  for (long long i = 0; i < m; ++i)
    if (!std::isfinite(b[i])) return fail("sweeptt_rayset_lsqr: b[%lld] is not finite", i);

  const BoxGeom& g = r->g;
  const long long nx = g.nx, ny = g.ny, nz = g.nz;  // kernel axes: the caller's through perm
  long long cd[3];
  for (int k = 0; k < 3; ++k) cd[g.perm[k]] = k == 0 ? nx : k == 1 ? ny : nz;
  LsqrSolve S;
  S.r = r;
  S.st = r->ctx->stream;
  S.D = cd[0] * cd[1] * cd[2];
  const long long D = S.D;
  const long long mD = smooth > 0 ? (cd[0] - 1) * cd[1] * cd[2] + cd[0] * (cd[1] - 1) * cd[2] + cd[0] * cd[1] * (cd[2] - 1) : 0;
  const long long mu = m + mD;
  const long long nblk = (std::max({mu, D, 1LL}) + 2047) / 2048;
  CK(cudaSetDevice(r->device));
  cudaStream_t st = S.st;
  {
    const size_t bytes = 8 * (size_t)mu + 24 * (size_t)D + 8 * (size_t)m + 8 * (size_t)(nblk + 1);
    const cudaError_t e = cudaMalloc(&S.dev, bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      S.dev = nullptr;
      return fail("sweeptt_rayset_lsqr: no device memory for the %.3f GB workspace (%s)", bytes / 1e9, cudaGetErrorString(e));
    }
    const cudaError_t eh = cudaMallocHost(&S.host, 32);
    if (eh != cudaSuccess) {
      cudaGetLastError();
      S.host = nullptr;
      return fail("sweeptt_rayset_lsqr: no page-locked host memory (%s)", cudaGetErrorString(eh));
    }
  }
  LsqrArgs& a = S.a;
  double* p = static_cast<double*>(S.dev);
  a.u = p; p += mu;
  a.x = p; p += D;
  a.v = p; p += D;
  a.w = p; p += D;
  a.row = reinterpret_cast<long long*>(p); p += m;
  a.part = p; p += nblk;
  a.wmax = reinterpret_cast<unsigned*>(p);
  a.m = m;
  a.mD = mD;
  a.nx = (int)cd[0]; a.ny = (int)cd[1]; a.nz = (int)cd[2];
  a.smooth = smooth;
  a.io = r->d_io;
  a.stage = r->d_stage;
  a.ctas = lsqr_ctas();

  CK(cudaEventRecord(r->ev0, st));
  const auto t_h2d = std::chrono::steady_clock::now();
  if (m) {
    CK(cudaMemcpyAsync(a.u, b, 8 * (size_t)m, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(const_cast<long long*>(a.row), row.data(), 8 * (size_t)m, cudaMemcpyHostToDevice, st));
  }
  CK(cudaStreamSynchronize(st));  // pageable sources: the copies are complete
  const double h2d_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_h2d).count();
  if (mD) CK(cudaMemsetAsync(a.u + m, 0, 8 * (size_t)mD, st));
  CK(cudaMemsetAsync(a.x, 0, 8 * (size_t)D, st));

  // scipy's lsqr, x0 = None, calc_var = False
  const double eps = std::numeric_limits<double>::epsilon();
  const double atol = opts->atol, btol = opts->btol, conlim = opts->conlim;
  const int iter_lim = opts->iter_lim;
  int itn = 0, istop = 0;
  double ctol = 0;
  if (conlim > 0) ctol = 1 / conlim;
  double anorm = 0, acond = 0, dampsq = damp * damp, ddnorm = 0, res2 = 0, xnorm = 0, xxnorm = 0, z = 0, cs2 = -1,
         sn2 = 0;
  double bnorm, alfa = 0, beta;
  CK(launch_lsqr_sumsq(a.u, m, a.part, a.ctas, st, &S.launches));
  if (!S.read_norm(&bnorm)) return 0;
  beta = bnorm;
  if (beta > 0) {
    if (!S.backproject(1 / beta)) return 0;
    CK(cudaMemsetAsync(a.v, 0, 8 * (size_t)D, st));
    CK(launch_lsqr_v(a, 0.0, st, &S.launches));  // v = A^T u (- 0 * 0)
    if (!S.read_norm(&alfa)) return 0;
  } else {
    CK(cudaMemsetAsync(a.v, 0, 8 * (size_t)D, st));
  }
  if (alfa > 0) {
    CK(launch_lsqr_scale(a.v, D, 1 / alfa, st));
    ++S.launches;
  }
  CK(cudaMemcpyAsync(a.w, a.v, 8 * (size_t)D, cudaMemcpyDeviceToDevice, st));
  double rhobar = alfa, phibar = beta, rnorm = beta, r1norm = rnorm, r2norm = rnorm, arnorm = alfa * beta;

  const bool solved = arnorm == 0;  // scipy returns x = 0 before its loop
  while (!solved && itn < iter_lim) {
    itn = itn + 1;
    if (!S.project()) return 0;
    CK(launch_lsqr_u(a, alfa, st, &S.launches));
    if (!S.read_norm(&beta)) return 0;
    if (beta > 0) {
      if (!S.backproject(1 / beta)) return 0;
      anorm = std::sqrt(anorm * anorm + alfa * alfa + beta * beta + dampsq);
      CK(launch_lsqr_v(a, beta, st, &S.launches));
      if (!S.read_norm(&alfa)) return 0;
      if (alfa > 0) {
        CK(launch_lsqr_scale(a.v, D, 1 / alfa, st));
        ++S.launches;
      }
    }
    double rhobar1, psi;
    if (damp > 0) {
      rhobar1 = std::sqrt(rhobar * rhobar + dampsq);
      const double cs1 = rhobar / rhobar1;
      const double sn1 = damp / rhobar1;
      psi = sn1 * phibar;
      phibar = cs1 * phibar;
    } else {
      rhobar1 = rhobar;
      psi = 0.;
    }
    double cs, sn, rho;
    sym_ortho(rhobar1, beta, &cs, &sn, &rho);
    const double theta = sn * alfa;
    rhobar = -cs * alfa;
    const double phi = cs * phibar;
    phibar = sn * phibar;
    const double tau = sn * phi;
    double t1 = phi / rho;
    const double t2 = -theta / rho;
    CK(launch_lsqr_xw(a, t1, t2, 1 / rho, st, &S.launches));  // x += t1 w; sumsq of dk = (1/rho) w; w = v + t2 w
    double dknorm;
    if (!S.read_norm(&dknorm)) return 0;
    ddnorm = ddnorm + dknorm * dknorm;

    const double delta = sn2 * rho;
    const double gambar = -cs2 * rho;
    const double rhs = phi - delta * z;
    const double zbar = rhs / gambar;
    xnorm = std::sqrt(xxnorm + zbar * zbar);
    const double gamma = std::sqrt(gambar * gambar + theta * theta);
    cs2 = gambar / gamma;
    sn2 = theta / gamma;
    z = rhs / gamma;
    xxnorm = xxnorm + z * z;

    acond = anorm * std::sqrt(ddnorm);
    const double res1 = phibar * phibar;
    res2 = res2 + psi * psi;
    rnorm = std::sqrt(res1 + res2);
    arnorm = alfa * std::fabs(tau);

    if (damp > 0) {
      const double r1sq = rnorm * rnorm - dampsq * xxnorm;
      r1norm = std::sqrt(std::fabs(r1sq));
      if (r1sq < 0) r1norm = -r1norm;
    } else {
      r1norm = rnorm;
    }
    r2norm = rnorm;

    const double test1 = rnorm / bnorm;
    const double test2 = arnorm / (anorm * rnorm + eps);
    const double test3 = 1 / (acond + eps);
    t1 = test1 / (1 + anorm * xnorm / bnorm);
    const double rtol = btol + atol * anorm * xnorm / bnorm;

    if (itn >= iter_lim) istop = 7;
    if (1 + test3 <= 1) istop = 6;
    if (1 + test2 <= 1) istop = 5;
    if (1 + t1 <= 1) istop = 4;

    if (test3 <= ctol) istop = 3;
    if (test2 <= atol) istop = 2;
    if (test1 <= rtol) istop = 1;

    if (istop != 0) break;
  }

  CK(cudaEventRecord(r->ev1, st));
  const auto t_x = std::chrono::steady_clock::now();
  CK(cudaMemcpyAsync(x_out, a.x, 8 * (size_t)D, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  S.d2h_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_x).count();
  S.d2h_bytes += 8 * D;
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, r->ev0, r->ev1));
  if (info) {
    info->istop = istop;
    info->itn = itn;
    info->r1norm = r1norm;
    info->r2norm = r2norm;
    info->anorm = anorm;
    info->acond = acond;
    info->arnorm = arnorm;
    info->xnorm = xnorm;
  }
  if (stats) {
    stats->struct_size = (int)sizeof *stats;
    stats->solve_ms = ms;
    stats->kernel_launches = S.launches;
    stats->devices_used = 1;
    stats->h2d_ms = h2d_ms;
    stats->h2d_bytes = 16 * m;
    stats->d2h_ms = S.d2h_ms;
    stats->d2h_bytes = S.d2h_bytes;
  }
  return 1;
}

// ---------------------------------------------------------------------------------------
// event location (include/sweeptt.h, sweeptt_locate_events / sweeptt_misfit_box)
// ---------------------------------------------------------------------------------------

// Checks shared by both location calls; then the picks of nev events (NaN left out) go to the device as a CSR with
// RN(1/k) per event, and *a describes them, the fields of the call's stations and the result slots.  Every refusal
// comes before the first allocation.  nodes_per_thread (may be NULL): the location kernel's shape for these stations.
static int locate_prepare(sweeptt_ctx* c, ConstLease* lease, const char* who, int source_begin, int source_count,
                          const float* picks, int nev, LocateArgs* a, int* nodes_per_thread, sweeptt_stats* stats) {
  if (!ready(c, lease)) return 0;
  if (stats) std::memset(stats, 0, sizeof *stats);
  if (!check_source_range(c, who, source_begin, source_count)) return 0;
  if (nodes_per_thread && (*nodes_per_thread = locate_nodes_per_thread(source_count, c->device)) == 0)
    return fail("%s: %d stations do not fit the location kernel's shared memory (8 bytes per station and node, 32 nodes)",
                who, source_count);
  if (nev < 0) return fail("%s: nev = %d is negative", who, nev);
  if (nev > 0 && !picks) return fail("%s: null picks", who);
  const BoxGeom& g = c->g;
  if ((unsigned long long)g.nx * g.ny * g.nz > (1ull << 32))
    return fail("%s: %d x %d x %d nodes exceed 2^32, the argmin key holds a node index in 32 bits", who, g.nx, g.ny, g.nz);
  std::vector<int> off(1, 0), sta;
  std::vector<double> obs, rk;
  off.reserve((size_t)nev + 1);
  rk.reserve(nev);
  for (int e = 0; e < nev; ++e) {
    for (int s = 0; s < source_count; ++s) {
      const float v = picks[(size_t)e * source_count + s];
      if (std::isnan(v)) continue;
      if (std::isinf(v)) return fail("%s: pick of event %d at station %d is %cINF (a pick is finite, or NaN for none)",
                                     who, e, s, v > 0 ? '+' : '-');
      sta.push_back(s);
      obs.push_back((double)v);
    }
    if (sta.size() > (size_t)INT32_MAX) return fail("%s: more than 2^31 picks in one call", who);
    const int k = (int)sta.size() - off.back();
    off.push_back((int)sta.size());
    rk.push_back(k ? 1.0 / k : 0.0);
  }
  const size_t np = sta.size(), n = (size_t)nev;
  auto up16 = [](size_t b) { return (b + 15) / 16 * 16; };
  const size_t part[10] = {up16(4 * (n + 1)), up16(4 * np), up16(8 * np), up16(8 * n), up16(8 * n),
                           up16(12 * n),      up16(4 * n),  up16(8 * n),  up16(4 * n), up16(4 * n)};
  size_t at[11] = {0};
  for (int i = 0; i < 10; ++i) at[i + 1] = at[i] + part[i];
  if (!ensure_dev(c, &c->d_loc, &c->loc_cap, at[10])) return 0;
  unsigned char* b = c->d_loc;
  *a = LocateArgs{};
  a->g = g;
  a->tt = c->d_tt + (size_t)source_begin * g.vol;
  a->nsta = source_count;
  a->pick_off = reinterpret_cast<const int*>(b + at[0]);
  a->pick_sta = reinterpret_cast<const int*>(b + at[1]);
  a->pick_obs = reinterpret_cast<const double*>(b + at[2]);
  a->pick_rk = reinterpret_cast<const double*>(b + at[3]);
  a->key = reinterpret_cast<unsigned long long*>(b + at[4]);
  a->node = reinterpret_cast<int*>(b + at[5]);
  a->misfit = reinterpret_cast<float*>(b + at[6]);
  a->origin = reinterpret_cast<double*>(b + at[7]);
  a->npicks = reinterpret_cast<int*>(b + at[8]);
  a->status = reinterpret_cast<int*>(b + at[9]);
  const auto t0 = std::chrono::steady_clock::now();
  CK(cudaMemcpyAsync(b + at[0], off.data(), 4 * (n + 1), cudaMemcpyHostToDevice, c->stream));
  if (np) {
    CK(cudaMemcpyAsync(b + at[1], sta.data(), 4 * np, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(b + at[2], obs.data(), 8 * np, cudaMemcpyHostToDevice, c->stream));
  }
  if (n) CK(cudaMemcpyAsync(b + at[3], rk.data(), 8 * n, cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (stats) {
    stats->struct_size = (int)sizeof *stats;
    stats->devices_used = 1;
    stats->h2d_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    stats->h2d_bytes = (long long)(4 * (n + 1) + 12 * np + 8 * n);
  }
  return 1;
}

// Events per location launch (SWEEPTT_LOCATE_CHUNK): bounds the run time of one launch; the result does not depend on it.
static int locate_chunk() {
  int chunk = 4096;
  if (const char* e = getenv("SWEEPTT_LOCATE_CHUNK")) chunk = std::max(1, atoi(e));
  return chunk;
}

extern "C" int sweeptt_locate_events(sweeptt_ctx* c, int source_begin, int source_count, const float* picks, int nev,
                                     struct START* best_out, float* misfit_out, double* origin_out,
                                     int32_t* npicks_out, int32_t* status_out, sweeptt_stats* stats) {
  static const char* who = "sweeptt_locate_events";
  if (!best_out || !status_out) return fail("%s: best_out and status_out are required", who);
  ConstLease lease;
  LocateArgs a;
  int nb = 0;
  if (!locate_prepare(c, &lease, who, source_begin, source_count, picks, nev, &a, &nb, stats)) return 0;
  if (nev == 0) return 1;
  const int chunk = locate_chunk();
  long long launches = 0;
  CK(cudaEventRecord(c->ev0, c->stream));
  CK(cudaMemsetAsync(a.key, 0xff, 8 * (size_t)nev, c->stream));
  for (int e0 = 0; e0 < nev; e0 += chunk) {
    a.e_begin = e0;
    a.e_count = std::min(chunk, nev - e0);
    CK(launch_locate(a, nb, c->stream));
    ++launches;
  }
  CK(launch_locate_finish(a, nev, c->stream));
  CK(cudaEventRecord(c->ev1, c->stream));
  CK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));

  const auto t_copy = std::chrono::steady_clock::now();
  const size_t n = (size_t)nev;
  long long bytes = 16 * (long long)n;
  static_assert(sizeof(START) == 3 * sizeof(int), "START is three ints");
  CK(cudaMemcpyAsync(best_out, a.node, 12 * n, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(status_out, a.status, 4 * n, cudaMemcpyDeviceToHost, c->stream));
  if (misfit_out) { CK(cudaMemcpyAsync(misfit_out, a.misfit, 4 * n, cudaMemcpyDeviceToHost, c->stream)); bytes += 4 * n; }
  if (origin_out) { CK(cudaMemcpyAsync(origin_out, a.origin, 8 * n, cudaMemcpyDeviceToHost, c->stream)); bytes += 8 * n; }
  if (npicks_out) { CK(cudaMemcpyAsync(npicks_out, a.npicks, 4 * n, cudaMemcpyDeviceToHost, c->stream)); bytes += 4 * n; }
  CK(cudaStreamSynchronize(c->stream));
  if (stats) {
    stats->solve_ms = ms;
    stats->kernel_launches = launches + 1;
    stats->d2h_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_copy).count();
    stats->d2h_bytes = bytes;
  }
  return 1;
}

extern "C" int sweeptt_misfit_box(sweeptt_ctx* c, int source_begin, int source_count, const float* picks,
                                  float* misfit_out, sweeptt_stats* stats) {
  static const char* who = "sweeptt_misfit_box";
  if (!picks || !misfit_out) return fail("%s: picks and misfit_out are required", who);
  ConstLease lease;
  LocateArgs a;
  if (!locate_prepare(c, &lease, who, source_begin, source_count, picks, 1, &a, nullptr, stats)) return 0;
  const size_t dense = (size_t)c->g.nx * c->g.ny * c->g.nz;
  if (!ensure_stage(c, dense)) return 0;
  CK(cudaEventRecord(c->ev0, c->stream));
  CK(launch_misfit_box(a, c->d_stage, c->stream));
  CK(cudaEventRecord(c->ev1, c->stream));
  CK(cudaEventSynchronize(c->ev1));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
  const auto t_copy = std::chrono::steady_clock::now();
  CK(cudaMemcpyAsync(misfit_out, c->d_stage, dense * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (stats) {
    stats->solve_ms = ms;
    stats->kernel_launches = 1;
    stats->d2h_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_copy).count();
    stats->d2h_bytes = (long long)dense * 4;
  }
  return 1;
}

extern "C" long long sweeptt_relaxations_per_round(sweeptt_ctx* c) { return c ? c->pulls_per_round : 0; }
extern "C" size_t sweeptt_pool_bytes(sweeptt_ctx* c) { return c ? c->pool_bytes : 0; }
extern "C" int sweeptt_debug_model_stats(sweeptt_ctx* c, float* vmin, float* vmax, float* vpos) {
  if (!c || !c->have_model) return fail("sweeptt_debug_model_stats: no model");
  if (vmin) *vmin = c->min_slowness;
  if (vmax) *vmax = c->max_slowness;
  if (vpos) *vpos = c->pos_slowness;
  return 1;
}
extern "C" long long sweeptt_tiles_per_source(sweeptt_ctx* c) {
  return (c && c->have_model) ? (long long)c->g.ntx * c->g.nty * c->g.ntz : 0;
}

// ---------------------------------------------------------------------------------------
// one-shot solve + multi-start dispatcher
// ---------------------------------------------------------------------------------------
static std::mutex g_cache_mu;
namespace { struct CacheEntry; }
extern "C" void sweeptt_release_cache(void);

// The device's cached context, held exclusively for one sweeptt_solve call (two host threads calling
// sweeptt_solve for the same device take turns)
namespace {
struct CacheEntry {
  std::mutex busy;
  sweeptt_ctx* ctx = nullptr;
};
std::map<int, CacheEntry*> g_cache_entries;
struct CachedCtx {
  CacheEntry* e = nullptr;
  sweeptt_ctx* ctx = nullptr;
  CachedCtx(int device, const sweeptt_opts& o) {
    {
      std::lock_guard<std::mutex> lk(g_cache_mu);
      auto it = g_cache_entries.find(device);
      if (it == g_cache_entries.end()) it = g_cache_entries.emplace(device, new CacheEntry()).first;
      e = it->second;
    }
    e->busy.lock();
    if (e->ctx) {
      sweeptt_ctx* c = e->ctx;
      const bool star_opts_changed = c->opts.star_used != o.star_used || c->opts.kernel != o.kernel;
      const bool plan_opts_changed = c->opts.loop != o.loop || c->opts.max_rounds != o.max_rounds ||
                                     c->opts.profile_kernels != o.profile_kernels;
      c->opts = o;
      c->opts.device = device;
      if (star_opts_changed) c->have_star = false;
      if (plan_opts_changed) invalidate_graph(c);
    } else {
      sweeptt_opts oo = o;
      oo.device = device;
      e->ctx = sweeptt_create(&oo);
    }
    ctx = e->ctx;
  }
  ~CachedCtx() { if (e) e->busy.unlock(); }
};
}  // namespace

extern "C" void sweeptt_release_cache(void) {
  std::lock_guard<std::mutex> lk(g_cache_mu);
  for (auto& kv : g_cache_entries) {
    std::lock_guard<std::mutex> use(kv.second->busy);
    if (kv.second->ctx) sweeptt_destroy(kv.second->ctx);
    kv.second->ctx = nullptr;
  }
}

namespace {
struct HostCopy { void* dst; const void* src; size_t bytes; };
void CUDART_CB host_copy_fn(void* p) {
  const HostCopy* j = static_cast<const HostCopy*>(p);
  std::memcpy(j->dst, j->src, j->bytes);
}
}  // namespace

// Ring of dense staging boxes for the way out: box s is un-padded on the solve stream (a few microseconds of SM
// time behind the wave that produced it) and copied to the host by the copy stream while the next wave is relaxed.
static int ensure_out_ring(sweeptt_ctx* c, size_t dense_floats, int want_boxes) {
  size_t boxes = std::max<size_t>(2, std::min<size_t>((size_t)want_boxes, std::max<size_t>(2, (size_t(1) << 30) / (dense_floats * 4))));
  if (c->out_ring_box_floats == dense_floats && c->out_ring_boxes >= boxes) return 1;
  if (c->copy_stream) CK(cudaStreamSynchronize(c->copy_stream));
  dev_free(c, c->d_out_ring, c->out_ring_boxes * c->out_ring_box_floats * 4);
  c->d_out_ring = nullptr; c->out_ring_boxes = 0; c->out_ring_box_floats = 0;
  if (c->h_out_ring) { cudaFreeHost(c->h_out_ring); c->h_out_ring = nullptr; }
  if (!dev_alloc(c, (void**)&c->d_out_ring, boxes * dense_floats * 4)) return 0;
  c->out_ring_boxes = boxes; c->out_ring_box_floats = dense_floats;
  while (c->ring_unpadded.size() < boxes) {
    cudaEvent_t a, b;
    CK(cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
    c->ring_unpadded.push_back(a); c->ring_copied.push_back(b);
  }
  if (!c->copy_stream) CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  return 1;
}

static int solve_on_device(int device, const sweeptt_opts& o, const float* slowness, int nx, int ny, int nz,
                           const FS* fs, int starsize, const START* starts, int numstart, float* const* tt_out,
                           sweeptt_stats* st) {
  static const bool timing = getenv("SWEEPTT_DEBUG_TIMING") != nullptr;
  const auto t0 = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (timing) fprintf(stderr, "[sweeptt-timing] dev %d %-12s +%.3f ms\n", device, what,
                        std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
  };
  CachedCtx cc(device, o);  // (exclusive use of the device's cached context for this call)
  sweeptt_ctx* c = cc.ctx;
  if (!c) return 0;
  std::memset(st, 0, sizeof *st);
  CK(cudaSetDevice(device));
  CK(cudaEventRecord(c->ev2, c->stream));
  if (!sweeptt_set_model(c, slowness, nx, ny, nz)) return 0;
  CK(cudaEventRecord(c->ev3, c->stream));
  CK(cudaEventSynchronize(c->ev3));
  float h2d_ms = 0;  // read now: the run below reuses these events
  CK(cudaEventElapsedTime(&h2d_ms, c->ev2, c->ev3));
  lap("set_model");
  const bool same_star = c->have_star && (int)c->fs.size() == starsize &&
                         std::memcmp(c->fs.data(), fs, sizeof(FS) * starsize) == 0;
  if (!same_star && !sweeptt_set_star(c, fs, starsize)) return 0;
  if (!sweeptt_set_sources(c, starts, numstart)) return 0;
  lap("star+sources");
  ConstLease lease;
  if (!ready(c, &lease)) return 0;
  lap("ready");
  // device -> host, overlapped with the solve of the later waves: un-pad into a ring of dense boxes on the solve
  // stream, one contiguous copy per source on the copy stream
  const size_t dense = (size_t)nx * ny * nz;
  if (!ensure_out_ring(c, dense, 2 * std::max(1, std::min(numstart, 16)))) return 0;
  size_t ring_pos = 0;
  std::vector<char> ring_used(c->out_ring_boxes, 0);
  // page-locked or pageable destination?  (all boxes of a call are assumed to be of one kind: the first decides)
  bool pageable_out = false;
  {
    cudaPointerAttributes pa{};
    if (cudaPointerGetAttributes(&pa, tt_out[0]) != cudaSuccess) { cudaGetLastError(); pageable_out = true; }
    else pageable_out = pa.type == cudaMemoryTypeUnregistered;
    if (getenv("SWEEPTT_NO_HOST_RING")) pageable_out = false;
    if (pageable_out && !c->h_out_ring &&
        cudaHostAlloc(&c->h_out_ring, c->out_ring_boxes * dense * 4, cudaHostAllocDefault) != cudaSuccess) {
      cudaGetLastError();
      c->h_out_ring = nullptr;
      pageable_out = false;  // no page-locked memory to be had: plain (staged) copies
    }
  }
  std::vector<HostCopy*> jobs;
  struct JobGuard {  // (an error return must not free a job whose callback is still queued)
    std::vector<HostCopy*>& j;
    cudaStream_t* st;
    ~JobGuard() {
      if (!j.empty() && *st) cudaStreamSynchronize(*st);
      for (auto* x : j) delete x;
    }
  } job_guard{jobs, &c->copy_stream};
  const auto t_first = std::chrono::steady_clock::now();
  auto drain = [&](int s0, int ns, cudaStream_t st) -> int {
    for (int s = s0; s < s0 + ns; ++s) {
      const size_t slot = ring_pos++ % c->out_ring_boxes;
      float* box = c->d_out_ring + slot * dense;
      if (ring_used[slot]) CK(cudaStreamWaitEvent(st, c->ring_copied[slot], 0));
      CK(launch_unpad_box(c->d_tt + (size_t)s * c->g.vol, box, c->g, st));
      CK(cudaEventRecord(c->ring_unpadded[slot], st));
      CK(cudaStreamWaitEvent(c->copy_stream, c->ring_unpadded[slot], 0));
      if (pageable_out) {
        // the caller's box is plain malloc memory (the reference's boxalloc): a device->pageable copy would block this
        // thread -- and with it the enqueueing of the next waves -- at the driver's staging speed.  Stop over in the
        // page-locked twin of the ring and let the copy stream's host callback do the memcpy behind the solve.
        float* hbox = c->h_out_ring + slot * dense;
        CK(cudaMemcpyAsync(hbox, box, dense * 4, cudaMemcpyDeviceToHost, c->copy_stream));
        jobs.push_back(new HostCopy{tt_out[s], hbox, dense * 4});
        CK(cudaLaunchHostFunc(c->copy_stream, host_copy_fn, jobs.back()));
      } else {
        CK(cudaMemcpyAsync(tt_out[s], box, dense * 4, cudaMemcpyDeviceToHost, c->copy_stream));
      }
      CK(cudaEventRecord(c->ring_copied[slot], c->copy_stream));
      ring_used[slot] = 1;
    }
    return 1;
  };
  if (!run_locked(c, st, drain)) return 0;
  lap("solved");
  const auto t_solved = std::chrono::steady_clock::now();
  CK(cudaStreamSynchronize(c->copy_stream));
  lap("copied");
  st->h2d_ms = h2d_ms;
  st->h2d_bytes = (long long)nx * ny * nz * 4;
  // what the copies cost on top of the solve: the tail after the last wave converged (the rest ran behind it)
  st->d2h_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_solved).count();
  (void)t_first;
  st->d2h_bytes = (long long)dense * 4 * numstart;
  st->kernel_launches += 2 + numstart;
  return 1;
}

extern "C" void* sweeptt_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (sweeptt_device_count() <= 0) { fail("no CUDA device available"); return nullptr; }
  const cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocPortable);
  if (e != cudaSuccess) { cudaGetLastError(); fail("cudaHostAlloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e)); return nullptr; }
  return p;
}
extern "C" void sweeptt_host_free(void* p) { if (p) cudaFreeHost(p); }

extern "C" int sweeptt_solve(const float* slowness, int nx, int ny, int nz, const struct FS* fs, int starsize,
                             const struct START* starts, int numstart, float* const* tt_out, const sweeptt_opts* opts,
                             sweeptt_stats* stats) {
  if (!slowness || !fs || !starts || !tt_out) return fail("sweeptt_solve: null argument");
  if (numstart <= 0) return fail("sweeptt_solve: need at least one start point");
  sweeptt_opts o{};
  if (opts) std::memcpy(&o, opts, std::min<size_t>(sizeof o, opts->struct_size > 0 ? opts->struct_size : sizeof o));
  const int ndev_avail = sweeptt_device_count();
  if (ndev_avail <= 0) return fail("no CUDA device available: the sweep has no CPU fallback");
  int ndev = std::max(1, o.num_devices);
  if (ndev > ndev_avail) return fail("num_devices = %d but only %d CUDA devices are visible", ndev, ndev_avail);
  ndev = std::min(ndev, numstart);
  sweeptt_stats total{};
  total.struct_size = sizeof total;
  if (ndev == 1) {
    int dev = o.device;
    if (dev < 0) cudaGetDevice(&dev);
    if (!solve_on_device(dev, o, slowness, nx, ny, nz, fs, starsize, starts, numstart, tt_out, &total)) return 0;
  } else {
    // Sources are independent (mpi/backup.c:351-363): deal them round-robin, one host thread
    // and one stream per GPU, no inter-GPU traffic.
    std::vector<std::vector<START>> shard(ndev);
    std::vector<std::vector<float*>> outs(ndev);
    for (int s = 0; s < numstart; ++s) {
      shard[s % ndev].push_back(starts[s]);
      outs[s % ndev].push_back(tt_out[s]);
    }
    std::vector<sweeptt_stats> st(ndev);
    std::vector<int> ok(ndev, 0);
    std::vector<std::string> errs(ndev);
    std::vector<std::thread> th;
    for (int d = 0; d < ndev; ++d)
      th.emplace_back([&, d] {
        ok[d] = solve_on_device(d, o, slowness, nx, ny, nz, fs, starsize, shard[d].data(), (int)shard[d].size(),
                                outs[d].data(), &st[d]);
        if (!ok[d]) errs[d] = g_err;
      });
    for (auto& t : th) t.join();
    for (int d = 0; d < ndev; ++d)
      if (!ok[d]) return fail("device %d: %s", d, errs[d].c_str());
    for (int d = 0; d < ndev; ++d) {
      total.rounds = std::max(total.rounds, st[d].rounds);
      total.kernel_used = st[d].kernel_used;
      total.kernel_launches += st[d].kernel_launches;
      total.relax_launches += st[d].relax_launches;
      total.tile_visits += st[d].tile_visits;
      total.relaxations += st[d].relaxations;
      total.solve_ms = std::max(total.solve_ms, st[d].solve_ms);
      total.relax_kernel_ms = std::max(total.relax_kernel_ms, st[d].relax_kernel_ms);
      total.h2d_ms = std::max(total.h2d_ms, st[d].h2d_ms);
      total.d2h_ms = std::max(total.d2h_ms, st[d].d2h_ms);
      total.h2d_bytes += st[d].h2d_bytes;
      total.d2h_bytes += st[d].d2h_bytes;
      total.units_run += st[d].units_run;
      total.units_changed += st[d].units_changed;
    }
  }
  total.devices_used = ndev;
  if (stats) *stats = total;
  return 1;
}

// ---------------------------------------------------------------------------------------
// single huge grid over the devices of one box: ONE shared box in peer memory
// ---------------------------------------------------------------------------------------
// Replaces the MPI ghost-cell decomposition (mpi/16partsmpi.c:740-909: 16 ranks, ghost width 7, Isend/Irecv of the
// ghost planes every sweep, Allreduce of the change flag).  B200-native form: the slowness box and the travel-time
// box are each ONE virtual address range (CUDA virtual memory management) whose physical pages live BLOCK-CYCLICALLY
// on the devices -- blocks of a few tiles along the kernel's x axis, dealt round-robin, so that a single expanding
// front keeps every device busy.  Every device ("part") relaxes the tiles of the blocks it owns with the unchanged
// tiled kernel: its TMA loads fetch halo planes that belong to a neighbour block straight from the owner's memory
// over NVLink, its stores go to its own pages, and a changed tile wakes a neighbour tile by an atomicMin on the key
// array of THAT tile's owner.  There is no halo exchange step, no ghost copy and no per-sweep host synchronisation of
// the data path: the transfer is fused into the relaxation kernel tile by tile.  All values only ever decrease and
// every read is a valid upper bound, so stale remote reads cost work, never correctness, and the fixed point is the
// single-device field bit for bit.  The devices follow ONE activation front (each publishes its smallest pending key,
// the bucket threshold hangs on the smallest one anywhere); termination is detected by the host threads without any
// barrier: all parts idle over a window in which every part ran a complete batch that found nothing.
namespace {

struct VmmApi {
  PFN_cuMemGetAllocationGranularity_v10020 granularity = nullptr;
  PFN_cuMemAddressReserve_v10020 reserve = nullptr;
  PFN_cuMemCreate_v10020 create = nullptr;
  PFN_cuMemMap_v10020 map = nullptr;
  PFN_cuMemSetAccess_v10020 set_access = nullptr;
  PFN_cuMemUnmap_v10020 unmap = nullptr;
  PFN_cuMemRelease_v10020 release = nullptr;
  PFN_cuMemAddressFree_v10020 address_free = nullptr;
  bool ok = false;
};
const VmmApi& vmm() {
  static VmmApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    auto get = [](const char* name) -> void* {
      void* p = nullptr;
      cudaDriverEntryPointQueryResult q;
      if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return nullptr;
      return p;
    };
    api.granularity = (PFN_cuMemGetAllocationGranularity_v10020)get("cuMemGetAllocationGranularity");
    api.reserve = (PFN_cuMemAddressReserve_v10020)get("cuMemAddressReserve");
    api.create = (PFN_cuMemCreate_v10020)get("cuMemCreate");
    api.map = (PFN_cuMemMap_v10020)get("cuMemMap");
    api.set_access = (PFN_cuMemSetAccess_v10020)get("cuMemSetAccess");
    api.unmap = (PFN_cuMemUnmap_v10020)get("cuMemUnmap");
    api.release = (PFN_cuMemRelease_v10020)get("cuMemRelease");
    api.address_free = (PFN_cuMemAddressFree_v10020)get("cuMemAddressFree");
    api.ok = api.granularity && api.reserve && api.create && api.map && api.set_access && api.unmap && api.release &&
             api.address_free;
  });
  return api;
}

// One virtual address range, chunk c backed by memory of device chunk_dev[c]; readable and writable by `devices`.
struct SharedBox {
  CUdeviceptr va = 0;
  size_t bytes = 0;
  struct Chunk { size_t off = 0, size = 0; int device = 0; bool mapped = false; };
  std::vector<Chunk> chunks;

  int create(const std::vector<size_t>& cuts, const std::vector<int>& chunk_dev, const std::vector<int>& devices) {
    const VmmApi& v = vmm();
    if (!v.ok) return fail("CUDA virtual memory management entry points are not available from this driver");
    bytes = cuts.back();
    CUresult r = v.reserve(&va, bytes, 0, 0, 0);
    if (r != CUDA_SUCCESS) { va = 0; return fail("cuMemAddressReserve(%zu bytes) failed: %d", bytes, (int)r); }
    for (size_t c = 0; c + 1 < cuts.size(); ++c) {
      Chunk ch;
      ch.off = cuts[c]; ch.size = cuts[c + 1] - cuts[c]; ch.device = chunk_dev[c];
      if (ch.size == 0) continue;
      CUmemAllocationProp prop = {};
      prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
      prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
      prop.location.id = ch.device;
      CUmemGenericAllocationHandle h;
      r = v.create(&h, ch.size, &prop, 0);
      if (r != CUDA_SUCCESS) return fail("cuMemCreate(%zu bytes on device %d) failed: %d", ch.size, ch.device, (int)r);
      r = v.map(va + ch.off, ch.size, 0, h, 0);
      v.release(h);  // the mapping keeps the memory alive
      if (r != CUDA_SUCCESS) return fail("cuMemMap failed: %d", (int)r);
      ch.mapped = true;
      chunks.push_back(ch);
    }
    std::vector<CUmemAccessDesc> acc;
    for (int d : devices) {
      CUmemAccessDesc a = {};
      a.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
      a.location.id = d;
      a.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
      acc.push_back(a);
    }
    r = v.set_access(va, bytes, acc.data(), acc.size());
    if (r != CUDA_SUCCESS) return fail("cuMemSetAccess failed: %d (peer access between the devices is required)", (int)r);
    return 1;
  }
  void destroy() {
    const VmmApi& v = vmm();
    for (auto& ch : chunks)
      if (ch.mapped) v.unmap(va + ch.off, ch.size);
    chunks.clear();
    if (va) v.address_free(va, bytes);
    va = 0; bytes = 0;
  }
};

struct Part {
  sweeptt_ctx* ctx = nullptr;
  int device = 0;
  std::vector<std::pair<int, int>> blocks;  // owned planes [x0,x1) of the kernel's x axis (logical coordinates)
  ConstLease lease;
  int ok = 1;
  std::string err;
  double min_slow = std::numeric_limits<double>::infinity(), sum_slow = 0;
  float max_slow = 0.f, pos_slow = std::numeric_limits<float>::infinity();  // domain guard (check_domain)
  unsigned long long cnt_slow = 0;
  bool bad_slow = false;
};

// simple reusable barrier for the setup phases (std::barrier needs C++20)
struct PhaseBarrier {
  std::mutex mu;
  std::condition_variable cv;
  int n, waiting = 0, phase = 0;
  explicit PhaseBarrier(int parts) : n(parts) {}
  void wait() {
    std::unique_lock<std::mutex> lk(mu);
    const int ph = phase;
    if (++waiting == n) { waiting = 0; ++phase; cv.notify_all(); }
    else cv.wait(lk, [&] { return phase != ph; });
  }
};
}  // namespace

// `fetch(origin, dims, dst)` fills dst with the caller-order sub-box of the slowness model
static int solve_slabs_impl(const std::function<int(const int*, const int*, float*)>& fetch, int nx, int ny, int nz,
                            const struct FS* fs, int starsize, struct START start, float* tt_out,
                            const sweeptt_opts* opts, sweeptt_stats* stats) {
  if (!fs || !tt_out) return fail("sweeptt_solve_slabs: null argument");
  sweeptt_opts o{};
  if (opts) std::memcpy(&o, opts, std::min<size_t>(sizeof o, opts->struct_size > 0 ? opts->struct_size : sizeof o));
  const int ndev = sweeptt_device_count();
  if (ndev <= 0) return fail("no CUDA device available: the sweep has no CPU fallback");
  const int G = std::max(1, o.num_devices);  // parts; more parts than devices share devices round-robin
  if (G > MAX_PARTS) return fail("at most %d parts", MAX_PARTS);
  const int axis = o.slab_axis;
  if (axis < 0 || axis > 2) return fail("slab_axis must be 0 (x), 1 (y) or 2 (z)");
  const int n[3] = {nx, ny, nz};
  if (nx <= 0 || ny <= 0 || nz <= 0) return fail("bad dimensions %d x %d x %d", nx, ny, nz);
  if (start.i < 0 || start.i >= nx || start.j < 0 || start.j >= ny || start.k < 0 || start.k >= nz)
    return fail("start point (%d,%d,%d) is outside the %d x %d x %d model", start.i, start.j, start.k, nx, ny, nz);
  if (G > n[axis]) return fail("more slabs (%d) than planes (%d) along the slab axis", G, n[axis]);

  std::vector<Part> parts(G);
  SharedBox box_tt;
  std::vector<int> devices;
  for (int p = 0; p < G; ++p) {
    parts[p].device = p % ndev;
    if (std::find(devices.begin(), devices.end(), parts[p].device) == devices.end()) devices.push_back(parts[p].device);
  }
  auto cleanup = [&] {
    for (auto& pt : parts) {
      pt.lease.release();
      if (pt.ctx) { cudaSetDevice(pt.device); cudaStreamSynchronize(pt.ctx->stream); sweeptt_destroy(pt.ctx); pt.ctx = nullptr; }
    }
    box_tt.destroy();
  };
  // ---- peer access for the per-part arrays (keys, bounds, state); the shared boxes get theirs from cuMemSetAccess ----
  for (int a : devices)
    for (int b : devices) {
      if (a == b) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, a, b);
      if (!can) return fail("devices %d and %d cannot access each other's memory", a, b);
      cudaSetDevice(a);
      if (cudaDeviceEnablePeerAccess(b, 0) != cudaSuccess) cudaGetLastError();  // (already enabled is fine)
    }
  // ---- one context per part, all with the same geometry: kernel x = the caller's slab axis ----
  BoxGeom g{};
  for (int p = 0; p < G; ++p) {
    Part& pt = parts[p];
    sweeptt_opts so = o;
    so.device = pt.device;
    so.num_devices = 1;
    so.kernel = SWEEPTT_KERNEL_TILED;
    pt.ctx = sweeptt_create(&so);
    if (!pt.ctx) { cleanup(); return 0; }
    pt.ctx->force_x_axis = axis;
    pt.ctx->external_boxes = true;
    if (!compute_geometry(pt.ctx, nx, ny, nz, &pt.ctx->g)) { cleanup(); return 0; }
    g = pt.ctx->g;
  }
  // Ownership blocks along kernel x, dealt round-robin (block-cyclic): G * cycles blocks of (almost) equal size, about
  // 8 tiles each (2 GPUs, 1201x1201x251: blocks of 2 tiles 267 ms, 4: 227, 8: 213, 16: 210), so that every part owns
  // the same number of tiles to within `cycles`.
  int tpb_target = 8;
  if (const char* e = getenv("SWEEPTT_BLOCK_TILES")) tpb_target = std::max(1, atoi(e));
  const int cycles = std::max(1, (g.ntx + G * tpb_target / 2) / (G * tpb_target));
  const int nblocks = std::min(g.ntx, G * cycles);
  std::vector<int> blk_start(nblocks + 1);
  for (int b = 0; b <= nblocks; ++b) blk_start[b] = (int)((long long)g.ntx * b / nblocks);
  int tpb = 1;  // largest block, in tiles
  std::vector<unsigned char> tx_owner(g.ntx);
  for (int b = 0; b < nblocks; ++b) {
    tpb = std::max(tpb, blk_start[b + 1] - blk_start[b]);
    const int x0 = blk_start[b] * TX, x1 = std::min(g.nx, blk_start[b + 1] * TX);
    if (x0 < x1) parts[b % G].blocks.push_back({x0, x1});
    for (int t = blk_start[b]; t < blk_start[b + 1]; ++t) tx_owner[t] = (unsigned char)(b % G);
  }
  // memory chunks follow the blocks (rounded to the allocation granularity; a chunk may be empty on small grids)
  {
    const VmmApi& v = vmm();
    if (!v.ok) { cleanup(); return fail("CUDA virtual memory management entry points are not available from this driver"); }
    size_t gran = 2u << 20;
    for (int d : devices) {
      CUmemAllocationProp prop = {};
      prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
      prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
      prop.location.id = d;
      size_t gd = 0;
      if (v.granularity(&gd, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) == CUDA_SUCCESS && gd > gran) gran = gd;
    }
    const size_t plane_bytes = (size_t)g.sx * 4;
    const size_t total = ((size_t)g.vol * 4 + gran - 1) / gran * gran;
    std::vector<size_t> cuts;
    std::vector<int> chunk_dev;
    for (int b = 0; b < nblocks; ++b) {
      const size_t first_plane = b == 0 ? 0 : (size_t)blk_start[b] * TX + AX;  // padded plane index where the block starts
      cuts.push_back(std::min(total, first_plane * plane_bytes / gran * gran));
      chunk_dev.push_back(parts[b % G].device);
    }
    cuts.push_back(total);
    for (int d : devices) { cudaSetDevice(d); cudaFree(0); }  // primary contexts exist before memory is placed
    if (!box_tt.create(cuts, chunk_dev, devices)) { cleanup(); return 0; }
  }
  int R = 0;
  for (int l = 0; l < starsize; ++l) R = std::max(R, std::abs(axis == 0 ? fs[l].i : axis == 1 ? fs[l].j : fs[l].k));
  (void)R;

  // ---- set-up, upload, solve and gather run in one host thread per part ----
  const auto t_begin = std::chrono::steady_clock::now();
  std::chrono::steady_clock::time_point t_solve0, t_solve1, t_end;
  PhaseBarrier bar(G);
  Quiescence quiet(G);
  const int K = o.rounds_per_poll > 0 ? o.rounds_per_poll : 4;
  float* const d_tt = reinterpret_cast<float*>(box_tt.va);
  const int PB = tpb * TX + 2 * RXY_MAX;  // planes per block of the local slowness copies (block + halo on both sides)
  const float INF = std::numeric_limits<float>::infinity();
  std::atomic<int> setup_failed{0};
  std::vector<long long> batches(G, 0), idle_batches(G, 0);
  std::vector<double> busy_ms(G, 0.0);

  auto part_main = [&](int p) {
    Part& pt = parts[p];
    sweeptt_ctx* c = pt.ctx;
    auto bail = [&](const char* what) { pt.ok = 0; pt.err = std::string(what) + ": " + g_err; setup_failed = 1; };
#define PCK(call)                                                                                       \
  do {                                                                                                  \
    cudaError_t e__ = (call);                                                                           \
    if (e__ != cudaSuccess && pt.ok) { pt.ok = 0; pt.err = std::string(#call) + ": " + cudaGetErrorString(e__); setup_failed = 1; } \
  } while (0)
    PCK(cudaSetDevice(pt.device));
    // phase 1: +INF into the pages of the shared travel-time box that this part's DEVICE holds, and into the part's
    // local slowness copy (every owned block with its halo planes; apron and out-of-grid planes stay +INF)
    for (const auto& ch : box_tt.chunks) {
      int first = -1;  // chunks of one device are filled by the first part on that device
      for (int q = 0; q < G && first < 0; ++q) if (parts[q].device == ch.device) first = q;
      if (first != p) continue;
      PCK(launch_fill(reinterpret_cast<float*>(box_tt.va + ch.off), (long long)(ch.size / 4), INF, c->stream));
    }
    c->slow_pb = PB;
    c->slow_planes = (long long)std::max<size_t>(1, pt.blocks.size()) * PB;
    if (pt.ok && !dev_alloc(c, (void**)&c->d_slow, (size_t)c->slow_planes * g.sx * 4)) bail("local slowness copy");
    if (pt.ok) PCK(launch_fill(c->d_slow, c->slow_planes * g.sx, INF, c->stream));
    PCK(cudaStreamSynchronize(c->stream));
    bar.wait();
    // phase 2: upload the owned blocks of the model + halo planes (sub-box in caller order -> padded local copy)
    c->d_tt = d_tt; c->tt_cap = 1;
    c->have_model = true;
    if (pt.ok && !setup_failed) {
      auto ext = [&](const std::pair<int, int>& b) {  // planes the block reads: itself + the star radius on both sides
        return std::make_pair(std::max(0, b.first - RXY_MAX), std::min(g.nx, b.second + RXY_MAX));
      };
      size_t stage_floats = 0;
      for (auto& b : pt.blocks) {
        int sub[3] = {nx, ny, nz};
        sub[axis] = ext(b).second - ext(b).first;
        stage_floats = std::max(stage_floats, (size_t)sub[0] * sub[1] * sub[2]);
      }
      float* h_stage = nullptr;
      if (stage_floats && (!ensure_stage(c, stage_floats) || cudaMallocHost(&h_stage, stage_floats * 4) != cudaSuccess)) bail("staging");
      for (size_t lb = 0; lb < pt.blocks.size(); ++lb) {
        if (!pt.ok) break;
        const auto b = pt.blocks[lb];
        const auto e = ext(b);
        int sub[3] = {nx, ny, nz}, org[3] = {0, 0, 0};
        sub[axis] = e.second - e.first;
        org[axis] = e.first;
        const size_t cnt = (size_t)sub[0] * sub[1] * sub[2];
        if (!fetch(org, sub, h_stage)) { bail("reading the model"); break; }
        PCK(cudaMemcpyAsync(c->d_stage, h_stage, cnt * 4, cudaMemcpyHostToDevice, c->stream));
        BoxGeom gs = g;
        gs.nx = e.second - e.first;
        const long long ds[3] = {(long long)sub[1] * sub[2], (long long)sub[2], 1};
        for (int q = 0; q < 3; ++q) gs.dstride[q] = ds[g.perm[q]];
        // local plane of logical plane x of this block: lb * PB + (x - b.first) + 7  (= padded plane x + AX of the
        // global box, shifted to the block's origin); launch_pad_box writes relative plane r at r + AX
        PCK(launch_pad_box(c->d_stage, c->d_slow + ((long long)lb * PB + (e.first - b.first) + RXY_MAX - AX) * g.sx, gs, c->stream));
        unsigned r[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        PCK(launch_min_slowness(c->d_stage, (long long)cnt, reinterpret_cast<unsigned*>(c->d_viol), c->stream));
        PCK(cudaMemcpyAsync(r, c->d_viol, sizeof r, cudaMemcpyDeviceToHost, c->stream));
        PCK(cudaStreamSynchronize(c->stream));
        float vmin, vmax, vpos; double sum; unsigned long long cn;
        std::memcpy(&vmin, &r[0], 4); std::memcpy(&sum, &r[2], 8); std::memcpy(&cn, &r[4], 8);
        std::memcpy(&vmax, &r[6], 4); std::memcpy(&vpos, &r[7], 4);
        if (r[1]) pt.bad_slow = true;
        pt.min_slow = std::min(pt.min_slow, (double)vmin);
        pt.max_slow = std::max(pt.max_slow, vmax);
        pt.pos_slow = std::min(pt.pos_slow, vpos);
        pt.sum_slow += sum; pt.cnt_slow += cn;
      }
      if (h_stage) cudaFreeHost(h_stage);
    }
    bar.wait();
    // phase 3: model statistics are global; star, start point, per-part scheduling arrays
    if (pt.ok && !setup_failed) {
      double mn = std::numeric_limits<double>::infinity(), sum = 0;
      float mx = 0.f, pos = INF;
      unsigned long long cn = 0;
      bool bad = false;
      for (auto& q : parts) {
        mn = std::min(mn, q.min_slow); mx = std::max(mx, q.max_slow); pos = std::min(pos, q.pos_slow);
        sum += q.sum_slow; cn += q.cnt_slow; bad = bad || q.bad_slow;
      }
      if (bad) { fail("the model holds negative or NaN slowness values"); bail("model"); }
      c->min_slowness = std::isfinite(mn) ? (float)mn : -1.f;
      c->max_slowness = mx;
      c->pos_slowness = pos;
      c->mean_slowness = cn ? sum / (double)cn : 0.0;
      c->allow_outside_sources = false;
      if (pt.ok && (!sweeptt_set_star(c, fs, starsize) || !sweeptt_set_sources(c, &start, 1))) bail("star / start point");
      if (pt.ok && c->kernel_used != SWEEPTT_KERNEL_TILED) { fail("one grid over several devices needs the tiled kernel (star too wide for its halo)"); bail("kernel"); }
    }
    bar.wait();
    // phase 4: everybody's arrays exist -> exchange the pointers, take the constant tables, reset
    if (pt.ok && !setup_failed) {
      c->mp_nparts = G; c->mp_part = p;
      {
        // per tile column: its owner, and (owned columns) where its staged box starts in the local slowness copy:
        // block lb of this part starts at local plane lb * PB, logical plane x of the block at lb * PB + (x - x0) + 7
        std::vector<int> slow0(g.ntx, -1);
        for (size_t lb = 0; lb < pt.blocks.size(); ++lb)
          for (int t = pt.blocks[lb].first / TX; t * TX < pt.blocks[lb].second; ++t) slow0[t] = (int)lb * PB + (t * TX - pt.blocks[lb].first);
        if (cudaMalloc(&c->d_tx_owner, g.ntx) != cudaSuccess || cudaMalloc(&c->d_tx_slow0, sizeof(int) * g.ntx) != cudaSuccess ||
            cudaMemcpy(c->d_tx_owner, tx_owner.data(), g.ntx, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(c->d_tx_slow0, slow0.data(), sizeof(int) * g.ntx, cudaMemcpyHostToDevice) != cudaSuccess) {
          fail("per-column ownership tables: %s", cudaGetErrorString(cudaGetLastError()));
          bail("tables");
        }
      }
      for (int q = 0; q < G; ++q) {
        c->mp_key[q] = parts[q].ctx->d_key;
        c->mp_tmax[q] = parts[q].ctx->d_tmax;
        c->mp_kmin[q] = &parts[q].ctx->d_state->kmin_pub;
      }
      if (!ready(c, &pt.lease)) bail("ready");
      if (pt.ok) PCK(launch_reset_part(make_args(c), o.max_rounds, c->stream));
      PCK(cudaStreamSynchronize(c->stream));
    }
    bar.wait();
    if (p == 0) t_solve0 = std::chrono::steady_clock::now();
    // phase 5: first work lists, then batches of K rounds until the job is quiescent
    if (pt.ok && !setup_failed) {
      PCK(launch_init_sources(make_args(c), c->stream));
      long long last_visits = 0;
      while (pt.ok) {
        int changed = 0;
        const auto tb0 = std::chrono::steady_clock::now();
        if (!run_rounds(c, false, K, &changed, nullptr)) { pt.ok = 0; pt.err = g_err; quiet.abort(); break; }
        batches[p] += 1;
        const SolveState& h = *c->h_state;
        const bool pending = h.count[h.parity] != 0 || h.kmin_pub != 0x7f800000u;
        const bool worked = (long long)h.tile_visits != last_visits;
        if (worked) busy_ms[p] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tb0).count();
        else idle_batches[p] += 1;
        last_visits = (long long)h.tile_visits;
        if (quiet.report(p, last_visits, !pending && !worked)) break;
        if (o.max_rounds > 0 && h.round >= o.max_rounds) { pt.ok = 0; pt.err = "not converged after max_rounds"; quiet.abort(); break; }
      }
    } else {
      quiet.abort();
    }
    bar.wait();
    if (p == 0) t_solve1 = std::chrono::steady_clock::now();
    // phase 6: gather the owned blocks
    if (pt.ok && !setup_failed && !quiet.failed) {
      float* h_stage = nullptr;
      size_t stage_floats = 0;
      for (auto& b : pt.blocks) {
        int sub[3] = {nx, ny, nz};
        sub[axis] = b.second - b.first;
        stage_floats = std::max(stage_floats, (size_t)sub[0] * sub[1] * sub[2]);
      }
      if (stage_floats && axis != 0 && cudaMallocHost(&h_stage, stage_floats * 4) != cudaSuccess) bail("staging");
      for (auto& b : pt.blocks) {
        if (!pt.ok) break;
        int sub[3] = {nx, ny, nz};
        sub[axis] = b.second - b.first;
        const size_t cnt = (size_t)sub[0] * sub[1] * sub[2];
        BoxGeom gs = g;
        gs.nx = b.second - b.first;
        const long long ds[3] = {(long long)sub[1] * sub[2], (long long)sub[2], 1};
        for (int q = 0; q < 3; ++q) gs.dstride[q] = ds[g.perm[q]];
        PCK(launch_unpad_box(d_tt + (size_t)b.first * g.sx, c->d_stage, gs, c->stream));
        if (axis == 0) {  // planes of the caller's slowest axis are contiguous in the caller's box
          PCK(cudaMemcpyAsync(tt_out + (size_t)b.first * ny * nz, c->d_stage, cnt * 4, cudaMemcpyDeviceToHost, c->stream));
          PCK(cudaStreamSynchronize(c->stream));
        } else {
          PCK(cudaMemcpyAsync(h_stage, c->d_stage, cnt * 4, cudaMemcpyDeviceToHost, c->stream));
          PCK(cudaStreamSynchronize(c->stream));
          for (int x = 0; x < sub[0]; ++x)
            for (int y = 0; y < sub[1]; ++y) {
              const size_t src = ((size_t)x * sub[1] + y) * sub[2];
              if (axis == 1)
                std::memcpy(tt_out + ((size_t)x * ny + (y + b.first)) * nz, h_stage + src, sizeof(float) * sub[2]);
              else
                std::memcpy(tt_out + ((size_t)x * ny + y) * nz + b.first, h_stage + src, sizeof(float) * sub[2]);
            }
        }
      }
      if (h_stage) cudaFreeHost(h_stage);
    }
#undef PCK
  };
  {
    std::vector<std::thread> th;
    for (int p = 0; p < G; ++p) th.emplace_back(part_main, p);
    for (auto& t : th) t.join();
  }
  t_end = std::chrono::steady_clock::now();
  for (int p = 0; p < G; ++p)
    if (!parts[p].ok) {
      const std::string e = parts[p].err;
      cleanup();
      return fail("part %d: %s", p, e.c_str());
    }
  if (setup_failed || quiet.failed) { cleanup(); return fail("one grid over several devices: a part failed"); }

  sweeptt_stats total{};
  total.struct_size = sizeof total;
  for (int p = 0; p < G; ++p) {
    sweeptt_ctx* c = parts[p].ctx;
    cudaSetDevice(parts[p].device);
    read_state(c);
    total.relaxations += (long long)c->h_state->pulls;
    total.tile_visits += (long long)c->h_state->tile_visits;
    total.units_run += (long long)c->h_state->units_run;
    total.units_changed += (long long)c->h_state->units_changed;
    total.rounds = std::max(total.rounds, c->h_state->round);
    total.kernel_launches += 3LL * c->h_state->round;
    total.relax_launches += c->h_state->round;
  }
  auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration<double, std::milli>(b - a).count();
  };
  total.kernel_used = SWEEPTT_KERNEL_TILED;
  total.devices_used = (int)devices.size();
  total.solve_ms = ms(t_solve0, t_solve1);
  total.h2d_ms = ms(t_begin, t_solve0);
  total.d2h_ms = ms(t_solve1, t_end);
  total.h2d_bytes = (long long)nx * ny * nz * 4;
  total.d2h_bytes = (long long)nx * ny * nz * 4;
  if (o.verbose > 0) {
    fprintf(stderr, "[sweeptt] one grid over %d parts (%zu devices), %d blocks of <= %d tiles: set-up %.1f ms, solve %.1f ms, gather %.1f ms; batches per part:",
            G, devices.size(), nblocks, tpb, total.h2d_ms, total.solve_ms, total.d2h_ms);
    for (int p = 0; p < G; ++p) fprintf(stderr, " %lld (%lld without work, %.1f ms in batches with work, %lld tiles)", batches[p], idle_batches[p], busy_ms[p], (long long)parts[p].ctx->h_state->tile_visits);
    fprintf(stderr, "\n");
  }
  if (stats) *stats = total;
  cleanup();
  return 1;
}

extern "C" int sweeptt_solve_slabs(const float* slowness, int nx, int ny, int nz, const struct FS* fs, int starsize,
                                   struct START start, float* tt_out, const sweeptt_opts* opts, sweeptt_stats* stats) {
  if (!slowness) return fail("sweeptt_solve_slabs: null argument");
  auto fetch = [&](const int* org, const int* dims, float* dst) -> int {
    if (org[1] == 0 && org[2] == 0 && dims[1] == ny && dims[2] == nz) {  // whole planes: one contiguous run
      std::memcpy(dst, slowness + (size_t)org[0] * ny * nz, sizeof(float) * (size_t)dims[0] * ny * nz);
      return 1;
    }
    for (int x = 0; x < dims[0]; ++x)
      for (int y = 0; y < dims[1]; ++y)
        std::memcpy(dst + ((size_t)x * dims[1] + y) * dims[2],
                    slowness + ((size_t)(x + org[0]) * ny + (y + org[1])) * nz + org[2], sizeof(float) * dims[2]);
    return 1;
  };
  return solve_slabs_impl(fetch, nx, ny, nz, fs, starsize, start, tt_out, opts, stats);
}

// Each part reads only the planes of its own blocks (+ halo planes) straight from the .vbox file with the subset
// loader (include/velocityboxfiler.h:741 vbfileloadbinarysubset) -- the full model never has to fit
// in host memory at once.
extern "C" int sweeptt_solve_slabs_vbox(const char* vbox_path, const struct FS* fs, int starsize, struct START start,
                                        float* tt_out, const sweeptt_opts* opts, sweeptt_stats* stats) {
  if (!vbox_path) return fail("sweeptt_solve_slabs_vbox: null argument");
  int dims[3];
  if (!sweeptt_vbox_dims(vbox_path, dims)) return 0;
  auto fetch = [&](const int* org, const int* d, float* dst) -> int {
    float* sub = nullptr;
    if (!sweeptt_vbox_load_subset(vbox_path, org, d, &sub)) return 0;
    std::memcpy(dst, sub, sizeof(float) * (size_t)d[0] * d[1] * d[2]);
    sweeptt_free(sub);
    return 1;
  };
  return solve_slabs_impl(fetch, dims[0], dims[1], dims[2], fs, starsize, start, tt_out, opts, stats);
}
