// engine.cu -- plan store, generic convolution engine and the resident
// deconvolution handle (see engine.cuh).
#include "engine.cuh"
#include "fft_generic.cuh"

#include <algorithm>
#include <atomic>
#ifdef _OPENMP
#include <omp.h>
#endif
#include <chrono>
#include <condition_variable>
#include <thread>
#include <cmath>
#include <cstdlib>

namespace lmvn {

// ------------------------------------------------------------------------------
// error / trace plumbing
// ------------------------------------------------------------------------------
static thread_local std::string g_last_error;

void set_last_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  // the reference prints and exits (ref: inc/cuda_helpers.cuh:17-24); we print and return
  fprintf(stderr, "[libmultiviewnative] error: %s\n", buf);
}
const char* last_error() { return g_last_error.c_str(); }
void clear_last_error() { g_last_error.clear(); }

bool trace_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("LMVN_TRACE");
    on = (e && *e && *e != '0') ? 1 : 0;
  }
  return on == 1;
}
void trace(const char* fmt, ...) {
  if (!trace_enabled()) return;
  va_list ap;
  va_start(ap, fmt);
  fprintf(stderr, "[lmvn trace] ");
  vfprintf(stderr, fmt, ap);
  fprintf(stderr, "\n");
  va_end(ap);
}

static std::atomic<int> g_default_strategy{-1};  // process wide; lmvn_set_default_strategy may race with calls on other threads
int default_strategy() {
  int cur = g_default_strategy.load(std::memory_order_relaxed);
  if (cur < 0) {
    const char* e = getenv("LMVN_STRATEGY");
    cur = 0;
    if (e && !strcmp(e, "generic")) cur = 1;
    if (e && !strcmp(e, "fused")) cur = 2;
    int expected = -1;
    g_default_strategy.compare_exchange_strong(expected, cur);
    cur = g_default_strategy.load();
  }
  return cur;
}
void set_default_strategy(int s) { g_default_strategy.store(s); }

// ------------------------------------------------------------------------------
// device selection (ref: inc/cuda_helpers.cuh:116-136)
// ------------------------------------------------------------------------------
int resolve_device(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    set_last_error("no CUDA device available");
    return -1;
  }
  if (device >= n) {
    set_last_error("device %d out of range (have %d)", device, n);
    return -1;
  }
  if (device >= 0) return device;
  int best = 0, best_cc = -1;
  for (int d = 0; d < n; ++d) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, d) != cudaSuccess) continue;
    int cc = p.major * 10 + p.minor;
    if (cc > best_cc) { best_cc = cc; best = d; }
  }
  return best;
}

// ------------------------------------------------------------------------------
// plan store
// ------------------------------------------------------------------------------
static void factorize(int n, gen::AxisPlan& P) {
  P.n = n;
  P.nf = 0;
  int m = n;
  while (m % 4 == 0) { P.factors[P.nf++] = 4; m /= 4; }
  while (m % 2 == 0) { P.factors[P.nf++] = 2; m /= 2; }
  for (int p = 3; p * p <= m; p += 2)
    while (m % p == 0) { P.factors[P.nf++] = p; m /= p; }
  if (m > 1) P.factors[P.nf++] = m;
}

FftPlan::~FftPlan() {
  for (int a = 0; a < 3; ++a)
    if (d_tw[a]) cudaFree(d_tw[a]);
}

static const size_t kMaxSmem = 200 * 1024;

static int build_axis(FftPlan& fp, int a, int n) {
  factorize(n, fp.ax[a]);
  std::vector<cplx> tw(n);
  for (int k = 0; k < n; ++k) {
    const double ang = -2.0 * M_PI * double(k) / double(n);
    tw[k] = cmake(float(cos(ang)), float(sin(ang)));
  }
  LMVN_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&fp.d_tw[a]), sizeof(cplx) * n));
  LMVN_CUDA_TRY(cudaMemcpy(fp.d_tw[a], tw.data(), sizeof(cplx) * n, cudaMemcpyHostToDevice));
  fp.ax[a].tw = fp.d_tw[a];
  int L = 2048 / n;
  if (L < 1) L = 1;
  if (L > 32) L = 32;
  fp.lines[a] = L;
  fp.smem[a] = size_t(2) * n * L * sizeof(cplx);
  if (fp.smem[a] > kMaxSmem) {
    set_last_error("axis length %d exceeds the shared-memory transform limit", n);
    return -1;
  }
  return 0;
}

struct PlanKey {
  int device, nz, ny, nx;
  bool operator<(const PlanKey& o) const {
    if (device != o.device) return device < o.device;
    if (nz != o.nz) return nz < o.nz;
    if (ny != o.ny) return ny < o.ny;
    return nx < o.nx;
  }
};
static std::mutex g_store_mutex;
static std::map<PlanKey, std::shared_ptr<FftPlan>> g_store;

std::shared_ptr<FftPlan> get_fft_plan(int device, int nz, int ny, int nx) {
  std::lock_guard<std::mutex> lock(g_store_mutex);
  PlanKey key{device, nz, ny, nx};
  auto it = g_store.find(key);
  if (it != g_store.end()) return it->second;
  if (cudaSetDevice(device) != cudaSuccess) {
    set_last_error("cudaSetDevice(%d) failed", device);
    return nullptr;
  }
  auto fp = std::make_shared<FftPlan>();
  fp->device = device;
  fp->nz = nz; fp->ny = ny; fp->nx = nx; fp->nxc = nx / 2 + 1;
  const int n[3] = {nz, ny, nx};
  for (int a = 0; a < 3; ++a)
    if (build_axis(*fp, a, n[a]) != 0) return nullptr;
  // the attribute is per (function, device): set it for every device that gets a plan (new plans are rare)
  cudaFuncSetAttribute(gen::k_rows_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kMaxSmem));
  cudaFuncSetAttribute(gen::k_rows_inv, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kMaxSmem));
  cudaFuncSetAttribute(gen::k_cols, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kMaxSmem));
  g_store[key] = fp;
  trace("new fft plan dev=%d dims=%dx%dx%d", device, nz, ny, nx);
  return fp;
}

// ------------------------------------------------------------------------------
// generic engine: five separable passes per convolution
// ------------------------------------------------------------------------------
static const int kGenThreads = 256;

struct GenericEngine : ConvEngine {
  int strategy() const override { return 1; }
  size_t khat_elems() const override { return plan->spec_elems(); }
  size_t work_elems() const override { return plan->spec_elems(); }
  int launches_per_conv() const override { return 5; }
  unsigned long long S() const { return plan->voxels() * sizeof(float); }
  unsigned long long C() const { return plan->spec_elems() * sizeof(cplx); }

  int rows_fwd(const gen::RealSource& src, cplx* spec, cudaStream_t s) {
    const FftPlan& p = *plan;
    const size_t rows = size_t(p.nz) * p.ny;
    dim3 grid(unsigned(ceil_div(rows, p.lines[2])));
    LMVN_LAUNCH(gen::k_rows_fwd, grid, dim3(kGenThreads), p.smem[2], s, src, spec, p.nz, p.ny, p.nx,
                p.ax[2], p.lines[2]);
    LMVN_CUDA_TRY(cudaGetLastError());
    mark("gen_rows_fwd", S() + C(), s);
    return 0;
  }
  int cols(cplx* data, const cplx* khat, int axis, int mode, float scale, cudaStream_t s) {
    const FftPlan& p = *plan;
    long long ostride, jstride, inner;
    unsigned outer;
    if (axis == 1) {  // y
      ostride = (long long)p.ny * p.nxc; jstride = p.nxc; inner = p.nxc; outer = unsigned(p.nz);
    } else {          // z
      ostride = 0; jstride = (long long)p.ny * p.nxc; inner = (long long)p.ny * p.nxc; outer = 1;
    }
    if (outer > 65535u) {
      set_last_error("z extent %u too large for the generic y pass", outer);
      return -1;
    }
    dim3 grid(unsigned(ceil_div(size_t(inner), p.lines[axis])), outer);
    LMVN_LAUNCH(gen::k_cols, grid, dim3(kGenThreads), p.smem[axis], s, data, khat, ostride, jstride,
                inner, p.ax[axis], p.lines[axis], mode, scale);
    LMVN_CUDA_TRY(cudaGetLastError());
    if (mode == gen::COLS_FWD_MUL_INV) mark("gen_cols_z_mul", 3 * C(), s);
    else mark(axis == 1 ? (mode == gen::COLS_FWD ? "gen_cols_y_fwd" : "gen_cols_y_inv") : "gen_cols_z", 2 * C(), s);
    return 0;
  }
  int rows_inv(const cplx* spec, float* out, const gen::Epilogue& ep, cudaStream_t s) {
    const FftPlan& p = *plan;
    const size_t rows = size_t(p.nz) * p.ny;
    dim3 grid(unsigned(ceil_div(rows, p.lines[2])));
    LMVN_LAUNCH(gen::k_rows_inv, grid, dim3(kGenThreads), p.smem[2], s, spec, out, p.nz, p.ny, p.nx,
                p.ax[2], p.lines[2], ep);
    LMVN_CUDA_TRY(cudaGetLastError());
    mark(ep.mode == gen::EPI_UPDATE ? "gen_rows_inv_update" : (ep.mode == gen::EPI_QUOTIENT ? "gen_rows_inv_quotient" : "gen_rows_inv"),
         C() + S() * (ep.mode == gen::EPI_UPDATE ? 3 : (ep.mode == gen::EPI_QUOTIENT ? 2 : 1)), s);
    return 0;
  }

  int kernel_spectrum(const float* d_kernel, const int kd[3], cplx* khat, cplx*, cudaStream_t s) override {
    gen::RealSource src{d_kernel, 1, kd[0], kd[1], kd[2]};
    LMVN_TRY(rows_fwd(src, khat, s));
    LMVN_TRY(cols(khat, nullptr, 1, gen::COLS_FWD, 1.f, s));
    // 1/N folded into K^ (decision q10; the reference scales after the c2r,
    // ref: inc/cpu_convolve.h:271-278)
    const float inv_n = float(1.0 / double(plan->voxels()));
    LMVN_TRY(cols(khat, nullptr, 0, gen::COLS_FWD, inv_n, s));
    return 0;
  }
  int convolve(const float* in, cplx* work, const cplx* khat, const gen::Epilogue& ep, float* out,
               cudaStream_t s) override {
    gen::RealSource src{in, 0, 0, 0, 0};
    LMVN_TRY(rows_fwd(src, work, s));
    LMVN_TRY(cols(work, nullptr, 1, gen::COLS_FWD, 1.f, s));
    LMVN_TRY(cols(work, khat, 0, gen::COLS_FWD_MUL_INV, 1.f, s));
    LMVN_TRY(cols(work, nullptr, 1, gen::COLS_INV, 1.f, s));
    LMVN_TRY(rows_inv(work, out, ep, s));
    return 0;
  }
};

std::unique_ptr<ConvEngine> make_generic_engine(std::shared_ptr<FftPlan> plan) {
  std::unique_ptr<GenericEngine> e(new GenericEngine());
  e->plan = plan;
  return std::unique_ptr<ConvEngine>(e.release());
}

#ifndef LMVN_HAVE_FUSED
std::unique_ptr<ConvEngine> make_fused_engine(std::shared_ptr<FftPlan>) { return nullptr; }
#endif

// ------------------------------------------------------------------------------
// resident deconvolution handle
// ------------------------------------------------------------------------------
static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Parked arenas (at most two per device).  Fiji calls inplace_gpu_deconvolve once per block with identical
// shapes (ref: bench/bench_gpu_deconvolve.cu:48-49); returning several GiB to the driver and asking
// for them again costs tens to hundreds of milliseconds per call (fresh pages are scrubbed).  A
// destroyed handle parks its arena here, the next handle on that device takes one that is large
// enough.  Two slots: the block pipeline (libmultiviewnative_b200/blocks.py) keeps two calls in flight per
// device so that the uploads of block b+1 overlap the loop of block b.  What stays allocated between calls
// is bounded: LMVN_CACHE_ARENA_MAX_MB per device (default: a quarter of the device's memory; anything
// larger goes straight back to the driver), lmvn_release_cached_memory() / LMVN_CACHE_ARENA=0 give
// everything back (a host application that shares the GPU with other libraries should call it when idle).
namespace {
struct ParkedArena { unsigned char* p = nullptr; size_t bytes = 0; };
static const int kParkSlots = 2;
std::mutex g_arena_mu;
std::map<int, std::vector<ParkedArena>> g_parked;
bool arena_cache_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("LMVN_CACHE_ARENA");
    v = (e && *e == '0') ? 0 : 1;
  }
  return v == 1;
}
size_t arena_cache_cap(int device) {
  if (const char* e = getenv("LMVN_CACHE_ARENA_MAX_MB")) return size_t(std::max(0.0, atof(e)) * 1048576.0);
  size_t free_b = 0, total_b = 0;
  (void)device;  // the caller has made `device` current
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { (void)cudaGetLastError(); return size_t(16) << 30; }
  return total_b / 4;
}
unsigned char* take_parked(int device, size_t bytes, size_t* capacity) {
  std::lock_guard<std::mutex> lk(g_arena_mu);
  auto it = g_parked.find(device);
  if (it == g_parked.end()) return nullptr;
  std::vector<ParkedArena>& v = it->second;
  // best fit among the parked arenas; wastefully large ones (> 1.5 x + 64 MiB) are not used for this request
  int best = -1;
  for (int i = 0; i < int(v.size()); ++i)
    if (v[i].bytes >= bytes && v[i].bytes <= bytes + bytes / 2 + (size_t(64) << 20) && (best < 0 || v[i].bytes < v[best].bytes))
      best = i;
  if (best < 0) {
    // nothing fits: the request will allocate; make room by returning what is parked
    for (auto& a : v) cudaFree(a.p);
    v.clear();
    return nullptr;
  }
  unsigned char* p = v[best].p;
  *capacity = v[best].bytes;
  v.erase(v.begin() + best);
  return p;
}
void park(int device, unsigned char* p, size_t bytes) {
  if (!arena_cache_enabled()) { cudaFree(p); return; }
  const size_t cap = arena_cache_cap(device);
  std::lock_guard<std::mutex> lk(g_arena_mu);
  std::vector<ParkedArena>& v = g_parked[device];
  size_t held = 0;
  for (auto& a : v) held += a.bytes;
  while (!v.empty() && (int(v.size()) >= kParkSlots || held + bytes > cap)) {  // oldest first
    held -= v.front().bytes;
    cudaFree(v.front().p);
    v.erase(v.begin());
  }
  if (bytes > cap) { cudaFree(p); return; }
  v.push_back(ParkedArena{p, bytes});
}
}  // namespace

namespace {
void release_stagers();  // pinned staging rings (below)
}

void release_cached_memory() {
  release_stagers();
  std::lock_guard<std::mutex> lk(g_arena_mu);
  for (auto& kv : g_parked) {
    cudaSetDevice(kv.first);
    for (auto& a : kv.second) cudaFree(a.p);
  }
  g_parked.clear();
}

int debug_fill_parked_arenas(int byte) {
  int prev = 0;
  LMVN_CUDA_TRY(cudaGetDevice(&prev));
  std::lock_guard<std::mutex> lk(g_arena_mu);
  for (auto& kv : g_parked) {
    LMVN_CUDA_TRY(cudaSetDevice(kv.first));
    for (auto& a : kv.second) LMVN_CUDA_TRY(cudaMemset(a.p, byte, a.bytes));
    LMVN_CUDA_TRY(cudaDeviceSynchronize());
  }
  LMVN_CUDA_TRY(cudaSetDevice(prev));
  return 0;
}

Deconv::~Deconv() {
  if (arena || stream) cudaSetDevice(device);
  if (stream) cudaStreamSynchronize(stream);
  if (ev0) cudaEventDestroy(ev0);
  if (ev1) cudaEventDestroy(ev1);
#ifndef LMVN_EMU
  if (sweep_graph) cudaGraphExecDestroy(sweep_graph);
#endif
  if (stream) cudaStreamDestroy(stream);
  if (arena) {
    arena_unpoison(arena, arena_capacity);
    park(device, arena, arena_capacity);
  }
}

static const size_t kMaxKernelVoxels = size_t(1) << 24;

int Deconv::init(const int* d, int nviews, int dev, int strategy) {
  NvtxRange nvtx_("lmvn::plan_create");
  if (!d || d[0] <= 0 || d[1] <= 0 || d[2] <= 0) {
    set_last_error("invalid image dims");
    return -1;
  }
  if (nviews <= 0 || nviews > 65535) {
    set_last_error("invalid number of views %d", nviews);
    return -1;
  }
  const auto t_begin = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (trace_enabled())
      trace("  init %-18s +%.2f ms", what,
            std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count());
  };
  device = resolve_device(dev);
  if (device < 0) return -1;
  LMVN_CUDA_TRY(cudaSetDevice(device));
  dims[0] = d[0]; dims[1] = d[1]; dims[2] = d[2];
  num_views = nviews;
  lap("device");
  auto fp = get_fft_plan(device, d[0], d[1], d[2]);
  if (!fp) return -1;
  lap("fft plan");
  if (strategy == 0) strategy = default_strategy();
  if (strategy == 0 || strategy == 2) {
    engine = make_fused_engine(fp);
    if (!engine && strategy == 2) {
      set_last_error("fused strategy not available for dims %dx%dx%d", d[0], d[1], d[2]);
      return -1;
    }
  }
  if (!engine) engine = make_generic_engine(fp);
  lap("engine");

  const size_t S = align_up(fp->voxels() * sizeof(float), 256);
  const size_t K = align_up(engine->khat_elems() * sizeof(cplx), 256);
  const size_t W = align_up(engine->work_elems() * sizeof(cplx), 256);
  kernel_stage_elems = std::min(kMaxKernelVoxels, fp->voxels());
  const size_t KS = align_up(kernel_stage_elems * sizeof(float), 256);
  // `integral` is sized like a spectrum buffer: the chained loop of an embedded plan never stores the quotient
  // and uses it as its second spectrum buffer
  const size_t SI = std::max(S, W);
  arena_bytes = 3 * SI + W + KS + size_t(nviews) * (2 * S + 2 * K) + kArenaRedzone * (5 + 4 * size_t(nviews));
  arena = take_parked(device, arena_bytes, &arena_capacity);
  if (!arena) {
    size_t free_b = 0, total_b = 0;
    LMVN_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    if (arena_bytes > free_b) {
      // ref: src/multiviewnative.cu:138-141 prints and returns with psi untouched
      set_last_error("deconvolution of %dx%dx%d with %d views needs %.2f GiB of device memory, %.2f GiB free",
                     d[0], d[1], d[2], nviews, arena_bytes / 1073741824.0, free_b / 1073741824.0);
      return -1;
    }
    LMVN_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&arena), arena_bytes));
    arena_capacity = arena_bytes;
  }
  lap("arena");
  unsigned char* p = arena;
  arena_unpoison(arena, arena_capacity);
  auto take = [&](size_t bytes) {
    unsigned char* r = p;
    p += bytes;
    arena_poison(p, kArenaRedzone);
    p += kArenaRedzone;
    return r;
  };
  psi = reinterpret_cast<float*>(take(SI));   // psi, psi2 and integral can change roles (lmvn_plan_convolve swaps
  psi2 = reinterpret_cast<float*>(take(SI));  // psi and integral): all three have the spectrum-buffer size
  integral = reinterpret_cast<float*>(take(SI));
  work = reinterpret_cast<cplx*>(take(W));
  kernel_stage = reinterpret_cast<float*>(take(KS));
  image.resize(nviews); weights.resize(nviews); khat1.resize(nviews); khat2.resize(nviews);
  view_set.assign(nviews, 0);
  for (int v = 0; v < nviews; ++v) {
    image[v] = reinterpret_cast<float*>(take(S));
    weights[v] = reinterpret_cast<float*>(take(S));
    khat1[v] = reinterpret_cast<cplx*>(take(K));
    khat2[v] = reinterpret_cast<cplx*>(take(K));
  }
  if (const char* e = getenv("LMVN_GRAPH")) use_graph = (*e != '0');
  LMVN_CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  LMVN_CUDA_TRY(cudaEventCreate(&ev0));
  LMVN_CUDA_TRY(cudaEventCreate(&ev1));
  lap("stream+events");
  trace("deconv handle dev=%d dims=%dx%dx%d views=%d strategy=%d arena=%.1f MiB", device, d[0], d[1],
        d[2], nviews, engine->strategy(), arena_bytes / 1048576.0);
  return 0;
}

static int check_kernel_dims(const int* kd, const int* dims, const char* what) {
  if (!kd) {
    set_last_error("%s dims missing", what);
    return -1;
  }
  for (int a = 0; a < 3; ++a) {
    if (kd[a] <= 0 || kd[a] > dims[a]) {
      // undefined in the reference (wraps into a too-small target,
      // ref: inc/padd_utils.h:19-38); rejected here, decision q11
      set_last_error("%s extent %d along axis %d does not fit the image extent %d", what, kd[a], a, dims[a]);
      return -1;
    }
  }
  return 0;
}

int Deconv::set_logical(const int* image_dims, const int* off) {
  for (int a = 0; a < 3; ++a) {
    if (image_dims[a] <= 0 || off[a] < 0 || image_dims[a] + off[a] > dims[a]) {
      set_last_error("zero-padded plan: image extent %d at offset %d does not fit the padded extent %d (axis %d)",
                     image_dims[a], off[a], dims[a], a);
      return -1;
    }
    logical[a] = image_dims[a];
    offset[a] = off[a];
  }
  padded = (logical[0] != dims[0] || logical[1] != dims[1] || logical[2] != dims[2]);
  return 0;
}

int Deconv::wrap_exterior(float* vol) {
  // exterior rows read interior rows only and interior rows only write their own x margins: no ordering hazard
  LMVN_LAUNCH(k_wrap_exterior, dim3(unsigned(dims[1]), unsigned(dims[0])), dim3(128), 0, stream, vol, dims[0], dims[1], dims[2],
              logical[0], logical[1], logical[2], offset[0], offset[1], offset[2]);
  LMVN_CUDA_TRY(cudaGetLastError());
  return 0;
}

// host stack (logical extents) -> device volume (plan extents), zero filled around it
// ---------------------------------------------------------------------------------
// Host staging for PAGEABLE caller buffers.  Fiji hands the library JNA / malloc'ed memory (ref:
// src/multiviewnative.cu:66); a cudaMemcpyAsync from such memory is staged by the driver on one thread at a
// fraction of the PCIe rate.  Here: a small ring of pinned chunks per device, filled by several host threads
// while the DMA of the previous chunk runs.  Pinned or registered buffers (cudaPointerGetAttributes) and small
// copies take the direct path.  LMVN_STAGED_COPY=0 disables.
// ---------------------------------------------------------------------------------
namespace {
#ifndef LMVN_EMU
// Host threads that move pageable caller memory into / out of the pinned staging ring.  A persistent pool that SLEEPS
// between copies: an OpenMP team per copy spin-waits after every parallel region, and with one process per GPU that
// meant 8 ranks x 8 spinning threads on a 32-core host (8 x B200 box: the staged upload of config 3 took 1.3 s per call
// instead of 0.4 s, profiles/r02_bench_8gpu_before_copy_pool.json).  Size: LMVN_STAGING_THREADS, else the machine's hardware
// threads divided by the number of visible GPUs (every GPU usually has its own process doing the same), 1 .. 8.
class CopyPool {
 public:
  explicit CopyPool(int n) {
    for (int i = 0; i < n; ++i) workers_.emplace_back([this] { run(); });
  }
  ~CopyPool() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      stop_ = true;
    }
    cv_.notify_all();
    for (auto& t : workers_) t.join();
  }
  void copy(void* dst, const void* src, size_t bytes) {
    static const size_t kPiece = size_t(1) << 20;
    const size_t pieces = (bytes + kPiece - 1) / kPiece;
    if (workers_.empty() || pieces < 2) { std::memcpy(dst, src, bytes); return; }
    std::unique_lock<std::mutex> job(job_mu_);  // one copy at a time through the pool
    {
      std::unique_lock<std::mutex> lk(mu_);
      done_cv_.wait(lk, [this] { return active_ == 0; });  // no straggler of the previous job is still looking at its fields
      dst_ = static_cast<unsigned char*>(dst);
      src_ = static_cast<const unsigned char*>(src);
      bytes_ = bytes;
      pieces_ = pieces;
      next_.store(0);
      left_ = pieces;
      ++generation_;
      hint_.store(generation_, std::memory_order_release);
    }
    cv_.notify_all();
    work(kPiece);  // the calling thread copies too
    std::unique_lock<std::mutex> lk(mu_);
    done_cv_.wait(lk, [this] { return left_ == 0 && active_ == 0; });
  }

 private:
  void work(size_t piece) {
    size_t mine = 0;
    for (;;) {
      const size_t i = next_.fetch_add(1);
      if (i >= pieces_) break;
      const size_t off = i * piece;
      std::memcpy(dst_ + off, src_ + off, std::min(piece, bytes_ - off));
      ++mine;
    }
    if (mine) {
      std::lock_guard<std::mutex> lk(mu_);
      left_ -= mine;
      if (left_ == 0) done_cv_.notify_all();
    }
  }
  void run() {
    unsigned long long seen = 0;
    for (;;) {
      // a stack is uploaded as a train of 16 MiB chunks a few hundred microseconds apart: poll for the next chunk for
      // a short while before going to sleep (a futex wake-up per worker and chunk cost ~15 % of the upload rate)
      const auto t0 = std::chrono::steady_clock::now();
      while (hint_.load(std::memory_order_acquire) == seen &&
             std::chrono::steady_clock::now() - t0 < std::chrono::microseconds(300)) {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
      }
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return stop_ || generation_ != seen; });
        if (stop_) return;
        seen = generation_;
        ++active_;  // the job's fields stay as they are while any worker is inside work()
      }
      work(size_t(1) << 20);
      {
        std::lock_guard<std::mutex> lk(mu_);
        if (--active_ == 0) done_cv_.notify_all();
      }
    }
  }
  std::vector<std::thread> workers_;
  std::mutex mu_, job_mu_;
  std::condition_variable cv_, done_cv_;
  unsigned char* dst_ = nullptr;
  const unsigned char* src_ = nullptr;
  size_t bytes_ = 0, pieces_ = 0, left_ = 0;
  int active_ = 0;
  std::atomic<size_t> next_{0};
  std::atomic<unsigned long long> hint_{0};  // copy of generation_ the workers may poll without the lock
  unsigned long long generation_ = 0;
  bool stop_ = false;
};
CopyPool& copy_pool() {
  static CopyPool* pool = [] {
    int threads = 0;
    if (const char* e = getenv("LMVN_STAGING_THREADS")) threads = atoi(e);
    if (threads <= 0) {
      int gpus = 1;
      if (cudaGetDeviceCount(&gpus) != cudaSuccess || gpus < 1) { (void)cudaGetLastError(); gpus = 1; }
      const int hw = int(std::thread::hardware_concurrency());
      threads = std::max(1, std::min(8, (hw > 0 ? hw : 8) / gpus));
    }
    return new CopyPool(threads - 1);  // + the calling thread; lives as long as the process
  }();
  return *pool;
}

struct HostStager {
  static const size_t kChunk = size_t(16) << 20;
  static const int kSlots = 3;
  std::mutex mu;
  unsigned char* pinned[kSlots] = {nullptr, nullptr, nullptr};
  cudaEvent_t done[kSlots] = {nullptr, nullptr, nullptr};
  bool inflight[kSlots] = {false, false, false};  // the slot's last DMA may still be running (any stream of the device)
  bool ready = false, failed = false;

  int wait_slot(int slot) {
    if (inflight[slot]) {
      LMVN_CUDA_TRY(cudaEventSynchronize(done[slot]));
      inflight[slot] = false;
    }
    return 0;
  }
  void release() {
    std::lock_guard<std::mutex> lk(mu);
    for (int i = 0; i < kSlots; ++i) {
      if (inflight[i]) cudaEventSynchronize(done[i]);
      inflight[i] = false;
      if (pinned[i]) cudaFreeHost(pinned[i]);
      if (done[i]) cudaEventDestroy(done[i]);
      pinned[i] = nullptr;
      done[i] = nullptr;
    }
    ready = false;
  }
  int init() {
    if (ready) return 0;
    if (failed) return -1;
    for (int i = 0; i < kSlots; ++i) {
      if (cudaHostAlloc(reinterpret_cast<void**>(&pinned[i]), kChunk, cudaHostAllocDefault) != cudaSuccess ||
          cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming) != cudaSuccess) {
        (void)cudaGetLastError();
        failed = true;
        return -1;
      }
    }
    ready = true;
    return 0;
  }
  // LMVN_STAGING_IMPL = pool | omp.  Default: the sleeping pool when the box has several GPUs (one process per GPU doing
  // the same: spinning OpenMP teams oversubscribe the host), an OpenMP team otherwise (lowest wake-up latency).
  static bool use_pool() {
    static int v = -1;
    if (v < 0) {
      const char* e = getenv("LMVN_STAGING_IMPL");
      if (e && e[0] == 'o') v = 0;
      else if (e && e[0] == 'p') v = 1;
      else {
        int gpus = 1;
        if (cudaGetDeviceCount(&gpus) != cudaSuccess) { (void)cudaGetLastError(); gpus = 1; }
        v = gpus > 1 ? 1 : 0;
      }
    }
    return v == 1;
  }
  static void parallel_copy(void* dst, const void* src, size_t bytes) {
    if (use_pool()) { copy_pool().copy(dst, src, bytes); return; }
    const size_t piece = size_t(1) << 20;
    const long long pieces = (long long)((bytes + piece - 1) / piece);
    int threads = 1;
#ifdef _OPENMP
    // the machine's cores, not omp_get_max_threads(): launchers such as torchrun export OMP_NUM_THREADS=1
    threads = std::max(1, std::min(8, omp_get_num_procs()));
    if (const char* e = getenv("LMVN_STAGING_THREADS")) threads = std::max(1, atoi(e));
#endif
#pragma omp parallel for num_threads(threads) schedule(static)
    for (long long i = 0; i < pieces; ++i) {
      const size_t off = size_t(i) * piece;
      std::memcpy(static_cast<unsigned char*>(dst) + off, static_cast<const unsigned char*>(src) + off,
                  std::min(piece, bytes - off));
    }
  }
  // host -> device, stream ordered on s; returns when src_h has been read completely (like a pageable cudaMemcpyAsync)
  int upload(void* dst_d, const void* src_h, size_t bytes, cudaStream_t s) {
    std::lock_guard<std::mutex> lk(mu);
    LMVN_TRY(init());
    size_t off = 0;
    for (int i = 0; off < bytes; ++i, off += kChunk) {
      const int slot = i % kSlots;
      const size_t len = std::min(kChunk, bytes - off);
      LMVN_TRY(wait_slot(slot));
      parallel_copy(pinned[slot], static_cast<const unsigned char*>(src_h) + off, len);
      LMVN_CUDA_TRY(cudaMemcpyAsync(static_cast<unsigned char*>(dst_d) + off, pinned[slot], len, cudaMemcpyHostToDevice, s));
      LMVN_CUDA_TRY(cudaEventRecord(done[slot], s));
      inflight[slot] = true;
    }
    return 0;
  }
  // device -> host; returns when dst_h is complete
  int download(void* dst_h, const void* src_d, size_t bytes, cudaStream_t s) {
    std::lock_guard<std::mutex> lk(mu);
    LMVN_TRY(init());
    const long long chunks = (long long)((bytes + kChunk - 1) / kChunk);
    auto issue = [&](long long i) -> int {
      const size_t off = size_t(i) * kChunk;
      LMVN_TRY(wait_slot(int(i % kSlots)));
      LMVN_CUDA_TRY(cudaMemcpyAsync(pinned[i % kSlots], static_cast<const unsigned char*>(src_d) + off,
                                    std::min(kChunk, bytes - off), cudaMemcpyDeviceToHost, s));
      LMVN_CUDA_TRY(cudaEventRecord(done[i % kSlots], s));
      inflight[i % kSlots] = true;
      return 0;
    };
    for (long long i = 0; i < std::min<long long>(chunks, kSlots - 1); ++i) LMVN_TRY(issue(i));
    for (long long i = 0; i < chunks; ++i) {
      if (i + kSlots - 1 < chunks) LMVN_TRY(issue(i + kSlots - 1));  // keep the DMA engine ahead of the host copy
      LMVN_TRY(wait_slot(int(i % kSlots)));
      const size_t off = size_t(i) * kChunk;
      parallel_copy(static_cast<unsigned char*>(dst_h) + off, pinned[i % kSlots], std::min(kChunk, bytes - off));
    }
    return 0;
  }
};

std::mutex g_stager_mu;
std::map<int, HostStager*> g_stagers;  // per device, lives as long as the process (pinned memory is expensive to get)

bool staged_copy_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("LMVN_STAGED_COPY");
    v = (e && *e == '0') ? 0 : 1;
  }
  return v == 1;
}

// the stager of `device` when `host_ptr` is pageable and the copy is large enough to pay for it
HostStager* stager_for(int device, const void* host_ptr, size_t bytes) {
  if (bytes < (size_t(4) << 20) || !staged_copy_enabled()) return nullptr;
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, host_ptr) != cudaSuccess) {
    (void)cudaGetLastError();
    return nullptr;
  }
  if (attr.type != cudaMemoryTypeUnregistered) return nullptr;  // pinned / registered / managed: direct copy
  std::lock_guard<std::mutex> lk(g_stager_mu);
  HostStager*& st = g_stagers[device];
  if (!st) st = new HostStager();
  return st->failed ? nullptr : st;
}

void release_stagers() {
  std::lock_guard<std::mutex> lk(g_stager_mu);
  for (auto& kv : g_stagers)
    if (kv.second) {
      cudaSetDevice(kv.first);
      kv.second->release();
    }
}

#else   // host emulation: plain copies
void release_stagers() {}
#endif
}  // namespace

// host <-> device copies of whole stacks on stream s: pageable host memory goes through the staging ring
int copy_to_device(int device, void* dst_d, const void* src_h, size_t bytes, cudaStream_t s) {
#ifndef LMVN_EMU
  if (HostStager* st = stager_for(device, src_h, bytes)) {
    if (st->upload(dst_d, src_h, bytes, s) == 0) return 0;
    if (!st->failed) return -1;  // a copy failed: the error is set
  }
#else
  (void)device;
#endif
  LMVN_CUDA_TRY(cudaMemcpyAsync(dst_d, src_h, bytes, cudaMemcpyHostToDevice, s));
  return 0;
}

// returns when dst_h is complete if the copy was staged; otherwise it is stream ordered like cudaMemcpyAsync
int copy_to_host(int device, void* dst_h, const void* src_d, size_t bytes, cudaStream_t s) {
#ifndef LMVN_EMU
  if (HostStager* st = stager_for(device, dst_h, bytes)) {
    if (st->download(dst_h, src_d, bytes, s) == 0) return 0;
    if (!st->failed) return -1;
  }
#else
  (void)device;
#endif
  LMVN_CUDA_TRY(cudaMemcpyAsync(dst_h, src_d, bytes, cudaMemcpyDeviceToHost, s));
  return 0;
}


int Deconv::upload_stack(float* dst, const float* src_h) {
  const size_t n = engine->plan->voxels();
  if (!padded) {
    LMVN_TRY(copy_to_device(device, dst, src_h, n * sizeof(float), stream));
    return 0;
  }
  // one contiguous copy into the (idle) spectrum work buffer, then a kernel places the box and zero fills the rest
  (void)n;
  float* stage = reinterpret_cast<float*>(work);
  const size_t ln = size_t(logical[0]) * logical[1] * logical[2];
  LMVN_TRY(copy_to_device(device, stage, src_h, ln * sizeof(float), stream));
  LMVN_LAUNCH(k_place_box, dim3(unsigned(dims[1]), unsigned(dims[0])), dim3(128), 0, stream, dst, stage, dims[1], dims[2],
              logical[0], logical[1], logical[2], offset[0], offset[1], offset[2]);
  LMVN_CUDA_TRY(cudaGetLastError());
  return 0;
}

int Deconv::download_stack(float* dst_h, const float* src) {
  if (!padded) {
    LMVN_TRY(copy_to_host(device, dst_h, src, engine->plan->voxels() * sizeof(float), stream));
    return 0;
  }
  float* stage = reinterpret_cast<float*>(work);
  LMVN_LAUNCH(k_gather_box, dim3(unsigned(logical[1]), unsigned(logical[0])), dim3(128), 0, stream, src, stage, dims[1], dims[2],
              logical[1], logical[2], offset[0], offset[1], offset[2]);
  LMVN_CUDA_TRY(cudaGetLastError());
  LMVN_TRY(copy_to_host(device, dst_h, stage, size_t(logical[0]) * logical[1] * logical[2] * sizeof(float), stream));
  return 0;
}

int Deconv::set_view(int v, const float* image_h, const float* weights_h, const float* k1, const int* k1d,
                     const float* k2, const int* k2d) {
  NvtxRange nvtx_("lmvn::set_view (upload + PSF spectra)");
  if (v < 0 || v >= num_views) {
    set_last_error("view index %d out of range", v);
    return -1;
  }
  if (!image_h || !weights_h || !k1 || !k2) {
    set_last_error("null buffer for view %d", v);
    return -1;
  }
  LMVN_TRY(check_kernel_dims(k1d, dims, "kernel1"));
  LMVN_TRY(check_kernel_dims(k2d, dims, "kernel2"));
  LMVN_CUDA_TRY(cudaSetDevice(device));
  LMVN_TRY(upload_stack(image[v], image_h));
  LMVN_TRY(upload_stack(weights[v], weights_h));
  const float* ks[2] = {k1, k2};
  const int* kds[2] = {k1d, k2d};
  cplx* dst[2] = {khat1[v], khat2[v]};
  for (int i = 0; i < 2; ++i) {
    const size_t kn = size_t(kds[i][0]) * kds[i][1] * kds[i][2];
    if (kn > kernel_stage_elems) {
      set_last_error("kernel too large for the staging buffer");
      return -1;
    }
    LMVN_CUDA_TRY(cudaMemcpyAsync(kernel_stage, ks[i], kn * sizeof(float), cudaMemcpyHostToDevice, stream));
    LMVN_TRY(engine->kernel_spectrum(kernel_stage, kds[i], dst[i], work, stream));
    // kernel_stage is reused by the next upload: pageable H2D copies are staged
    // synchronously by the runtime, stream order keeps the device side safe
  }
  view_set[v] = 1;
  return 0;
}

int Deconv::set_psi(const float* psi_h) {
  NvtxRange nvtx_("lmvn::set_psi (upload)");
  if (!psi_h) {
    set_last_error("psi is null");
    return -1;
  }
  LMVN_CUDA_TRY(cudaSetDevice(device));
  LMVN_TRY(upload_stack(psi, psi_h));
  psi_set = true;
  return 0;
}

int Deconv::get_psi(float* psi_h) {
  NvtxRange nvtx_("lmvn::get_psi (download)");
  if (!psi_h) {
    set_last_error("psi is null");
    return -1;
  }
  LMVN_CUDA_TRY(cudaSetDevice(device));
  LMVN_TRY(download_stack(psi_h, psi));
  LMVN_CUDA_TRY(cudaStreamSynchronize(stream));
  return 0;
}

int Deconv::synchronize() {
  LMVN_CUDA_TRY(cudaSetDevice(device));
  LMVN_CUDA_TRY(cudaStreamSynchronize(stream));
  return 0;
}

int Deconv::iterate(int iterations, double lambda, float min_value, float* device_ms) {
  NvtxRange nvtx_("lmvn::iterate (RL loop)");
  if (!psi_set) {
    set_last_error("psi has not been set");
    return -1;
  }
  for (int v = 0; v < num_views; ++v)
    if (!view_set[v]) {
      set_last_error("view %d has not been set", v);
      return -1;
    }
  LMVN_CUDA_TRY(cudaSetDevice(device));
  const UpdateParams up = make_update_params(lambda, min_value);
  LMVN_CUDA_TRY(cudaEventRecord(ev0, stream));
  if (periodic && engine->can_chain_embedded() && iterations > 0) {
    // periodic embedding, chained: the link kernel itself continues the stack periodically (rows outside the box
    // recompute the interior row they alias and write to the other spectrum buffer), no refill pass in the loop
    LMVN_TRY(wrap_exterior(psi));
    LMVN_TRY(engine->chain_begin(psi, work, stream));
    cplx* cur = work;
    cplx* other = reinterpret_cast<cplx*>(integral);  // the quotient is never stored in this loop
    for (int it = 0; it < iterations; ++it) {
      for (int v = 0; v < num_views; ++v) {
        const bool last = (it == iterations - 1 && v == num_views - 1);
        LMVN_TRY(engine->chain_middle(cur, khat1[v], stream));
        gen::Epilogue e1{gen::EPI_QUOTIENT, 1.f, image[v], nullptr, nullptr, up};
        LMVN_TRY(engine->chain_link_embedded(cur, other, e1, nullptr, logical, offset, stream));
        std::swap(cur, other);
        LMVN_TRY(engine->chain_middle(cur, khat2[v], stream));
        gen::Epilogue e2{gen::EPI_UPDATE, 1.f, nullptr, psi, weights[v], up};
        if (last) {
          LMVN_TRY(engine->chain_end(cur, e2, psi, stream));
        } else {
          LMVN_TRY(engine->chain_link_embedded(cur, other, e2, psi2, logical, offset, stream));
          std::swap(cur, other);
          std::swap(psi, psi2);  // the interior of psi2 now holds the new estimate; the exterior is never read
        }
      }
    }
  } else if (periodic) {
    // periodic embedding: both inputs of a step get their exterior refilled; the convolutions are the plain five-pass form
    for (int it = 0; it < iterations; ++it) {
      for (int v = 0; v < num_views; ++v) {
        LMVN_TRY(wrap_exterior(psi));
        gen::Epilogue e1{gen::EPI_QUOTIENT, 1.f, image[v], nullptr, nullptr, up};
        LMVN_TRY(engine->convolve(psi, work, khat1[v], e1, integral, stream));
        LMVN_TRY(wrap_exterior(integral));
        gen::Epilogue e2{gen::EPI_UPDATE, 1.f, nullptr, psi, weights[v], up};
        LMVN_TRY(engine->convolve(integral, work, khat2[v], e2, psi, stream));
      }
    }
  } else if (engine->can_chain() && iterations > 0) {
    const int zero_guard = padded ? 1 : 0;  // zero-padded stacks: see Epilogue::zero_view_guard
    // chained loop: every x-inverse pass also runs the x-forward pass of the convolution that follows it
    auto sweep = [&](bool ends_call) -> int {  // one iteration = one sweep over all views
      for (int v = 0; v < num_views; ++v) {
        LMVN_TRY(engine->chain_middle(work, khat1[v], stream));
        // (view_v / (psi (*) kernel1_v)) stays on chip and is transformed again   ref: src/multiviewnative.cpp:195-205
        gen::Epilogue e1{gen::EPI_QUOTIENT, 1.f, image[v], nullptr, nullptr, up, zero_guard};
        LMVN_TRY(engine->chain_link(work, e1, stream));
        LMVN_TRY(engine->chain_middle(work, khat2[v], stream));
        // psi = update(psi, ., weights_v); the new psi is stored AND transformed for the next view   ref: :209-227
        gen::Epilogue e2{gen::EPI_UPDATE, 1.f, nullptr, psi, weights[v], up};
        if (ends_call && v == num_views - 1) LMVN_TRY(engine->chain_end(work, e2, psi, stream));
        else LMVN_TRY(engine->chain_link(work, e2, stream));
      }
      return 0;
    };
    LMVN_TRY(engine->chain_begin(psi, work, stream));
    int done = 0;
#ifndef LMVN_EMU
    // All sweeps but the last are identical launch sequences: capture one into a CUDA graph and replay it
    // (the launch-bound inner loop of small volumes; ~1.5 % on config 3).  Re-captured when the update parameters change.
    if (use_graph && iterations > 2) {
      if (!sweep_graph || graph_lambda != lambda || graph_min != min_value || graph_psi != psi) {
        if (sweep_graph) { cudaGraphExecDestroy(sweep_graph); sweep_graph = nullptr; }
        cudaGraph_t g = nullptr;
        // a failing capture is treated like every other graph failure: plain launches from now on
        const cudaError_t be = cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal);
        const int rc = (be == cudaSuccess) ? sweep(false) : -1;
        const cudaError_t ce = (be == cudaSuccess) ? cudaStreamEndCapture(stream, &g) : be;
        if (rc != 0 || ce != cudaSuccess || !g) {
          if (g) cudaGraphDestroy(g);
          (void)cudaGetLastError();
          use_graph = false;  // fall back to plain launches for the lifetime of the handle
        } else {
          const cudaError_t ie = cudaGraphInstantiate(&sweep_graph, g, 0);
          cudaGraphDestroy(g);
          if (ie != cudaSuccess) { sweep_graph = nullptr; use_graph = false; (void)cudaGetLastError(); }
          graph_lambda = lambda;
          graph_min = min_value;
          graph_psi = psi;  // lmvn_plan_convolve swaps psi and integral
        }
      }
      if (sweep_graph)
        for (; done < iterations - 1; ++done) LMVN_CUDA_TRY(cudaGraphLaunch(sweep_graph, stream));
    }
#endif
    for (; done < iterations; ++done) LMVN_TRY(sweep(done == iterations - 1));
  } else {
    for (int it = 0; it < iterations; ++it) {
      for (int v = 0; v < num_views; ++v) {
        // integral = view_v / (psi (*) kernel1_v)      ref: src/multiviewnative.cpp:195-205
        gen::Epilogue e1{gen::EPI_QUOTIENT, 1.f, image[v], nullptr, nullptr, up, padded ? 1 : 0};
        LMVN_TRY(engine->convolve(psi, work, khat1[v], e1, integral, stream));
        // psi = update(psi, integral (*) kernel2_v, weights_v)   ref: :209-227
        gen::Epilogue e2{gen::EPI_UPDATE, 1.f, nullptr, psi, weights[v], up};
        LMVN_TRY(engine->convolve(integral, work, khat2[v], e2, psi, stream));
      }
    }
  }
  LMVN_CUDA_TRY(cudaEventRecord(ev1, stream));
  if (device_ms) {
    LMVN_CUDA_TRY(cudaEventSynchronize(ev1));
    LMVN_CUDA_TRY(cudaEventElapsedTime(device_ms, ev0, ev1));
  }
  return 0;
}

int Deconv::convolve_psi(int view, int which, int repeats, float* device_ms) {
  NvtxRange nvtx_("lmvn::convolve");
  if (view < 0 || view >= num_views || !view_set[view] || !psi_set) {
    set_last_error("convolve: view %d / psi not set", view);
    return -1;
  }
  LMVN_CUDA_TRY(cudaSetDevice(device));
  const cplx* kh = (which == 2) ? khat2[view] : khat1[view];
  const UpdateParams up = make_update_params(0.0, 0.f);
  LMVN_CUDA_TRY(cudaEventRecord(ev0, stream));
  for (int r = 0; r < repeats; ++r) {
    gen::Epilogue e{gen::EPI_STORE, 1.f, nullptr, nullptr, nullptr, up};
    if (periodic) LMVN_TRY(wrap_exterior(psi));
    LMVN_TRY(engine->convolve(psi, work, kh, e, integral, stream));
    std::swap(psi, integral);
  }
  LMVN_CUDA_TRY(cudaEventRecord(ev1, stream));
  if (device_ms) {
    LMVN_CUDA_TRY(cudaEventSynchronize(ev1));
    LMVN_CUDA_TRY(cudaEventElapsedTime(device_ms, ev0, ev1));
  }
  return 0;
}


int PassTimer::begin(cudaStream_t s) {
  LMVN_CUDA_TRY(cudaEventCreate(&start));
  LMVN_CUDA_TRY(cudaEventRecord(start, s));
  return 0;
}
void PassTimer::mark(const char* name, unsigned long long alg_bytes, cudaStream_t s) {
  Mark m{name, alg_bytes, nullptr};
  if (cudaEventCreate(&m.ev) != cudaSuccess) return;
  cudaEventRecord(m.ev, s);
  marks.push_back(m);
}
PassTimer::~PassTimer() {
  if (start) cudaEventDestroy(start);
  for (auto& m : marks)
    if (m.ev) cudaEventDestroy(m.ev);
}

int Deconv::profile(double lambda, float min_value, std::vector<std::string>& names, std::vector<float>& ms,
                    std::vector<unsigned long long>& alg_bytes) {
  if (!psi_set || !view_set[0]) {
    set_last_error("profile: psi / view 0 not set");
    return -1;
  }
  LMVN_CUDA_TRY(cudaSetDevice(device));
  const size_t S = engine->plan->voxels() * sizeof(float);
  // keep psi: the profiled step runs on a copy parked in `integral`'s place afterwards
  std::vector<float> dummy;
  float* saved = nullptr;
  LMVN_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&saved), S));
  LMVN_CUDA_TRY(cudaMemcpyAsync(saved, psi, S, cudaMemcpyDeviceToDevice, stream));
  const UpdateParams up = make_update_params(lambda, min_value);
  PassTimer t;
  int rc = 0;
  const bool chain = engine->can_chain() && !periodic;
  // chained loop: the steady state of iterate() is profiled (the one x-forward pass that opens a call is not part of it)
  if (chain) rc = engine->chain_begin(psi, work, stream);
  if (rc == 0) rc = t.begin(stream);
  engine->timer = &t;
  gen::Epilogue e1{gen::EPI_QUOTIENT, 1.f, image[0], nullptr, nullptr, up, (padded && !periodic) ? 1 : 0};
  gen::Epilogue e2{gen::EPI_UPDATE, 1.f, nullptr, psi, weights[0], up};
  if (chain) {
    if (rc == 0) rc = engine->chain_middle(work, khat1[0], stream);
    if (rc == 0) rc = engine->chain_link(work, e1, stream);
    if (rc == 0) rc = engine->chain_middle(work, khat2[0], stream);
    if (rc == 0) rc = engine->chain_link(work, e2, stream);
  } else {
    if (rc == 0) rc = engine->convolve(psi, work, khat1[0], e1, integral, stream);
    if (rc == 0) rc = engine->convolve(integral, work, khat2[0], e2, psi, stream);
  }
  engine->timer = nullptr;
  cudaMemcpyAsync(psi, saved, S, cudaMemcpyDeviceToDevice, stream);
  cudaStreamSynchronize(stream);
  cudaFree(saved);
  if (rc != 0) return rc;
  cudaEvent_t prev = t.start;
  for (auto& m : t.marks) {
    float v = 0.f;
    LMVN_CUDA_TRY(cudaEventElapsedTime(&v, prev, m.ev));
    names.push_back(m.name);
    ms.push_back(v);
    alg_bytes.push_back(m.alg_bytes);
    prev = m.ev;
  }
  return 0;
}

// ------------------------------------------------------------------------------
// helpers behind the debug hooks and the legacy single-step entry points
// ------------------------------------------------------------------------------
// natural-layout transforms through the generic passes (tests)
struct DevBuf {
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  int alloc(size_t n) { LMVN_CUDA_TRY(cudaMalloc(&p, n)); return 0; }
};

int debug_transform(const float* in, const int* dims, float* out, int device, bool inverse) {
  if (!in || !dims || !out) { set_last_error("null argument"); return -1; }
  int dev = resolve_device(device);
  if (dev < 0) return -1;
  LMVN_CUDA_TRY(cudaSetDevice(dev));
  auto fp = get_fft_plan(dev, dims[0], dims[1], dims[2]);
  if (!fp) return -1;
  const size_t S = fp->voxels() * sizeof(float), C = fp->spec_elems() * sizeof(cplx);
  DevBuf real, spec;
  LMVN_TRY(real.alloc(S));
  LMVN_TRY(spec.alloc(C));
  const FftPlan& p = *fp;
  const size_t rows = size_t(p.nz) * p.ny;
  dim3 grid_rows(unsigned(ceil_div(rows, p.lines[2])));
  dim3 grid_y(unsigned(ceil_div(size_t(p.nxc), p.lines[1])), unsigned(p.nz));
  dim3 grid_z(unsigned(ceil_div(size_t(p.ny) * p.nxc, p.lines[0])), 1);
  cplx* sp = static_cast<cplx*>(spec.p);
  float* re = static_cast<float*>(real.p);
  if (!inverse) {
    LMVN_CUDA_TRY(cudaMemcpy(re, in, S, cudaMemcpyHostToDevice));
    gen::RealSource src{re, 0, 0, 0, 0};
    LMVN_LAUNCH(gen::k_rows_fwd, grid_rows, dim3(256), p.smem[2], 0, src, sp, p.nz, p.ny, p.nx, p.ax[2], p.lines[2]);
    LMVN_LAUNCH(gen::k_cols, grid_y, dim3(256), p.smem[1], 0, sp, (const cplx*)nullptr, (long long)p.ny * p.nxc,
                (long long)p.nxc, (long long)p.nxc, p.ax[1], p.lines[1], int(gen::COLS_FWD), 1.f);
    LMVN_LAUNCH(gen::k_cols, grid_z, dim3(256), p.smem[0], 0, sp, (const cplx*)nullptr, 0ll,
                (long long)p.ny * p.nxc, (long long)p.ny * p.nxc, p.ax[0], p.lines[0], int(gen::COLS_FWD), 1.f);
    LMVN_CUDA_TRY(cudaGetLastError());
    LMVN_CUDA_TRY(cudaMemcpy(out, sp, C, cudaMemcpyDeviceToHost));
  } else {
    LMVN_CUDA_TRY(cudaMemcpy(sp, in, C, cudaMemcpyHostToDevice));
    LMVN_LAUNCH(gen::k_cols, grid_z, dim3(256), p.smem[0], 0, sp, (const cplx*)nullptr, 0ll,
                (long long)p.ny * p.nxc, (long long)p.ny * p.nxc, p.ax[0], p.lines[0], int(gen::COLS_INV), 1.f);
    LMVN_LAUNCH(gen::k_cols, grid_y, dim3(256), p.smem[1], 0, sp, (const cplx*)nullptr, (long long)p.ny * p.nxc,
                (long long)p.nxc, (long long)p.nxc, p.ax[1], p.lines[1], int(gen::COLS_INV), 1.f);
    gen::Epilogue ep{gen::EPI_STORE, 1.f, nullptr, nullptr, nullptr, make_update_params(0.0, 0.f)};
    LMVN_LAUNCH(gen::k_rows_inv, grid_rows, dim3(256), p.smem[2], 0, (const cplx*)sp, re, p.nz, p.ny, p.nx,
                p.ax[2], p.lines[2], ep);
    LMVN_CUDA_TRY(cudaGetLastError());
    LMVN_CUDA_TRY(cudaMemcpy(out, re, S, cudaMemcpyDeviceToHost));
  }
  return 0;
}

static __global__ void k_unpitch(const float* __restrict__ src, float* __restrict__ dst, size_t rows, int nx, int pitch,
                          int to_pitched) {
  size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t stride = size_t(gridDim.x) * blockDim.x;
  const size_t n = rows * size_t(nx);
  for (; i < n; i += stride) {
    const size_t r = i / nx, x = i % nx;
    if (to_pitched) dst[r * pitch + x] = src[i];
    else dst[i] = src[r * pitch + x];
  }
}

int legacy_core_impl(float* d_im, const int* imDim, const float* d_kernel, const int* kernelDim, int dev) {
  if (!d_im || !imDim || !d_kernel || !kernelDim) { set_last_error("null argument"); return -1; }
  int device = resolve_device(dev);
  if (device < 0) return -1;
  LMVN_CUDA_TRY(cudaSetDevice(device));
  for (int a = 0; a < 3; ++a)
    if (kernelDim[a] <= 0 || kernelDim[a] > imDim[a]) { set_last_error("kernel does not fit image"); return -1; }
  auto fp = get_fft_plan(device, imDim[0], imDim[1], imDim[2]);
  if (!fp) return -1;
  std::unique_ptr<ConvEngine> eng = make_fused_engine(fp);
  if (!eng) eng = make_generic_engine(fp);
  const size_t rows = size_t(fp->nz) * fp->ny;
  const int pitch = 2 * fp->nxc;
  DevBuf real, khat, work;
  LMVN_TRY(real.alloc(fp->voxels() * sizeof(float)));
  LMVN_TRY(khat.alloc(eng->khat_elems() * sizeof(cplx)));
  LMVN_TRY(work.alloc(eng->work_elems() * sizeof(cplx)));
  float* re = static_cast<float*>(real.p);
  const unsigned blocks = unsigned(std::min<size_t>(ceil_div(fp->voxels(), 256), 148 * 16));
  LMVN_LAUNCH(k_unpitch, dim3(blocks), dim3(256), 0, 0, (const float*)d_im, re, rows, fp->nx, pitch, 0);
  const int kd[3] = {kernelDim[0], kernelDim[1], kernelDim[2]};
  LMVN_TRY(eng->kernel_spectrum(d_kernel, kd, static_cast<cplx*>(khat.p), static_cast<cplx*>(work.p), 0));
  gen::Epilogue ep{gen::EPI_STORE, 1.f, nullptr, nullptr, nullptr, make_update_params(0.0, 0.f)};
  // in == out is not allowed by the engines, go through the pitched buffer as scratch target
  DevBuf out;
  LMVN_TRY(out.alloc(fp->voxels() * sizeof(float)));
  LMVN_TRY(eng->convolve(re, static_cast<cplx*>(work.p), static_cast<cplx*>(khat.p), ep, static_cast<float*>(out.p), 0));
  LMVN_LAUNCH(k_unpitch, dim3(blocks), dim3(256), 0, 0, (const float*)out.p, d_im, rows, fp->nx, pitch, 1);
  LMVN_CUDA_TRY(cudaGetLastError());
  LMVN_CUDA_TRY(cudaDeviceSynchronize());
  return 0;
}

int quotient_impl(const float* in, float* out, size_t n, int dev) {
  if (!in || !out) { set_last_error("null argument"); return -1; }
  int device = resolve_device(dev);
  if (device < 0) return -1;
  LMVN_CUDA_TRY(cudaSetDevice(device));
  DevBuf a, b;
  LMVN_TRY(a.alloc(n * sizeof(float)));
  LMVN_TRY(b.alloc(n * sizeof(float)));
  LMVN_CUDA_TRY(cudaMemcpy(a.p, in, n * sizeof(float), cudaMemcpyHostToDevice));
  LMVN_CUDA_TRY(cudaMemcpy(b.p, out, n * sizeof(float), cudaMemcpyHostToDevice));
  const unsigned blocks = unsigned(std::max<size_t>(1, std::min<size_t>(ceil_div(n, 1024), 148 * 8)));
  LMVN_LAUNCH(k_divide, dim3(blocks), dim3(256), 0, 0, (const float*)a.p, (float*)b.p, n);
  LMVN_CUDA_TRY(cudaGetLastError());
  LMVN_CUDA_TRY(cudaMemcpy(out, b.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

int final_values_impl(float* image, const float* integral, const float* weight, size_t n, float min_value,
                      double lambda, int dev) {
  if (!image || !integral || !weight) { set_last_error("null argument"); return -1; }
  int device = resolve_device(dev);
  if (device < 0) return -1;
  LMVN_CUDA_TRY(cudaSetDevice(device));
  DevBuf a, b, c;
  LMVN_TRY(a.alloc(n * sizeof(float)));
  LMVN_TRY(b.alloc(n * sizeof(float)));
  LMVN_TRY(c.alloc(n * sizeof(float)));
  LMVN_CUDA_TRY(cudaMemcpy(a.p, image, n * sizeof(float), cudaMemcpyHostToDevice));
  LMVN_CUDA_TRY(cudaMemcpy(b.p, integral, n * sizeof(float), cudaMemcpyHostToDevice));
  LMVN_CUDA_TRY(cudaMemcpy(c.p, weight, n * sizeof(float), cudaMemcpyHostToDevice));
  const unsigned blocks = unsigned(std::max<size_t>(1, std::min<size_t>(ceil_div(n, 1024), 148 * 8)));
  LMVN_LAUNCH(k_final_values, dim3(blocks), dim3(256), 0, 0, (float*)a.p, (const float*)b.p, (const float*)c.p, n,
              make_update_params(lambda, min_value));
  LMVN_CUDA_TRY(cudaGetLastError());
  LMVN_CUDA_TRY(cudaMemcpy(image, a.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}


}  // namespace lmvn
