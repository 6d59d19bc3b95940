// api.cu -- the C ABI: include/multiviewnative.h (reference drop-in) and
// include/lmvn_b200.h (persistent handle + diagnostics).
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>

#include "engine.cuh"
#include "lmvn_b200.h"
#include "multiviewnative.h"

using namespace lmvn;

static_assert(sizeof(view_data) == 64, "view_data must stay ABI compatible (ref: inc/multiviewnative.h:15-26)");
static_assert(sizeof(workspace) == 32, "workspace must stay ABI compatible (ref: inc/multiviewnative.h:28-35)");
static_assert(offsetof(workspace, num_views_) == 8 && offsetof(workspace, lambda_) == 16 &&
                  offsetof(workspace, minValue_) == 24 && offsetof(workspace, num_iterations_) == 28,
              "workspace field offsets");

struct lmvn_plan {
  Deconv d;
};

// ---------------------------------------------------------------------------------
// extension API
// ---------------------------------------------------------------------------------
extern "C" const char* lmvn_last_error(void) { return last_error(); }
extern "C" void lmvn_clear_error(void) { clear_last_error(); }
extern "C" const char* lmvn_version(void) {
#ifdef LMVN_EMU
  return "libmultiviewnative-b200 0.1 (host emulation build, tests only)";
#else
  return "libmultiviewnative-b200 0.1 (sm_100a)";
#endif
}
extern "C" int lmvn_set_default_strategy(int s) {
  if (s < 0 || s > 2) {
    set_last_error("unknown strategy %d", s);
    return -1;
  }
  set_default_strategy(s);
  return 0;
}

extern "C" void lmvn_release_cached_memory(void) { release_cached_memory(); }

extern "C" int lmvn_plan_create(lmvn_plan** out, const int* dims_zyx, int num_views, int device) {
  if (!out) {
    set_last_error("out is null");
    return -1;
  }
  *out = nullptr;
  lmvn_plan* p = new (std::nothrow) lmvn_plan();
  if (!p) {
    set_last_error("out of host memory");
    return -1;
  }
  if (p->d.init(dims_zyx, num_views, device, 0) != 0) {
    delete p;
    return -1;
  }
  *out = p;
  return 0;
}
namespace {
// smallest extent >= n that the power-of-two fast path takes on this axis (0: none)
int fast_extent(int n, bool x_axis) {
  for (int e = x_axis ? 64 : 16; e <= 1024; e *= 2)
    if (e >= n) return e;
  return 0;
}
int pad_mode_from_env() {
  const char* e = getenv("LMVN_PAD");
  return (e && (e[0] == 'z' || e[0] == 'Z')) ? LMVN_PAD_ZERO : LMVN_PAD_NONE;
}
std::atomic<int> g_pad_mode{-1};  // process wide (lmvn_set_padding); every call samples it once
}  // namespace

extern "C" int lmvn_set_padding(int mode) {
  if (mode != LMVN_PAD_NONE && mode != LMVN_PAD_ZERO) {
    set_last_error("unknown padding mode %d", mode);
    return -1;
  }
  g_pad_mode.store(mode);
  return 0;
}
static int current_pad_mode() {
  const int m = g_pad_mode.load();
  return m >= 0 ? m : pad_mode_from_env();
}

namespace {
thread_local int g_last_geometry = LMVN_GEOMETRY_NONE;

// extents >= image + kernel - 1 that the fast path takes; false when an axis has none
bool fast_extents(const int* image_dims, const int* kmax, int* out) {
  for (int a = 0; a < 3; ++a) {
    out[a] = fast_extent(image_dims[a] + kmax[a] - 1, a == 2);
    if (out[a] <= 0) return false;
  }
  // a plane count that keeps the rows kernels' 128-row granularity
  while ((size_t(out[0]) * out[1]) % 128 != 0 && out[1] < 1024) out[1] *= 2;
  return fused_shape_ok(out[0], out[1], out[2]);
}

int create_padded(lmvn_plan** out, const int* image_dims, const int* kmax, int num_views, int device, bool periodic,
                  bool fast_only) {
  if (!out || !image_dims || !kmax) {
    set_last_error("null argument");
    return -1;
  }
  *out = nullptr;
  int padded[3], off[3], fast[3];
  for (int a = 0; a < 3; ++a) {
    if (image_dims[a] <= 0 || kmax[a] <= 0) { set_last_error("invalid extents"); return -1; }
    if (periodic && kmax[a] > image_dims[a]) {
      set_last_error("kernel extent %d along axis %d does not fit the image extent %d", kmax[a], a, image_dims[a]);
      return -1;
    }
    padded[a] = image_dims[a] + kmax[a] - 1;  // ref: inc/padd_utils.h:133-134
    // zero padding: ref inc/padd_utils.h:136-137; periodic embedding: the left margin must hold the kernel's
    // right half (k - 1 - k/2), the right margin its left half (k/2)
    off[a] = periodic ? kmax[a] - 1 - kmax[a] / 2 : (kmax[a] - 1) / 2;
  }
  const bool have_fast = fast_extents(image_dims, kmax, fast);
  if (fast_only && !have_fast) {
    set_last_error("no power-of-two extents for image + kernel - 1");
    return -1;
  }
  // any extent >= image + kernel - 1 gives the same voxels inside the image; prefer one the fast path takes
  // unless that more than doubles the volume (periodic embedding exists only for the fast path)
  if (have_fast && (fast_only || double(fast[0]) * fast[1] * fast[2] <= 2.0 * double(padded[0]) * padded[1] * padded[2]))
    for (int a = 0; a < 3; ++a) padded[a] = fast[a];
  lmvn_plan* p = new (std::nothrow) lmvn_plan();
  if (!p) { set_last_error("out of host memory"); return -1; }
  if (p->d.init(padded, num_views, device, 0) != 0 || p->d.set_logical(image_dims, off) != 0) {
    delete p;
    return -1;
  }
  p->d.periodic = periodic;
  *out = p;
  return 0;
}

// circular semantics for extents the fast path does not take: embed periodically when that costs at most
// `LMVN_EMBED_MAX_BLOWUP` (default 8) times the voxels -- measured on B200 the embedded fast path still beats the
// generic passes by 2x at that blow-up (400x400x200: 2.1x faster at 2.1x the voxels) -- else the generic passes
bool want_embedding(const int* image_dims, const int* kmax) {
  const char* e = getenv("LMVN_EMBED");
  if (e && *e == '0') return false;
  if (fused_shape_ok(image_dims[0], image_dims[1], image_dims[2])) return false;
  for (int a = 0; a < 3; ++a)
    if (kmax[a] > image_dims[a]) return false;
  int fast[3];
  if (!fast_extents(image_dims, kmax, fast)) return false;
  double limit = 8.0;
  if (const char* m = getenv("LMVN_EMBED_MAX_BLOWUP")) limit = atof(m);
  const double blowup = double(fast[0]) * fast[1] * fast[2] / (double(image_dims[0]) * image_dims[1] * image_dims[2]);
  return blowup <= limit;
}
}  // namespace

extern "C" int lmvn_last_geometry(void) { return g_last_geometry; }

extern "C" int lmvn_plan_create_zero_padded(lmvn_plan** out, const int* image_dims, const int* max_kernel_dims,
                                            int num_views, int device) {
  return create_padded(out, image_dims, max_kernel_dims, num_views, device, false, false);
}

extern "C" int lmvn_plan_create_embedded(lmvn_plan** out, const int* image_dims, const int* max_kernel_dims,
                                         int num_views, int device) {
  return create_padded(out, image_dims, max_kernel_dims, num_views, device, true, true);
}

extern "C" void lmvn_plan_destroy(lmvn_plan* plan) { delete plan; }

extern "C" int lmvn_plan_get_info(const lmvn_plan* plan, lmvn_plan_info* info) {
  if (!plan || !info) {
    set_last_error("null argument");
    return -1;
  }
  const Deconv& d = plan->d;
  const FftPlan& fp = *d.engine->plan;
  std::memset(info, 0, sizeof(*info));
  for (int a = 0; a < 3; ++a) info->dims[a] = d.dims[a];
  info->num_views = d.num_views;
  info->device = d.device;
  info->strategy = d.engine->strategy();
  info->launches_per_view_iteration = d.engine->launches_per_view_iteration();
  info->arena_bytes = d.arena_bytes;
  info->real_bytes = fp.voxels() * sizeof(float);
  info->spectrum_bytes = fp.spec_elems() * sizeof(cplx);
  info->alg_bytes_per_view_iteration = 7ull * info->real_bytes + 10ull * info->spectrum_bytes;
  return 0;
}

extern "C" int lmvn_plan_set_view(lmvn_plan* plan, int view, const float* image, const float* weights,
                                  const float* kernel1, const int* kernel1_dims, const float* kernel2,
                                  const int* kernel2_dims) {
  if (!plan) { set_last_error("plan is null"); return -1; }
  return plan->d.set_view(view, image, weights, kernel1, kernel1_dims, kernel2, kernel2_dims);
}
extern "C" int lmvn_plan_set_psi(lmvn_plan* plan, const float* psi) {
  if (!plan) { set_last_error("plan is null"); return -1; }
  return plan->d.set_psi(psi);
}
extern "C" int lmvn_plan_get_psi(lmvn_plan* plan, float* psi) {
  if (!plan) { set_last_error("plan is null"); return -1; }
  return plan->d.get_psi(psi);
}
extern "C" int lmvn_plan_iterate(lmvn_plan* plan, int iterations, double lambda, float min_value,
                                 float* device_ms) {
  if (!plan) { set_last_error("plan is null"); return -1; }
  return plan->d.iterate(iterations, lambda, min_value, device_ms);
}
extern "C" int lmvn_plan_convolve(lmvn_plan* plan, int view, int which_kernel, int repeats, float* device_ms) {
  if (!plan) { set_last_error("plan is null"); return -1; }
  return plan->d.convolve_psi(view, which_kernel, repeats, device_ms);
}
extern "C" int lmvn_plan_profile(lmvn_plan* plan, double lambda, float min_value, int max_entries, char* names,
                                 float* ms, unsigned long long* alg_bytes, int* count) {
  if (!plan || !names || !ms || !alg_bytes || !count) { set_last_error("null argument"); return -1; }
  std::vector<std::string> n;
  std::vector<float> t;
  std::vector<unsigned long long> b;
  LMVN_TRY(plan->d.profile(lambda, min_value, n, t, b));
  const int k = std::min<int>(max_entries, int(n.size()));
  for (int i = 0; i < k; ++i) {
    std::snprintf(names + size_t(i) * 48, 48, "%s", n[i].c_str());
    ms[i] = t[i];
    alg_bytes[i] = b[i];
  }
  *count = k;
  return 0;
}
extern "C" int lmvn_plan_synchronize(lmvn_plan* plan) {
  if (!plan) { set_last_error("plan is null"); return -1; }
  return plan->d.synchronize();
}

extern "C" int lmvn_debug_rfftn(const float* in, const int* dims_zyx, float* spectrum, int device) {
  return lmvn::debug_transform(in, dims_zyx, spectrum, device, false);
}
extern "C" int lmvn_debug_irfftn(const float* spectrum, const int* dims_zyx, float* out, int device) {
  return lmvn::debug_transform(spectrum, dims_zyx, out, device, true);
}
extern "C" int lmvn_debug_fill_parked_arenas(int byte) {
  return lmvn::debug_fill_parked_arenas(byte);
}

// ---------------------------------------------------------------------------------
// reference C API: GPU entry points (ref: src/multiviewnative.cu:58-142)
// ---------------------------------------------------------------------------------
namespace {

// RAII so that every early return releases the handle
struct PlanGuard {
  lmvn_plan* p = nullptr;
  ~PlanGuard() { delete p; }
};

int gpu_deconvolve_impl(float* psi, const workspace& in, int device) {
  if (!psi || !in.data_ || in.num_views_ == 0) {
    set_last_error("inplace_gpu_deconvolve: null psi / workspace or zero views");
    return -1;
  }
  const int* dims = in.data_[0].image_dims_;
  if (!dims) { set_last_error("view 0 has no image dims"); return -1; }
  // psi takes view 0's dims and every view is assumed identical
  // (ref: src/multiviewnative.cpp:180-181); enforced here, decision q6
  for (int v = 0; v < in.num_views_; ++v) {
    const int* d = in.data_[v].image_dims_;
    if (!d || d[0] != dims[0] || d[1] != dims[1] || d[2] != dims[2]) {
      set_last_error("view %d: image dims differ from view 0", v);
      return -1;
    }
  }
  if (in.num_iterations_ <= 0) return 0;  // psi unchanged (ref: tests/test_gpu_deconvolve_impl.cu:333-377)
  PlanGuard g;
  int kmax[3] = {1, 1, 1};
  for (int v = 0; v < in.num_views_; ++v)
    for (int a = 0; a < 3; ++a) {
      if (in.data_[v].kernel1_dims_) kmax[a] = std::max(kmax[a], in.data_[v].kernel1_dims_[a]);
      if (in.data_[v].kernel2_dims_) kmax[a] = std::max(kmax[a], in.data_[v].kernel2_dims_[a]);
    }
  if (current_pad_mode() == LMVN_PAD_ZERO) {
    // the reference's GPU geometry: extents = image + largest kernel - 1 (ref: src/gpu_deconvolve_methods.cuh:366-379)
    LMVN_TRY(lmvn_plan_create_zero_padded(&g.p, dims, kmax, in.num_views_, device));
    g_last_geometry = LMVN_GEOMETRY_ZERO_PADDED;
  } else if (default_strategy() != 1 && want_embedding(dims, kmax) &&
             lmvn_plan_create_embedded(&g.p, dims, kmax, in.num_views_, device) == 0) {
    // circular semantics on the fast path for extents it does not take itself (when the larger arena does not
    // fit, the call falls through to the native extents)
    g_last_geometry = LMVN_GEOMETRY_EMBEDDED;
  } else {
    clear_last_error();
    LMVN_TRY(lmvn_plan_create(&g.p, dims, in.num_views_, device));
    g_last_geometry = LMVN_GEOMETRY_NATIVE;
  }
  for (int v = 0; v < in.num_views_; ++v) {
    const view_data& vd = in.data_[v];
    LMVN_TRY(g.p->d.set_view(v, vd.image_, vd.weights_, vd.kernel1_, vd.kernel1_dims_, vd.kernel2_, vd.kernel2_dims_));
  }
  LMVN_TRY(g.p->d.set_psi(psi));
  LMVN_TRY(g.p->d.iterate(in.num_iterations_, in.lambda_, in.minValue_, nullptr));
  // psi is written only after the whole loop succeeded
  LMVN_TRY(g.p->d.get_psi(psi));
  return 0;
}

int gpu_convolution_impl(float* im, const int* imDim, const float* kernel, const int* kernelDim, int device) {
  if (!im || !imDim || !kernel || !kernelDim) {
    set_last_error("inplace_gpu_convolution: null argument");
    return -1;
  }
  PlanGuard g;
  if (current_pad_mode() == LMVN_PAD_ZERO) {
    LMVN_TRY(lmvn_plan_create_zero_padded(&g.p, imDim, kernelDim, 1, device));
    g_last_geometry = LMVN_GEOMETRY_ZERO_PADDED;
  } else if (default_strategy() != 1 && want_embedding(imDim, kernelDim) &&
             lmvn_plan_create_embedded(&g.p, imDim, kernelDim, 1, device) == 0) {
    g_last_geometry = LMVN_GEOMETRY_EMBEDDED;
  } else {
    clear_last_error();
    LMVN_TRY(lmvn_plan_create(&g.p, imDim, 1, device));
    g_last_geometry = LMVN_GEOMETRY_NATIVE;
  }
  Deconv& d = g.p->d;
  // a one-view handle: only kernel1's spectrum is used, the image doubles as the
  // view/weights upload (never read by convolve_psi)
  LMVN_CUDA_TRY(cudaSetDevice(d.device));
  const int kd[3] = {kernelDim[0], kernelDim[1], kernelDim[2]};
  LMVN_TRY(d.set_psi(im));
  {
    // upload + spectrum of the single kernel without touching the view buffers
    const size_t kn = size_t(kd[0]) * kd[1] * kd[2];
    for (int a = 0; a < 3; ++a)
      if (kd[a] <= 0 || kd[a] > imDim[a]) {
        set_last_error("kernel extent %d along axis %d does not fit the image extent %d", kd[a], a, imDim[a]);
        return -1;
      }
    if (kn > d.kernel_stage_elems) { set_last_error("kernel too large"); return -1; }
    LMVN_CUDA_TRY(cudaMemcpyAsync(d.kernel_stage, kernel, kn * sizeof(float), cudaMemcpyHostToDevice, d.stream));
    LMVN_TRY(d.engine->kernel_spectrum(d.kernel_stage, kd, d.khat1[0], d.work, d.stream));
    d.view_set[0] = 1;
  }
  LMVN_TRY(d.convolve_psi(0, 1, 1, nullptr));
  LMVN_TRY(d.get_psi(im));
  return 0;
}

}  // namespace

extern "C" void inplace_gpu_deconvolve(imageType* psi, workspace input, int device) {
  (void)gpu_deconvolve_impl(psi, input, device);
}

extern "C" void inplace_gpu_convolution(imageType* im, int* imDim, imageType* kernel, int* kernelDim, int device) {
  (void)gpu_convolution_impl(im, imDim, kernel, kernelDim, device);
}

// ---------------------------------------------------------------------------------
// legacy single-step API (ref: src/multiviewnative.cu:199-595) -- thin wrappers
// ---------------------------------------------------------------------------------
extern "C" void convolution3DfftCUDAInPlace(imageType* im, int* imDim, imageType* kernel, int* kernelDim,
                                            int devCUDA) {
  // Same circular convolution as inplace_gpu_convolution.  The reference's version is not reproducible bit for bit
  // because it reads uninitialised device memory: it cudaMalloc's imSize + 2 d0 d1 floats (ref: src/multiviewnative.cu:
  // 210-216), copies the imSize UNPITCHED image floats in (:225) and runs the in-place R2C, which reads rows at pitch
  // d2 + 2 -- i.e. a sheared image whose last rows come from the never-written tail of the allocation.  Only sums are
  // (approximately) preserved, and sums are all its tests check (ref: tests/test_gpu_convolve.cpp:12-191); those tests pass
  // against this entry point (tests/parity_cases.py case_conv_fixture(entry="convolution3DfftCUDAInPlace")).
  (void)gpu_convolution_impl(im, imDim, kernel, kernelDim, devCUDA);
}

namespace {
// One RL step with kernel2 = 0.1 everywhere, weights = 1, as the legacy entry
// points hard-code (ref: src/multiviewnative.cu:420-421, 489).
int legacy_iterate_impl(const float* input, const float* kernel, float* output, const int* dims, const int* kdims,
                        float min_value, double lambda, int device) {
  if (!input || !kernel || !output || !dims || !kdims) { set_last_error("null argument"); return -1; }
  const size_t n = size_t(dims[0]) * dims[1] * dims[2];
  const size_t kn = size_t(kdims[0]) * kdims[1] * kdims[2];
  std::vector<float> k2(kn, 0.1f), w(n, 1.f);
  PlanGuard g;
  LMVN_TRY(lmvn_plan_create(&g.p, dims, 1, device));
  LMVN_TRY(g.p->d.set_view(0, input, w.data(), kernel, kdims, k2.data(), kdims));
  LMVN_TRY(g.p->d.set_psi(input));
  LMVN_TRY(g.p->d.iterate(1, lambda, min_value, nullptr));
  LMVN_TRY(g.p->d.get_psi(output));
  return 0;
}
}  // namespace

extern "C" void convolution3DfftCUDAInPlace_core(imageType* _d_imCUDA, int* imDim, imageType* _d_kernelCUDA,
                                                 int* kernelDim, int devCUDA) {
  (void)legacy_core_impl(_d_imCUDA, imDim, _d_kernelCUDA, kernelDim, devCUDA);
}
extern "C" void compute_quotient(imageType* _input, imageType* _output, size_t _size, int _device) {
  (void)quotient_impl(_input, _output, _size, _device);
}
extern "C" void compute_final_values(imageType* _image, imageType* _integral, imageType* _weight, size_t _size,
                                     float _minValue, double _lambda, int _device) {
  (void)final_values_impl(_image, _integral, _weight, _size, _minValue, _lambda, _device);
}
extern "C" void iterate_fft_plain(imageType* _input, imageType* _kernel, imageType* _output, int* _input_dims,
                                  int* _kernel_dims, int _device) {
  (void)legacy_iterate_impl(_input, _kernel, _output, _input_dims, _kernel_dims, 1e-4f, 0.0, _device);
}
extern "C" void iterate_fft_tikhonov(imageType* _input, imageType* _kernel, imageType* _output, int* _input_dims,
                                     int* _kernel_dims, size_t, float _minValue, double _lambda, int _device) {
  // Like the reference, this entry point IGNORES _minValue and _lambda: it hard-codes minValue = 1e-4 and lambda = 0.2
  // (ref: src/multiviewnative.cu:582-583 `device_finalValues_tikhonov<<<...>>>(d_initial_, d_image_, d_weights_, .0001f,
  // .2f, inputSize)`).  Its older update rule, new = w (max(min, v) - v) + v with v = (sqrt(1 + 2 lambda psi integral) - 1)
  // / lambda (ref: inc/cuda_kernels.cuh:161-194), blends towards the VALUE instead of towards the last psi; with the
  // weights of 1 this entry point hard-codes (:527) both rules give max(min, v), so the main path's update is exact here.
  // (The reference additionally passes `&weights_[0]` / `&kernel2_[0]` of POINTERS to vectors (:548, :573), i.e. it
  // uploads the vector objects' own bytes instead of their data -- undefined behaviour that is not reproduced; the
  // intended values 1 and 0.1 are used.)  LMVN_LEGACY_HONOUR_ARGS=1 makes the entry point use its arguments instead.
  (void)_minValue; (void)_lambda;
  float min_value = 1e-4f;
  double lambda = 0.2;
  if (const char* e = getenv("LMVN_LEGACY_HONOUR_ARGS"))
    if (*e == '1') { min_value = _minValue; lambda = _lambda; }
  (void)legacy_iterate_impl(_input, _kernel, _output, _input_dims, _kernel_dims, min_value, lambda, _device);
}

// ---------------------------------------------------------------------------------
// device queries (ref: inc/cuda_helpers.cuh:70-136)
// ---------------------------------------------------------------------------------
extern "C" int selectDeviceWithHighestComputeCapability() { return resolve_device(-1); }
extern "C" int getNumDevicesCUDA() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}
static bool props_of(int dev, cudaDeviceProp* p) {
  int n = getNumDevicesCUDA();
  if (dev < 0 || dev >= n) {
    set_last_error("device %d out of range (have %d)", dev, n);
    return false;
  }
  return cudaGetDeviceProperties(p, dev) == cudaSuccess;
}
extern "C" int getCUDAcomputeCapabilityMajorVersion(int devCUDA) {
  cudaDeviceProp p;
  return props_of(devCUDA, &p) ? p.major : -1;
}
extern "C" int getCUDAcomputeCapabilityMinorVersion(int devCUDA) {
  cudaDeviceProp p;
  return props_of(devCUDA, &p) ? p.minor : -1;
}
extern "C" void getNameDeviceCUDA(int devCUDA, char* name) {
  if (!name) return;
  std::memset(name, 0, 256);  // the reference copies 256 bytes (ref: inc/cuda_helpers.cuh:90-95)
  cudaDeviceProp p;
  if (props_of(devCUDA, &p)) std::memcpy(name, p.name, 256);
}
extern "C" long long int getMemDeviceCUDA(int devCUDA) {
  cudaDeviceProp p;
  return props_of(devCUDA, &p) ? (long long)p.totalGlobalMem : -1;
}
