// engine.cuh -- host side of the all-on-device strategy.
//
//   FftPlan      twiddle tables + per-axis factorisation for one (device, dims);
//                kept in a process-wide, mutex-protected store keyed by shape
//                (replaces ref: inc/plan_store.cuh:20-217, which caches cufftHandles
//                in an unsynchronised singleton).
//   ConvEngine   one FFT-convolution strategy: kernel-spectrum precompute and
//                `out = epilogue(irfftn(rfftn(in) * K^))`.
//   Deconv       the persistent handle behind lmvn_plan_* / inplace_gpu_deconvolve:
//                one arena allocation, views + weights + 2V spectra resident,
//                the (iteration, view) loop of ref: src/multiviewnative.cpp:191-229
//                with no host round trip (replaces ref:
//                src/gpu_deconvolve_methods.cuh:345-562, which re-uploads four
//                stacks and re-transforms both kernels every step).
#pragma once
#include <map>
#include <memory>
#include <mutex>
#include <vector>

#include "fft_types.cuh"
#include "lmvn_common.cuh"

namespace lmvn {

bool trace_enabled();
void trace(const char* fmt, ...);

struct FftPlan {
  int device = 0;
  int nz = 0, ny = 0, nx = 0, nxc = 0;
  gen::AxisPlan ax[3];  // 0: z, 1: y, 2: x
  cplx* d_tw[3] = {nullptr, nullptr, nullptr};
  int lines[3] = {1, 1, 1};    // lines per CTA in the generic passes
  size_t smem[3] = {0, 0, 0};  // dynamic shared memory of the generic passes
  // device tables of the fast path, built once per (device, dims) and shared by every engine on the plan
  std::shared_ptr<void> fast_tables;
  std::mutex fast_mu;
  size_t voxels() const { return size_t(nz) * ny * nx; }
  size_t spec_elems() const { return size_t(nz) * ny * nxc; }
  ~FftPlan();
};

// returns nullptr (and sets the last error) on failure
std::shared_ptr<FftPlan> get_fft_plan(int device, int nz, int ny, int nx);

// Optional per-launch timing: engines call mark() after every kernel launch; the
// events sit on the same stream as the kernels.
struct PassTimer {
  struct Mark { const char* name; unsigned long long alg_bytes; cudaEvent_t ev; };
  cudaEvent_t start = nullptr;
  std::vector<Mark> marks;
  int begin(cudaStream_t s);
  void mark(const char* name, unsigned long long alg_bytes, cudaStream_t s);
  ~PassTimer();
};

struct ConvEngine {
  std::shared_ptr<FftPlan> plan;
  PassTimer* timer = nullptr;  // set only while profiling
  void mark(const char* name, unsigned long long bytes, cudaStream_t s) { if (timer) timer->mark(name, bytes, s); }
  virtual ~ConvEngine() {}
  virtual int strategy() const = 0;
  virtual size_t khat_elems() const = 0;  // complex elements of one precomputed PSF spectrum
  virtual size_t work_elems() const = 0;  // complex elements of the spectrum work buffer
  virtual int launches_per_conv() const = 0;
  virtual int launches_per_view_iteration() const { return 2 * launches_per_conv(); }
  // K^ = rfftn(wrap(kernel)) / N in this engine's layout.  d_kernel: device, unpadded.
  virtual int kernel_spectrum(const float* d_kernel, const int kd[3], cplx* khat, cplx* work,
                              cudaStream_t s) = 0;
  virtual int convolve(const float* in, cplx* work, const cplx* khat, const gen::Epilogue& ep,
                       float* out, cudaStream_t s) = 0;
  // Chained form of the same convolution for the RL loop (optional).  The x pass that ENDS one convolution
  // and the x pass that STARTS the next work on the same rows, so they are one kernel: the quotient never goes
  // to HBM and the updated psi is not read back.
  //   chain_begin(in, work)            work <- x forward of `in`
  //   chain_middle(work, khat)         y forward, z forward * K^ * z inverse, y inverse
  //   chain_link(work, ep)             x inverse + pointwise (ep) + x forward of the result, in place in `work`
  //                                    (EPI_UPDATE also stores psi; EPI_QUOTIENT stores nothing)
  //   chain_end(work, ep, out)         x inverse + pointwise, no follow-up transform
  virtual bool can_chain() const { return false; }
  virtual int chain_begin(const float*, cplx*, cudaStream_t) { return -1; }
  virtual int chain_middle(cplx*, const cplx*, cudaStream_t) { return -1; }
  virtual int chain_link(cplx*, const gen::Epilogue&, cudaStream_t) { return -1; }
  virtual int chain_end(cplx*, const gen::Epilogue&, float*, cudaStream_t) { return -1; }
  // chain_link for a periodically embedded stack (logical box inside the plan extents): rows outside the box recompute
  // the interior row they alias, so the result goes to a second buffer `out` (same size as `work`)
  virtual bool can_chain_embedded() const { return false; }
  // (EPI_UPDATE: the new psi is written to `psi_out`, the old one in ep.psi stays intact)
  virtual int chain_link_embedded(cplx*, cplx*, const gen::Epilogue&, float* /*psi_out*/, const int*, const int*,
                                  cudaStream_t) { return -1; }
};

// What the slab-decomposed (multi-GPU) engine needs from the power-of-two fast path: the same
// kernels with explicit geometry.  All pointers are device pointers; spectra use row pitch nxp().
struct StridedGeom {
  cplx* data = nullptr;        // transformed in place (except for scattered final stores)
  const cplx* khat = nullptr;  // merged z pass only
  int n = 0;                   // transform length (the axis whose twiddle tables are used: tw_axis)
  int tw_axis = 1;             // 1: tables of the plan's ny, 0: tables of the plan's nz
  int row_stride = 0;          // complex elements between consecutive rows of the transform axis
  long long tile_stride = 0;   // between consecutive slow indices
  unsigned slow = 1;           // number of slow indices (grid.y)
  int mode = 0;                // fast::StridedMode
  float scale = 1.f;
  Scatter sc{};                // SM_*_SCATTER
  cplx* nyq = nullptr;         // split layout: Nyquist plane of `data` (nullptr: the column is inside the rows)
  const cplx* nyq_khat = nullptr;
  // column window (whole-row layouts only): the pass covers kx columns [col0, col0 + ncols) -- col0 a multiple of the
  // tile width.  ncols = 0: all columns.  The slab-decomposed plans pipeline their exchanges over such windows.
  int col0 = 0, ncols = 0;
  bool khat_half = false;      // merged z pass: khat / nyq_khat hold __half2 elements + un-scale factor (opt-in)
};
struct FastOps {
  virtual ~FastOps() {}
  virtual int nxp_pitch() const = 0;
  // x transform of nz_local planes: src -> spec.  Wrapped (PSF) sources take the global plane offset / count.
  virtual int rows_fwd_planes(const gen::RealSource& src, cplx* spec, int nz_local, int z0_global, int nz_global,
                              cudaStream_t s) = 0;
  virtual int rows_inv_planes(const cplx* spec, float* out, const gen::Epilogue& ep, int nz_local, cudaStream_t s) = 0;
  virtual int strided_geom(const StridedGeom& g, cudaStream_t s) = 0;
  virtual int strided_tile_cols(int n) const = 0;  // tile width (kx columns) of the strided passes along an axis of length n
  // chained x passes (x inverse + pointwise + x forward in place on nz_local planes of `spec`); false: not available
  virtual bool can_chain_rows() const = 0;
  virtual int rows_inv_fwd_planes(cplx* spec, const gen::Epilogue& ep, int nz_local, cudaStream_t s) = 0;
};
// nullptr (last error set) when the global shape is not eligible for the fast path
std::unique_ptr<FastOps> make_fast_ops(std::shared_ptr<FftPlan> plan_global);

std::unique_ptr<ConvEngine> make_generic_engine(std::shared_ptr<FftPlan> plan);
// nullptr when the shape is not eligible (no error set)
std::unique_ptr<ConvEngine> make_fused_engine(std::shared_ptr<FftPlan> plan);
bool fused_shape_ok(int nz, int ny, int nx);  // extents the power-of-two fast path takes

int default_strategy();
void set_default_strategy(int s);

struct Deconv {
  int device = 0;
  int dims[3] = {0, 0, 0};
  int num_views = 0;
  std::unique_ptr<ConvEngine> engine;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  unsigned char* arena = nullptr;
  size_t arena_bytes = 0;
  size_t arena_capacity = 0;  // bytes of the underlying allocation (>= arena_bytes when taken from the park)
  float* psi = nullptr;
  float* psi2 = nullptr;          // embedded plans, chained loop: the update link writes the new psi out of place
  float* integral = nullptr;
  cplx* work = nullptr;
  float* kernel_stage = nullptr;  // device staging for the unpadded PSFs
  size_t kernel_stage_elems = 0;
  std::vector<float*> image, weights;
  std::vector<cplx*> khat1, khat2;
  std::vector<char> view_set;
  bool psi_set = false;

  // zero_padd mode (ref: inc/padd_utils.h:102-249, src/gpu_deconvolve_methods.cuh:366-449): the plan works on
  // `dims` = image + kernel - 1 (rounded up to a fast-path extent), the caller's stacks have `logical` extents
  // and sit at `offset` = (kernel - 1) / 2 inside it; uploads zero-fill, downloads crop.
  // CUDA graph of one sweep over all views (chained loop), replayed for every iteration but the last
#ifndef LMVN_EMU
  cudaGraphExec_t sweep_graph = nullptr;
#endif
  bool use_graph = true;
  double graph_lambda = 0.0;
  float graph_min = 0.f;
  const float* graph_psi = nullptr;

  bool padded = false;
  // periodic embedding: the exterior of the logical box is refilled by periodic continuation before every
  // convolution, so that the result inside the box is the CIRCULAR convolution at the logical extents (the CPU
  // path's semantics) although the transform runs at power-of-two extents
  bool periodic = false;
  int logical[3] = {0, 0, 0};
  int offset[3] = {0, 0, 0};
  int set_logical(const int* image_dims, const int* off);
  int wrap_exterior(float* vol);
  int upload_stack(float* dst, const float* src_h);
  int download_stack(float* dst_h, const float* src);

  ~Deconv();
  int init(const int* dims_zyx, int nviews, int dev, int strategy);
  int set_view(int v, const float* image_h, const float* weights_h, const float* k1, const int* k1d,
               const float* k2, const int* k2d);
  int set_psi(const float* psi_h);
  int get_psi(float* psi_h);
  int iterate(int iterations, double lambda, float min_value, float* device_ms);
  int convolve_psi(int view, int which, int repeats, float* device_ms);
  int synchronize();
  // one (view 0, iteration) with an event after every launch; psi is restored afterwards
  int profile(double lambda, float min_value, std::vector<std::string>& names, std::vector<float>& ms,
              std::vector<unsigned long long>& alg_bytes);
};

void release_cached_memory();  // frees the arenas parked by destroyed handles
int debug_fill_parked_arenas(int byte);  // memsets every parked arena (tests: the next handle starts on dirty memory)
int resolve_device(int device);  // < 0 -> highest compute capability; validates range

// debug hooks / legacy single-step entry points (host pointers unless noted)
int debug_transform(const float* in, const int* dims, float* out, int device, bool inverse);
int legacy_core_impl(float* d_im, const int* imDim, const float* d_kernel, const int* kernelDim, int dev);  // device ptrs
int quotient_impl(const float* in, float* out, size_t n, int dev);
int final_values_impl(float* image, const float* integral, const float* weight, size_t n, float min_value,
                      double lambda, int dev);

// Whole-stack copies between caller memory and the device on stream s.  Pageable host memory (what JNA hands over)
// is staged through a per-device ring of pinned chunks filled by several host threads (engine.cu, HostStager);
// pinned / registered memory and small copies go straight to cudaMemcpyAsync.
int copy_to_device(int device, void* dst_d, const void* src_h, size_t bytes, cudaStream_t s);
int copy_to_host(int device, void* dst_h, const void* src_d, size_t bytes, cudaStream_t s);

}  // namespace lmvn
