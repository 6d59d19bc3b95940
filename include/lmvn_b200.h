/*
 * lmvn_b200.h -- additions of the B200-native build that sit NEXT TO the
 * reference C ABI (include/multiviewnative.h) without changing it.
 *
 *  - lmvn_last_error():  the reference reports failures by exit()ing the host
 *    process (ref: inc/cuda_helpers.cuh:17-24); this build never does, the text
 *    of the last failure of the calling thread is available here instead.
 *  - lmvn_plan_*: a persistent handle for the same deconvolution
 *    (SURVEY.md §8f-1).  Fiji drives the reference by calling
 *    inplace_gpu_deconvolve repeatedly with few iterations each
 *    (ref: bench/bench_gpu_deconvolve.cu:48-49); the handle keeps views, weights
 *    and the precomputed PSF spectra resident so that only psi moves.  The
 *    one-shot entry points of multiviewnative.h are thin wrappers over it.
 *  - lmvn_debug_*: forward / inverse transforms in natural layout, for tests.
 *
 * All functions return 0 on success and non-zero on failure (message via
 * lmvn_last_error()).  Plain C, plain pointers, no C++ or torch types.
 */
#ifndef LMVN_B200_EXT_H
#define LMVN_B200_EXT_H

#include "multiviewnative.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lmvn_plan lmvn_plan;

enum lmvn_strategy {
  LMVN_STRATEGY_AUTO = 0,    /* fused power-of-two path when the shape allows, else generic */
  LMVN_STRATEGY_GENERIC = 1, /* any shape: five separable passes per convolution             */
  LMVN_STRATEGY_FUSED = 2    /* three fused passes per convolution (power-of-two extents)    */
};

typedef struct lmvn_plan_info {
  int dims[3];
  int num_views;
  int device;
  int strategy;                        /* resolved strategy, LMVN_STRATEGY_GENERIC or _FUSED */
  int launches_per_view_iteration;     /* kernels of this library per (view, iteration)      */
  unsigned long long arena_bytes;      /* device memory held by the handle                    */
  unsigned long long real_bytes;       /* S = 4*N                                             */
  unsigned long long spectrum_bytes;   /* C = 8*nz*ny*(nx/2+1)                                */
  unsigned long long alg_bytes_per_view_iteration; /* 7S + 10C (SURVEY.md §8d)                */
} lmvn_plan_info;

LMVN_EXPORT const char* lmvn_last_error(void);
LMVN_EXPORT void lmvn_clear_error(void);
LMVN_EXPORT const char* lmvn_version(void);

/* process-wide default used by plans created afterwards (also env LMVN_STRATEGY=generic|fused) */
LMVN_EXPORT int lmvn_set_default_strategy(int strategy);

/* A destroyed plan (and every one-shot inplace_gpu_* call) parks its device arena for the next plan on
 * that device instead of returning it to the driver (env LMVN_CACHE_ARENA=0 disables).  Pageable host stacks of
 * 4 MB and more are staged through a per-device ring of pinned chunks (3 x 16 MiB, env LMVN_STAGED_COPY=0 leaves the
 * staging to the driver).  This frees both. */
LMVN_EXPORT void lmvn_release_cached_memory(void);

LMVN_EXPORT int lmvn_plan_create(lmvn_plan** out, const int* dims_zyx, int num_views, int device);
/* zero_padd mode of the reference's GPU path (ref: inc/padd_utils.h:102-249, src/gpu_deconvolve_methods.cuh:366-449):
 * the plan works on image + kernel - 1 extents (rounded up to a fast-path extent when that is cheap), the caller's
 * stacks keep the image extents and sit at offset (kernel - 1) / 2; uploads zero-fill, get_psi crops.  Linear instead of
 * circular convolution at the image borders.  One rule differs from the reference's arithmetic: the quotient of a voxel
 * whose view is exactly zero (all of the padding) is zero; the reference computes 0 * (1 / blurred) there, which is the
 * same number unless blurred is exactly zero -- then it is a NaN that the second convolution spreads over the stack.  lmvn_set_padding / env LMVN_PAD=zero switch the one-shot entry points
 * (inplace_gpu_deconvolve, inplace_gpu_convolution) to it; the default is the CPU path's circular geometry. */
enum lmvn_padding { LMVN_PAD_NONE = 0, LMVN_PAD_ZERO = 1 };
LMVN_EXPORT int lmvn_set_padding(int mode);
LMVN_EXPORT int lmvn_plan_create_zero_padded(lmvn_plan** out, const int* image_dims_zyx, const int* max_kernel_dims_zyx,
                                             int num_views, int device);
/* Periodic embedding: CIRCULAR convolution at the image extents (the CPU path's semantics, like lmvn_plan_create) for
 * extents the power-of-two fast path does not take.  The stacks sit inside power-of-two extents >= image + kernel - 1;
 * before every convolution the exterior is refilled with the periodic continuation of the interior, so the result inside
 * the image equals the circular convolution at the image extents.  The one-shot entry points choose it by themselves when
 * the image extents are not fast-path extents and the embedding costs at most 8x the voxels (and fits the device) (env LMVN_EMBED=0 disables,
 * LMVN_EMBED_MAX_BLOWUP changes the bound); otherwise they use the generic passes.  lmvn_last_geometry(): what the last
 * one-shot call of this thread used. */
enum lmvn_geometry { LMVN_GEOMETRY_NONE = 0, LMVN_GEOMETRY_NATIVE = 1, LMVN_GEOMETRY_EMBEDDED = 2, LMVN_GEOMETRY_ZERO_PADDED = 3 };
LMVN_EXPORT int lmvn_plan_create_embedded(lmvn_plan** out, const int* image_dims_zyx, const int* max_kernel_dims_zyx,
                                          int num_views, int device);
LMVN_EXPORT int lmvn_last_geometry(void);
LMVN_EXPORT void lmvn_plan_destroy(lmvn_plan* plan);
LMVN_EXPORT int lmvn_plan_get_info(const lmvn_plan* plan, lmvn_plan_info* info);

/* Host pointers.  Uploads image and weights of one view and precomputes both PSF spectra
 * (kernel wrap-around + forward transform + 1/N, ref: src/multiviewnative.cpp:146-174).
 * BUFFER LIFETIME: lmvn_plan_set_view / lmvn_plan_set_psi (and lmvn_dist_set_*_slab) return once the copy is QUEUED on
 * the plan's stream.  Pageable buffers have been read completely by then (they go through the library's pinned staging
 * ring); PINNED or cudaHostRegister'ed buffers are read by the DMA engine asynchronously and must stay unmodified
 * until lmvn_plan_synchronize (or any call that returns results: lmvn_plan_iterate with device_ms, lmvn_plan_get_psi). */
LMVN_EXPORT int lmvn_plan_set_view(lmvn_plan* plan, int view, const float* image,
                                   const float* weights, const float* kernel1,
                                   const int* kernel1_dims, const float* kernel2,
                                   const int* kernel2_dims);
LMVN_EXPORT int lmvn_plan_set_psi(lmvn_plan* plan, const float* psi);
LMVN_EXPORT int lmvn_plan_get_psi(lmvn_plan* plan, float* psi);

/* `iterations` sweeps over all views on the device (ref: src/multiviewnative.cpp:191-229).
 * device_ms (may be NULL) receives the CUDA-event time of the loop on the plan's stream. */
LMVN_EXPORT int lmvn_plan_iterate(lmvn_plan* plan, int iterations, double lambda, float min_value,
                                  float* device_ms);

/* psi <- psi (*) kernel{1,2} of `view`, `repeats` times (config 2: FFT convolution GB/s). */
LMVN_EXPORT int lmvn_plan_convolve(lmvn_plan* plan, int view, int which_kernel, int repeats,
                                   float* device_ms);
/* Runs ONE (view 0, iteration) with a CUDA event after every kernel launch (same stream) and
 * reports, per launch, its name, device time and algorithmic bytes.  psi is restored.
 * names: count entries of 48 chars; returns the number of launches in *count. */
LMVN_EXPORT int lmvn_plan_profile(lmvn_plan* plan, double lambda, float min_value, int max_entries,
                                  char* names, float* ms, unsigned long long* alg_bytes, int* count);
/* blocks until everything queued on the plan's stream is done */
LMVN_EXPORT int lmvn_plan_synchronize(lmvn_plan* plan);

/* ---------------------------------------------------------------------------------------------
 * ONE volume over several GPUs (BASELINE config 5; the reference has no such path): slabs of
 * nz/G planes in real space, pencils of ny/G rows for the z pass, both all-to-all exchanges of a
 * convolution fused into the transform kernels as stores into peer memory over NVLink.
 * Power-of-two fast-path shapes only (nx in {64,128,256,512,1024}; ny, nz in {16..1024}); G a power of two <= 8.
 *
 * One handle per rank.  Ranks are separate processes (one per GPU: exchange the 64-byte handles of
 * lmvn_dist_export_handle with any transport and pass them to lmvn_dist_connect_ipc, then use
 * lmvn_dist_iterate) or several handles of one process (lmvn_dist_connect_local; the caller issues
 * lmvn_dist_*_phase for every rank and synchronises between phases).
 * Every rank must make the same sequence of calls.  Slab buffers are host pointers to the rank's
 * nz/G planes ([nz/G][ny][nx] floats). */
typedef struct lmvn_dist lmvn_dist;

typedef struct lmvn_dist_info {
  int dims[3];
  int num_views;
  int rank, world, device;
  int planes_per_rank;                 /* nz / G */
  int rows_per_rank;                   /* ny / G */
  int spectrum_pitch;                  /* complex elements per spectrum row */
  unsigned long long arena_bytes;      /* device memory held by this rank */
  unsigned long long exchange_bytes;   /* size of the peer-visible region */
  unsigned long long alg_bytes_per_view_iteration;      /* 7S + 10C of the WHOLE volume */
  unsigned long long exchange_bytes_per_view_iteration; /* 4 C (G-1)/G, all ranks together */
} lmvn_dist_info;

LMVN_EXPORT int lmvn_dist_create(lmvn_dist** out, const int* dims_zyx, int num_views, int rank, int world,
                                 int device);
LMVN_EXPORT void lmvn_dist_destroy(lmvn_dist* plan);
LMVN_EXPORT int lmvn_dist_get_info(const lmvn_dist* plan, lmvn_dist_info* info);
LMVN_EXPORT int lmvn_dist_export_handle(lmvn_dist* plan, void* handle64);
LMVN_EXPORT int lmvn_dist_connect_ipc(lmvn_dist* plan, int peer_rank, const void* handle64);
LMVN_EXPORT int lmvn_dist_connect_local(lmvn_dist* plan, int peer_rank, lmvn_dist* peer);
LMVN_EXPORT int lmvn_dist_set_view_slab(lmvn_dist* plan, int view, const float* image_slab,
                                        const float* weights_slab);
LMVN_EXPORT int lmvn_dist_set_psi_slab(lmvn_dist* plan, const float* psi_slab);
LMVN_EXPORT int lmvn_dist_get_psi_slab(lmvn_dist* plan, float* psi_slab);
/* PSF spectrum of kernel 1 / 2 of a view, straight into the pencil layout.  phase 0: wrap-around +
 * x,y forward + scatter (needs the whole kernel, host pointer); [barrier]; phase 1: z forward, 1/N. */
LMVN_EXPORT int lmvn_dist_psf_phase(lmvn_dist* plan, int view, int which_kernel, int phase,
                                    const float* kernel, const int* kernel_dims);
/* One phase of convolution 1 (psi (*) kernel1 -> quotient) or 2 (integral (*) kernel2 -> update):
 * 0: x,y forward + scatter; [barrier]; 1: z forward * K^ * z inverse + scatter; [barrier]; 2: y,x inverse + pointwise. */
LMVN_EXPORT int lmvn_dist_conv_phase(lmvn_dist* plan, int view, int which_conv, int phase, double lambda,
                                     float min_value);
/* device-side cross-GPU barrier on the plan's stream (no-op for in-process groups) */
LMVN_EXPORT int lmvn_dist_barrier(lmvn_dist* plan);
/* A device-side barrier waits at most LMVN_BARRIER_TIMEOUT_S seconds (default 600) for its peers.  After a timeout
 * lmvn_dist_iterate fails, the result of that call is invalid and the plan refuses further work until EVERY rank has
 * called lmvn_dist_reset_barrier (collective: line the ranks up on the host before and after it). */
LMVN_EXPORT int lmvn_dist_reset_barrier(lmvn_dist* plan);
/* the whole loop, barriers on the device, no host round trip (one process per rank) */
LMVN_EXPORT int lmvn_dist_iterate(lmvn_dist* plan, int iterations, double lambda, float min_value,
                                  float* device_ms);
LMVN_EXPORT int lmvn_dist_synchronize(lmvn_dist* plan);

/* Comparator path: the same exchanges staged through local buffers and moved by the CALLER with a library
 * all-to-all (NCCL).  set_staged(1): phase 0 / 1 scatter into STAGE_SEND as G contiguous blocks
 * [dest][nz/G][ny/G][pitch]; the caller all-to-alls them into PENCIL_WORK (forward) or into STAGE_RECV and
 * then interleaves the sources into SLAB_WORK ([nz/G][src][ny/G][pitch]) (backward).  set_stream makes the
 * plan issue its kernels on the caller's stream so that both sides are stream ordered. */
enum lmvn_dist_buffer_id { LMVN_DIST_SLAB_WORK = 0, LMVN_DIST_PENCIL_WORK = 1, LMVN_DIST_STAGE_SEND = 2, LMVN_DIST_STAGE_RECV = 3 };
LMVN_EXPORT int lmvn_dist_set_stream(lmvn_dist* plan, void* cuda_stream);
LMVN_EXPORT int lmvn_dist_set_staged(lmvn_dist* plan, int on);
LMVN_EXPORT int lmvn_dist_buffer(lmvn_dist* plan, int which, void** device_ptr, unsigned long long* bytes);

/* r2c / c2r of a host volume through the generic passes, natural layout:
 * spectrum = nz*ny*(nx/2+1) interleaved (re,im) pairs.  c2r is unnormalised. */
LMVN_EXPORT int lmvn_debug_rfftn(const float* in, const int* dims_zyx, float* spectrum, int device);
LMVN_EXPORT int lmvn_debug_irfftn(const float* spectrum, const int* dims_zyx, float* out, int device);
/* Sets every byte of every arena parked for later handles (what lmvn_release_cached_memory frees), on every device, to
 * `byte` and waits for it:
 * the next handle that takes one starts on memory full of that pattern (0xff: NaN, 0x3f: about 0.75), so that a read
 * of a buffer the call did not write shows up in its result. */
LMVN_EXPORT int lmvn_debug_fill_parked_arenas(int byte);

#ifdef __cplusplus
}
#endif
#endif /* LMVN_B200_EXT_H */
