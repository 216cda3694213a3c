/*
 * include/fslic_b200.h -- C ABI of the B200-native SLIC engine (libfslic_b200.so).
 *
 * This is the drop-in boundary for the reference's hot path.  The reference crosses from
 * Cython into C++ through `fslic::ContextBuilder().build(H, W, K, image, clusters)`,
 * public config fields, `initialize_clusters()` and `iterate(uint16_t*, max_iter)`
 * (/root/reference/src/context.h:24-75,138-150; call sites cfast_slic.pyx:124-147,150-197)
 * and `cca::ConnectivityEnforcer(...).execute()` (src/cca.h:73-81; cfast_slic.pyx:371-396).
 * The entry points below mirror that lifecycle with plain pointers and sizes -- no C++ or
 * torch types -- so any FFI (ctypes, Cython, cgo, JNI) can bind them.  See INTEGRATION.md.
 *
 * Conventions: every function returns 0 on success, a negative FSLIC_E* code otherwise;
 * `fslic_b200_last_error()` gives the message (thread local).  Pointers named d_* are
 * device pointers on the context's device, h_* are host pointers.  `stream` is a
 * cudaStream_t passed as void* (NULL = default stream); device entry points are
 * asynchronous on that stream.
 */
#ifndef FSLIC_B200_H
#define FSLIC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* == `Cluster`, /root/reference/src/fast-slic-common.h:10-23 (32 bytes, align 4). */
typedef struct fslic_cluster {
    float y, x;          /* centre; always integer-valued on this path (context.cpp:368-373) */
    float r, g, b, a;    /* colour; L*2,a,b when convert_to_lab (cielab.h:308-325), `a` unused */
    uint16_t number;     /* == index */
    uint8_t is_active;   /* 1 after iterate (preemptive.h:69-74) */
    uint8_t is_updatable;/* 2 after iterate (preemptive.h:59-67) */
    uint32_t num_members;/* member count of the LAST subsampled update (context.cpp:360-364) */
} fslic_cluster;

/* == the public config fields of fslic::BaseContext (src/context.h:26-36) that the default
 *    Slic path reads; the values SlicModel.iterate() copies in (cfast_slic.pyx:179-187). */
typedef struct fslic_params {
    float compactness;       /* context.h:28 */
    float min_size_factor;   /* context.h:29 */
    int32_t subsample_stride;/* context.h:26 (subsample_stride_config) */
    int32_t convert_to_lab;  /* context.h:30 */
    int32_t max_iter;        /* argument of iterate(), context.h:72 */
    int32_t collect_timing;  /* 1: per-stage CUDA-event timings (fstimer analogue, timer.cpp:4-49); 2: + per-launch assign kernel */
} fslic_params;

enum {
    FSLIC_OK = 0,
    FSLIC_EINVAL = -1,   /* bad argument (reference: ValueError, cfast_slic.pyx:24-27,125,153) */
    FSLIC_ECUDA = -2,    /* CUDA runtime error */
    FSLIC_ENOMEM = -3,
    FSLIC_ERANGE = -4    /* compactness so large the u16 distance would overflow (UB in the reference); bounded by the
                            largest patch value of the metric in use */
};

typedef struct fslic_ctx fslic_ctx;

/* Stage ids for fslic_b200_stage_ms(): same section names as the reference's timing report
 * (context.cpp:112-192, cca.cpp:194-259). */
enum {
    FSLIC_T_CIELAB = 0, FSLIC_T_ASSIGN = 1, FSLIC_T_UPDATE = 2, FSLIC_T_FULL_ASSIGN = 3,
    FSLIC_T_CCA = 4, FSLIC_T_TOTAL = 5, FSLIC_T_COUNT = 6
};

const char* fslic_b200_last_error(void);
const char* fslic_b200_version(void);
int fslic_b200_sizeof_cluster(void);

/* == ContextBuilder::build + BaseContext ctor (context.h:59-66,149): fixes H, W, K and
 *    S = (int16)sqrt(H*W/K); allocates every scratch buffer for up to max_batch images.
 *    Unlike the reference (which rebuilds a Context per call, cfast_slic.pyx:171-197) the
 *    context is meant to be kept and reused. */
int fslic_b200_create(int device, int H, int W, int K, int max_batch, fslic_ctx** out);
int fslic_b200_destroy(fslic_ctx* ctx);

/* == the scratch of cca::ConnectivityEnforcer alone (cca.cpp:176-192: it needs H, W and nothing of the SLIC
 *    context): a context on which only fslic_b200_enforce_connectivity may be called.  No K is fixed here --
 *    K (max_label_size) is an argument of that call, exactly like the reference's constructor argument. */
int fslic_b200_create_cca(int device, int H, int W, int max_batch, fslic_ctx** out);

/* == the public context field `manhattan_spatial_dist` (context.h:35; cfast_slic.pyx:186,246): nonzero (the default) for
 *    the L1 spatial term coef * (|di| + |dj|), 0 for the Euclidean coef * hypotf(di, dj) of classic SLIC
 *    (context.cpp:23-40, :462-499).  Every iterate entry point reads it when it enqueues work; a call already enqueued
 *    keeps the metric it was enqueued with. */
int fslic_b200_set_manhattan_spatial_dist(fslic_ctx* ctx, int manhattan);

/* == BaseContext::initialize_clusters (context.cpp:43-97), for `batch` images [B,H,W,3] u8. */
int fslic_b200_initialize_clusters(fslic_ctx* ctx, const uint8_t* d_images, fslic_cluster* d_clusters, int batch,
                                   void* stream);

/* == BaseContext::iterate (context.cpp:109-197): Lab LUT -> max_iter x (assign + update on a
 *    row subsample) -> full assign -> connectivity enforcement.  d_images [B,H,W,3] u8,
 *    d_clusters [B,K] (read and updated in place), d_labels [B,H,W] u16 (0xFFFF = unassigned). */
int fslic_b200_iterate(fslic_ctx* ctx, const uint8_t* d_images, fslic_cluster* d_clusters, uint16_t* d_labels,
                       int batch, const fslic_params* params, void* stream);

/* == the float-distance contexts ContextRealDist / ContextRealDistL2 / ContextRealDistNoQ (context.h:100-125,
 *    context.cpp:394-499; selected in cfast_slic.pyx:198-252 by SlicModel.real_dist_type): `variant` 0 = "standard"
 *    (the default kernel with float distances and an untruncated float spatial term), 1 = "l2" (squared colour and
 *    spatial distances), 2 = "noq" (float centroids, no quantisation in the update).  The spatial term follows
 *    fslic_b200_set_manhattan_spatial_dist, except for "l2", whose squared term ignores it (context.cpp:435-445).  Same
 *    buffers and semantics as fslic_b200_iterate; results bit-identical to the reference (every float operation in its
 *    order and rounding). */
int fslic_b200_iterate_real(fslic_ctx* ctx, int variant, const uint8_t* d_images, fslic_cluster* d_clusters,
                            uint16_t* d_labels, int batch, const fslic_params* params, void* stream);

/* == BaseContext::iterate with `preemptive = true` (context.h:32-33, preemptive.h; cfast_slic.pyx:183-184): clusters that
 *    stop moving (L1 movement below max(round(2 S preemptive_thres), 1) pixels in two updates in a row) and have no
 *    moving cluster within 2S stop being assigned and updated; `is_updatable` of the returned records holds the
 *    countdown where it got to.  Same buffers as fslic_b200_iterate; bit-identical to the reference.  S >= 1. */
int fslic_b200_iterate_preemptive(fslic_ctx* ctx, const uint8_t* d_images, fslic_cluster* d_clusters, uint16_t* d_labels,
                                  int batch, const fslic_params* params, float preemptive_thres, void* stream);

/* The same call as the reference-facing plugin makes it: HOST buffers in, HOST buffers out
 * (what SlicModel.iterate does with a numpy image, cfast_slic.pyx:150-260).  H2D copy, kernels and
 * D2H copy are pipelined over chunks of 32 images on three streams (pass pinned buffers for true overlap);
 * returns when the results are in the host buffers. */
int fslic_b200_iterate_host(fslic_ctx* ctx, const uint8_t* h_images, fslic_cluster* h_clusters, uint16_t* h_labels,
                            int batch, const fslic_params* params);
int fslic_b200_initialize_clusters_host(fslic_ctx* ctx, const uint8_t* h_images, fslic_cluster* h_clusters,
                                        int batch);

/* Streaming form of fslic_b200_iterate_host (no counterpart in the reference, whose iterate() blocks): enqueue
 * the same H2D -> kernels -> D2H work and return at once; fslic_b200_wait() blocks until the labels and clusters
 * are in the host buffers.  The host buffers must be pinned and stay untouched until then.  One batch per
 * context may be in flight (a second _async call waits for the first); a caller that alternates between two
 * contexts overlaps one batch's PCIe copies with the other's kernels. */
int fslic_b200_iterate_host_async(fslic_ctx* ctx, const uint8_t* h_images, fslic_cluster* h_clusters,
                                  uint16_t* h_labels, int batch, const fslic_params* params);
int fslic_b200_wait(fslic_ctx* ctx);

/* == cca::ConnectivityEnforcer(labels,H,W,K,min_threshold).execute(labels) (cca.cpp:178-265),
 *    in place on d_labels [B,H,W] u16.  H, W come from the context; K (= max label + 1 in
 *    cfast_slic.pyx:377-382) is given by the caller. */
int fslic_b200_enforce_connectivity(fslic_ctx* ctx, uint16_t* d_labels, int batch, int K, int min_threshold,
                                    void* stream);

/* == fast_slic_get_connectivity (src/fast-slic.cpp:16-78; cfast_slic.pyx:262-270): the superpixel adjacency graph of
 *    one label map d_labels u16[H*W] -> d_counts int32[K], d_neighbors u32[K*12] (row k: the first d_counts[k] entries,
 *    in the order the reference's raster scan links them; at most 12 per label, like the reference).  Stateless:
 *    d_scratch must hold fslic_b200_connectivity_scratch_bytes(K) bytes.  Synchronises `stream` once. */
size_t fslic_b200_connectivity_scratch_bytes(int K);
int fslic_b200_get_connectivity(int device, int H, int W, int K, const uint16_t* d_labels, int32_t* d_counts,
                                uint32_t* d_neighbors, void* d_scratch, size_t scratch_bytes, void* stream);

/* == fast_slic_get_mask_density / fast_slic_cluster_density_to_mask (src/fast-slic.cpp:141-168; cfast_slic.pyx:283-320).
 *    d_mask u8[H*W], d_densities u8[K]; d_scratch int32[K].  Asynchronous on `stream`. */
int fslic_b200_get_mask_density(int device, int H, int W, int K, const fslic_cluster* d_clusters, const uint16_t* d_labels,
                                const uint8_t* d_mask, uint8_t* d_densities, int32_t* d_scratch, void* stream);
int fslic_b200_cluster_density_to_mask(int device, int H, int W, int K, const uint16_t* d_labels, const uint8_t* d_densities,
                                       uint8_t* d_result, void* stream);

/* Stage probes for the parity tests (the reference's protected quad_image / assignment,
 * context.h:48-50): copies of the last iterate()'s Lab quad image [B,H,W,4] u8 and pre-CCA
 * labels [B,H,W] u16 into caller device buffers (either may be NULL). */
int fslic_b200_debug_stages(fslic_ctx* ctx, uint8_t* d_quad_out, uint16_t* d_precca_out, int batch, void* stream);

/* RGB -> quad stage alone (cielab.h:337-353): d_quad_out [B,H,W,4] u8. */
int fslic_b200_rgb_to_quad(fslic_ctx* ctx, const uint8_t* d_images, uint8_t* d_quad_out, int batch,
                           int convert_to_lab, void* stream);

/* libstdc++ std::partial_sort set selection on the device (cca.cpp:225-228), exposed for
 * differential tests: d_area int32[n]; writes d_kept u8[n] (1 = in the selected top-`middle`). */
int fslic_b200_debug_heap_select(fslic_ctx* ctx, const int32_t* d_area, int n, int middle, uint8_t* d_kept,
                                 void* stream);

/* With collect_timing >= 2: summed device time (CUDA events on the launch stream) and launch count of the
 * dominant kernel -- the fused assign+update kernel on the subsampled passes -- in the last iterate(). */
int fslic_b200_assign_kernel_time(fslic_ctx* ctx, float* total_ms, int* launches);

/* Diagnostics: the 8 int32 CCA counters of image `image` of the last (sub-)batch:
 * ncomp, ncand, nkept, sel_mode, keep_thres, need_sim, heap_ops, kth_area. */
int fslic_b200_debug_cca_counters(fslic_ctx* ctx, int32_t* out8, int image);

/* Diagnostics (contexts created with FSLIC_SELPROF=1 in the environment): 8 int64 words written by the
 * std::partial_sort replay of image `image`: total / filter / heap build / replay clocks, replay loop trips,
 * queued candidates, chunks, components. */
int fslic_b200_debug_select_profile(fslic_ctx* ctx, long long* out8, int image);

/* Milliseconds spent per stage in the last iterate() with collect_timing != 0. */
int fslic_b200_stage_ms(fslic_ctx* ctx, float* out_ms, int count);

/* Milliseconds of the connectivity stage's sub-sections in the last iterate() with collect_timing != 0 and fewer than
 * 4 images, in the reference's order and names (cca.cpp:194-263): build_disjoint_set, flatten, threshold_by_area,
 * sort, substitute, output.  Zeros when the stage was not timed (larger batches overlap the tail on a side stream). */
int fslic_b200_cca_stage_ms(fslic_ctx* ctx, float* out_ms, int count);

/* Geometry queries (S = (int16)sqrt(H*W/K), context.h:60; number of kernel launches per iterate). */
int fslic_b200_get_S(const fslic_ctx* ctx);
int fslic_b200_launches_last_iterate(const fslic_ctx* ctx);

/* Diagnostics: which assign kernel the last pass of the last iterate() used -- 5: the TMA-staged kernel
 * (k_assign5; needs W % 8 == 0 and subsample_stride 3), 4: the LDG kernel (k_assign_warp; any shape; forced
 * by the environment variable FSLIC_ASSIGN=4 at context creation), 0: the brute-force kernel / none yet. */
int fslic_b200_debug_assign_impl(const fslic_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* FSLIC_B200_H */
