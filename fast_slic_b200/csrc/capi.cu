// fast_slic_b200/csrc/capi.cu -- host orchestration + the extern "C" boundary (include/fslic_b200.h).
//
// Plays the role of BaseContext<uint16_t>::iterate (/root/reference/src/context.cpp:109-197) and of
// the Cython glue that drives it (cfast_slic.pyx:124-197): owns the scratch buffers, sequences the
// kernels on one stream, never touches the CPU for the data path.
#include <math.h>
#include <stdlib.h>
#include <new>
#include <cstring>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>  // library sort for the adjacency-graph utility only (not on the hot path)

#include "assign.cuh"
#include "assign5.cuh"
#include "graph.cuh"
#include "realdist.cuh"
#include "preempt.cuh"
#include "cca.cuh"
#include "common.cuh"
#include "lab.cuh"

#define SPT_MAX_ELEMS (128 * 1024)  // u16 elements per spatial patch buffer

typedef void (*assign_fn)(AssignParams, const uint32_t*, uint16_t*, const CInfo*, const int*, unsigned long long*,
                          const uint16_t*);
static assign_fn pick_assign(int TS, int stride, bool update);

typedef void (*assign5_fn)(const AssignParams, const CUtensorMap, const CUtensorMap, const uint32_t*, uint16_t*, const CInfo*,
                           const int*, unsigned long long*, const uint16_t*, fslic_cluster*, CInfo*, int*, unsigned int*);
static assign5_fn pick_assign5(int TS, bool update, int tps, bool fuse = false);

static thread_local std::string g_err;
static int set_err(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
// Every entry point runs on the context's device and puts the caller's current device back on return
// (a single-process multi-GPU PyTorch program must not find its current device changed behind its back).
struct DeviceGuard {
    int prev = -1;
    bool changed = false;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int dev) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) {
            err = cudaSetDevice(dev);
            changed = err == cudaSuccess;
        }
    }
    ~DeviceGuard() {
        if (changed) cudaSetDevice(prev);
    }
};
#define USE_DEVICE(dev)                                                                               \
    DeviceGuard dev_guard__(dev);                                                                     \
    if (dev_guard__.err != cudaSuccess)                                                               \
        return set_err(FSLIC_ECUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(dev_guard__.err))

#define CK(call)                                                                                      \
    do {                                                                                              \
        cudaError_t e__ = (call);                                                                     \
        if (e__ != cudaSuccess)                                                                       \
            return set_err(FSLIC_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e__));         \
    } while (0)

struct fslic_ctx {
    int device = 0, H = 0, W = 0, K = 0, maxB = 0, S = 0, N = 0;
    bool cca_only = false;  // fslic_b200_create_cca: connectivity scratch only
    int num_sms = 148;
    // tables
    uint16_t *d_gamma = nullptr, *d_labtbl = nullptr;
    LabConsts lc;
    // assign state
    uint32_t* quad = nullptr;      // [B][N]   Lab quad image
    uint16_t* labels = nullptr;    // [B][N]   pre-CCA labels
    CInfo* cinfo = nullptr;        // [B][K]
    unsigned long long* acc = nullptr;  // [B][K][4] packed sums (assign.cuh)
    int* cell_start = nullptr;     // [B][ncell+1]
    CInfo* cinfo_tmp = nullptr;    // [B][K] scratch of k_prepare (records by cluster index)
    int* cell_cnt = nullptr;       // [B][ncell+1] cell histogram of k_prepare2 (zero between launches)
    unsigned int* prep_tickets = nullptr;  // [B] arrival counters of k_prepare2 (zero between launches)
    uint16_t* sptable = nullptr;   // two linear spatial patches: [0] subsampled passes, [1] full pass
    int G = 1, cellW = 1, cellH = 1, ncell = 1;
    // cca state (sized for cca_batch images at a time)
    int cca_batch = 1;
    int* par = nullptr;            // [Bc][N]
    uint32_t* aux = nullptr;       // [Bc][N]  area at root pixel, then component number
    int* cleader = nullptr;        // [Bc][N]
    uint32_t* carea = nullptr;     // [Bc][N]
    uint16_t* cnew = nullptr;      // [Bc][N]
    uint16_t* fin = nullptr;       // [Bc][N]  (second half of the cnew allocation)
    int* rootbuf = nullptr;        // [Bc][N] ordered root lists of k_ccl_flatten
    int* blkcnt = nullptr;         // [Bc][nblk]
    int* blkoff = nullptr;         // [Bc][nblk]
    CcaCounters* counters = nullptr;  // [Bc]
    unsigned int* ahist = nullptr;    // [Bc][CCA_HIST] histogram of candidate areas
    unsigned long long* heap = nullptr;  // [Bc][Kheap]
    int heap_K = 0;
    // staging for the host entry points
    uint8_t* d_img = nullptr;
    fslic_cluster* d_cl = nullptr;
    uint16_t* d_lab = nullptr;
    cudaStream_t own_stream = nullptr, in_stream = nullptr, out_stream = nullptr, side_stream = nullptr;
    cudaEvent_t side_fork = nullptr, side_join = nullptr, tail_done = nullptr;
    // second lane of the blocking host path (the two halves of a batch overlap on the device)
    cudaStream_t own_stream2 = nullptr, side_stream2 = nullptr;
    cudaEvent_t side_fork2 = nullptr, side_join2 = nullptr, tail_done2 = nullptr, front_done = nullptr;
    // the `preemptive` option (preempt.cuh), allocated at the first such call
    uint8_t* pre_cellmap = nullptr;     // [B][ceil(H/2S) * ceil(W/2S)] active 2S x 2S cells
    int* pre_nactive = nullptr;         // [B] active clusters
    float preempt_l1 = 0.f;             // max(roundf(2 S thres), 1) of the call in progress
    long long* selprof = nullptr;       // FSLIC_SELPROF=1: 8 words per image written by k_cca_select (diagnostics)
    CcaCounters* h_counters = nullptr;  // pinned, 64 entries: lets the host path learn which images need the replay
    std::vector<cudaEvent_t> pipe_ev;  // [2 * chunks]: input-ready / compute-done events of iterate_host
    // timing
    cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // the reference's sub-sections of "cca" (cca.cpp:194-263): build_disjoint_set, flatten, threshold_by_area, sort,
    // substitute, output -- event-timed when collect_timing is on and the batch is not split across streams
    cudaEvent_t cev[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    float cca_ms[6] = {0, 0, 0, 0, 0, 0};
    bool cca_timing = false, cca_timed = false;
    float stage_ms[FSLIC_T_COUNT] = {0, 0, 0, 0, 0, 0};
    int last_launches = 0;
    int slice = 0;  // first image of the batch slice the front half (Lab + passes) currently works on
    int max_smem_optin = 0;
    // per-launch timing of the dominant kernel (k_assign_tiles on the subsampled passes)
    std::vector<cudaEvent_t> kev;
    int kev_used = 0;
    bool kev_on = false;
    bool pending = false;  // an iterate_host_async batch is in flight on this context's streams
    // small host batches replay one captured CUDA graph per call instead of ~45 launches (FSLIC_GRAPH=0 turns it off)
    bool graphs_enabled = true;
    cudaGraphExec_t gexec = nullptr;
    struct GraphKey {
        const void *img, *cl, *lab;
        int batch;
        fslic_params p;
        int manhattan;  // the spatial metric is baked into the captured kernels' parameters
    } gkey = {nullptr, nullptr, nullptr, 0, {0.f, 0.f, 0, 0, 0, 0}, 1}, gkey_seen = {nullptr, nullptr, nullptr, 0, {0.f, 0.f, 0, 0, 0, 0}, 1};
    int glaunches = 0;
    float assign_kernel_ms = 0.f;
    int assign_kernel_launches = 0;
    bool spt_valid = false, spt_has_sub = false;  // what c->sptable currently holds (build_patches)
    int spt_stride = 0;
    cudaStream_t spt_stream = nullptr;
    uint32_t spt_coef_bits = 0;
    bool spt_manhattan = true;
    // the reference's public context field manhattan_spatial_dist (context.h:35): L1 (default) or Euclidean spatial term;
    // read by every entry point when it enqueues work (fslic_b200_set_manhattan_spatial_dist)
    bool manhattan = true;
    int assign_impl = 5;       // 5: TMA-staged kernel where it applies (default), 4: always the LDG kernel (FSLIC_ASSIGN=4)
    int last_assign_impl = 0;  // which kernel the last subsampled / full pass used (tests, bench)
};

extern "C" const char* fslic_b200_last_error(void) { return g_err.c_str(); }
extern "C" const char* fslic_b200_version(void) { return "fast_slic_b200 0.1 (sm_100a)"; }
extern "C" int fslic_b200_sizeof_cluster(void) { return (int)sizeof(fslic_cluster); }
extern "C" int fslic_b200_get_S(const fslic_ctx* ctx) { return ctx ? ctx->S : -1; }
extern "C" int fslic_b200_launches_last_iterate(const fslic_ctx* ctx) { return ctx ? ctx->last_launches : -1; }
extern "C" int fslic_b200_debug_assign_impl(const fslic_ctx* ctx) { return ctx ? ctx->last_assign_impl : -1; }
extern "C" int fslic_b200_set_manhattan_spatial_dist(fslic_ctx* ctx, int manhattan) {
    if (!ctx) return set_err(FSLIC_EINVAL, "ctx is NULL");
    ctx->manhattan = manhattan != 0;
    return FSLIC_OK;
}

// ---- Lab tables: FastCIELabCvt ctor, /root/reference/src/cielab.h:297-305 ----------------------
// _srgb_gamma_tbl (cielab.h:22-279) is the sRGB inverse companding curve documented at
// cielab.h:12-20; it is regenerated here from that formula (bit-identical, checked in tests over the
// whole 2^24 colour cube against the compiled reference).
static void build_lab_tables(std::vector<uint16_t>& gamma, std::vector<uint16_t>& labtbl, LabConsts& lc) {
    static const float C[9] = {0.43395633f, 0.37621531f, 0.18984309f, 0.2126729f, 0.7151522f,
                               0.072175f,   0.01775782f, 0.1094756f,  0.87283638f};
    gamma.resize(256);
    labtbl.resize(8193);
    for (int i = 0; i < 256; i++) {
        const double v = i / 255.0;
        const double X = (v <= 0.04045) ? v / 12.92 : pow((v + 0.055) / 1.055, 2.4);
        gamma[i] = (uint16_t)(int)((float)X * 8192);
    }
    for (int i = 0; i < 9; i++) lc.Cb[i] = (int)roundf(C[i] * 65536);
    for (int i = 0; i <= 8192; i++) {
        const float v = (float)i / 8192;
        const float lo = 7.787f * v + 0.137931f;
        const float hi = powf(v, 0.333333f);
        labtbl[i] = (uint16_t)(int)roundf(((v > 0.008856f) ? hi : lo) * 8192);
    }
}

template <typename T>
static cudaError_t dalloc(T** p, size_t count) {
    return cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T) + 256);
}

extern "C" int fslic_b200_destroy(fslic_ctx* c) {
    if (!c) return FSLIC_OK;
    DeviceGuard dev_guard__(c->device);
    void* ptrs[] = {c->d_gamma, c->d_labtbl, c->quad,   c->labels,  c->cinfo,  c->acc,    c->cell_start,
                    c->cinfo_tmp, c->cell_cnt, c->prep_tickets, c->sptable, c->par,  c->aux,    c->cleader, c->carea,
                    c->cnew,    c->rootbuf, c->blkcnt, c->blkoff,  c->counters, c->ahist, c->heap, c->d_img,
                    c->d_cl,    c->d_lab};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    for (auto& e : c->ev)
        if (e) cudaEventDestroy(e);
    for (auto& e : c->cev)
        if (e) cudaEventDestroy(e);
    for (auto& e : c->kev) cudaEventDestroy(e);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    if (c->in_stream) cudaStreamDestroy(c->in_stream);
    if (c->out_stream) cudaStreamDestroy(c->out_stream);
    if (c->side_stream) cudaStreamDestroy(c->side_stream);
    if (c->side_fork) cudaEventDestroy(c->side_fork);
    if (c->side_join) cudaEventDestroy(c->side_join);
    if (c->tail_done) cudaEventDestroy(c->tail_done);
    if (c->own_stream2) cudaStreamDestroy(c->own_stream2);
    if (c->side_stream2) cudaStreamDestroy(c->side_stream2);
    for (cudaEvent_t e : {c->side_fork2, c->side_join2, c->tail_done2, c->front_done})
        if (e) cudaEventDestroy(e);
    if (c->gexec) cudaGraphExecDestroy(c->gexec);
    if (c->h_counters) cudaFreeHost(c->h_counters);
    if (c->selprof) cudaFree(c->selprof);
    if (c->pre_cellmap) cudaFree(c->pre_cellmap);
    if (c->pre_nactive) cudaFree(c->pre_nactive);
    for (auto& e : c->pipe_ev) cudaEventDestroy(e);
    delete c;
    return FSLIC_OK;
}

static int create_impl(int device, int H, int W, int K, int max_batch, bool cca_only, fslic_ctx** out) {
    if (!out) return set_err(FSLIC_EINVAL, "out is NULL");
    *out = nullptr;
    if (H <= 0 || W <= 0) return set_err(FSLIC_EINVAL, "H and W must be positive");
    if (K <= 0) return set_err(FSLIC_EINVAL, "num_components should be a non-negative integer");  // cfast_slic.pyx:26-27
    if (K >= 65534) return set_err(FSLIC_EINVAL, "num_components cannot exceed 65534");              // cfast_slic.pyx:24-25
    if (max_batch <= 0) return set_err(FSLIC_EINVAL, "max_batch must be positive");
    if ((long)H * W >= (1L << 30)) return set_err(FSLIC_EINVAL, "image too large (H*W must be < 2^30)");
    if (H > 32767 || W > 32767) return set_err(FSLIC_EINVAL, "H and W must fit int16 (the reference truncates centres to int16)");
    USE_DEVICE(device);
    fslic_ctx* c = new (std::nothrow) fslic_ctx();
    if (!c) return set_err(FSLIC_ENOMEM, "out of host memory");
    c->device = device;
    c->cca_only = cca_only;
    c->H = H; c->W = W; c->K = K; c->maxB = max_batch; c->N = H * W;
    c->S = (int)(int16_t)sqrt((double)(H * W / K));  // context.h:60 (integer division first)
    if (c->S < 1 && !cca_only) {  // the reference divides by zero here (PreemptiveGrid: ceil_int(W, 2*S), preemptive.h:37-38)
        delete c;
        return set_err(FSLIC_EINVAL, "num_components exceeds the number of pixels (S = 0): the reference crashes on this input");
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) {
        c->num_sms = prop.multiProcessorCount;
        c->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    }
    const size_t B = (size_t)max_batch, N = (size_t)c->N;
#define CKC(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            std::string m = std::string(#call) + ": " + cudaGetErrorString(e__);                   \
            fslic_b200_destroy(c);                                                                 \
            return set_err(e__ == cudaErrorMemoryAllocation ? FSLIC_ENOMEM : FSLIC_ECUDA, m);      \
        }                                                                                          \
    } while (0)
    std::vector<uint16_t> gamma, labtbl;
    build_lab_tables(gamma, labtbl, c->lc);
    CKC(dalloc(&c->d_gamma, 256));
    CKC(dalloc(&c->d_labtbl, 8200));
    CKC(cudaMemcpy(c->d_gamma, gamma.data(), 256 * 2, cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(c->d_labtbl, labtbl.data(), 8193 * 2, cudaMemcpyHostToDevice));

    // candidate cell grid: pitch G >= max(S,1), at most ~16K cells so the histogram fits in smem
    int G = c->S > 2 ? c->S : 2;  // >= 2 so that ceil(2^32/G) fits 32 bits (div_g)
    while ((long)ceil_div(H, G) * ceil_div(W, G) > 16000) G++;
    c->G = G; c->cellW = ceil_div(W, G); c->cellH = ceil_div(H, G); c->ncell = c->cellW * c->cellH;

    if (!cca_only) {  // assign state (a connectivity-only context needs none of it)
        CKC(dalloc(&c->quad, B * N));
        CKC(dalloc(&c->labels, B * N));
        CKC(dalloc(&c->cinfo, B * K));
        CKC(dalloc(&c->acc, B * K * 4));
        CKC(cudaMemset(c->acc, 0, B * K * 4 * sizeof(unsigned long long)));
        CKC(dalloc(&c->cell_start, B * (c->ncell + 1)));
        CKC(dalloc(&c->cinfo_tmp, B * K));
        CKC(dalloc(&c->cell_cnt, B * (c->ncell + 1)));
        CKC(cudaMemset(c->cell_cnt, 0, B * (c->ncell + 1) * sizeof(int)));
        CKC(dalloc(&c->prep_tickets, B));
        CKC(cudaMemset(c->prep_tickets, 0, B * sizeof(unsigned int)));
        CKC(dalloc(&c->sptable, (size_t)2 * SPT_MAX_ELEMS));
    }

    // CCA scratch: 26 B/pixel/image; cap the resident set at ~12 GB
    const size_t per_img = N * 26 + 4096;
    size_t bc = (12ull << 30) / per_img;
    if (bc < 1) bc = 1;
    if (bc > B) bc = B;
    if (const char* e = getenv("FSLIC_CCA_BATCH")) {  // test hook: force the sub-batched CCA path
        const long v = atol(e);
        if (v >= 1 && (size_t)v < bc) bc = (size_t)v;
    }
    c->cca_batch = (int)bc;
    if (const char* e = getenv("FSLIC_GRAPH")) c->graphs_enabled = atoi(e) != 0;
    const int nblk = ceil_div(c->N, CCA_BLOCK);
    CKC(dalloc(&c->par, bc * N));
    CKC(dalloc(&c->aux, bc * N));
    CKC(dalloc(&c->cleader, bc * N));
    CKC(dalloc(&c->carea, bc * N));
    CKC(dalloc(&c->cnew, 2 * bc * N));
    c->fin = c->cnew + bc * N;
    CKC(dalloc(&c->rootbuf, bc * N));  // (its own array: two halves of a batch may be in different phases at the same time)
    CKC(dalloc(&c->blkcnt, bc * nblk));
    CKC(dalloc(&c->blkoff, bc * nblk));
    CKC(dalloc(&c->counters, bc));
    CKC(cudaMemset(c->counters, 0, bc * sizeof(CcaCounters)));  // the diagnostics entry may read them before the first run
    CKC(dalloc(&c->ahist, bc * CCA_HIST));
    c->heap_K = 65536 + 8;
    CKC(dalloc(&c->heap, bc * (size_t)c->heap_K));
    for (auto& e : c->ev) CKC(cudaEventCreate(&e));
    for (auto& e : c->cev) CKC(cudaEventCreate(&e));
    CKC(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    CKC(cudaStreamCreateWithFlags(&c->in_stream, cudaStreamNonBlocking));
    CKC(cudaStreamCreateWithFlags(&c->out_stream, cudaStreamNonBlocking));
    CKC(cudaStreamCreateWithFlags(&c->side_stream, cudaStreamNonBlocking));
    CKC(cudaEventCreateWithFlags(&c->side_fork, cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&c->side_join, cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&c->tail_done, cudaEventDisableTiming));
    CKC(cudaStreamCreateWithFlags(&c->own_stream2, cudaStreamNonBlocking));
    CKC(cudaStreamCreateWithFlags(&c->side_stream2, cudaStreamNonBlocking));
    CKC(cudaEventCreateWithFlags(&c->side_fork2, cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&c->side_join2, cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&c->tail_done2, cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&c->front_done, cudaEventDisableTiming));
    CKC(cudaMallocHost(reinterpret_cast<void**>(&c->h_counters), 64 * sizeof(CcaCounters)));
    if (const char* e = getenv("FSLIC_SELPROF")) {
        if (atoi(e) != 0) {
            CKC(cudaMalloc(reinterpret_cast<void**>(&c->selprof), (size_t)c->cca_batch * 8 * sizeof(long long)));
            CKC(cudaMemset(c->selprof, 0, (size_t)c->cca_batch * 8 * sizeof(long long)));
        }
    }

    // opt in to large dynamic shared memory once
    for (int ts : {128, 192, 256, 384})
        for (int stride : {0, 1, 3})
            for (int upd = 0; upd < 2; upd++)
                CKC(cudaFuncSetAttribute(pick_assign(ts, stride, upd != 0), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         c->max_smem_optin - 1024));
    for (int ts : {128, 192, 256})
        for (int upd = 0; upd < 2; upd++)
            for (int tps : {1, 4})
                for (int fuse = 0; fuse <= upd; fuse++)
                    CKC(cudaFuncSetAttribute(pick_assign5(ts, upd != 0, tps, fuse != 0), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             c->max_smem_optin - 1024));
    if (const char* e = getenv("FSLIC_ASSIGN")) c->assign_impl = atoi(e) == 4 ? 4 : 5;
    CKC(cudaFuncSetAttribute(k_cca_select, cudaFuncAttributeMaxDynamicSharedMemorySize, c->max_smem_optin - 4 * 1024));
    CKC(cudaFuncSetAttribute(k_debug_heap_select, cudaFuncAttributeMaxDynamicSharedMemorySize, c->max_smem_optin - 4 * 1024));
    CKC(cudaFuncSetAttribute(k_prepare, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    CKC(cudaFuncSetAttribute(k_prepare2, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    CKC(cudaFuncSetAttribute(k_prepare3, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    CKC(cudaFuncSetAttribute(k_rgb_to_lab16, cudaFuncAttributeMaxDynamicSharedMemorySize, LAB16_SMEM));
    *out = c;
    return FSLIC_OK;
}

extern "C" int fslic_b200_create(int device, int H, int W, int K, int max_batch, fslic_ctx** out) {
    return create_impl(device, H, W, K, max_batch, false, out);
}

extern "C" int fslic_b200_create_cca(int device, int H, int W, int max_batch, fslic_ctx** out) {
    return create_impl(device, H, W, 1, max_batch, true, out);
}

static int check_batch(fslic_ctx* c, int batch, bool needs_assign_state = true) {
    if (!c) return set_err(FSLIC_EINVAL, "ctx is NULL");
    if (batch <= 0 || batch > c->maxB) return set_err(FSLIC_EINVAL, "batch out of range for this context");
    if (needs_assign_state && c->cca_only)
        return set_err(FSLIC_EINVAL, "this context was created by fslic_b200_create_cca: only enforce_connectivity is available");
    return FSLIC_OK;
}

extern "C" int fslic_b200_initialize_clusters(fslic_ctx* c, const uint8_t* d_images, fslic_cluster* d_clusters,
                                              int batch, void* stream) {
    int rc = check_batch(c, batch);
    if (rc) return rc;
    USE_DEVICE(c->device);
    dim3 grid(ceil_div(c->K, 128), batch);
    k_init_clusters<<<grid, 128, 0, (cudaStream_t)stream>>>(d_images, d_clusters, c->H, c->W, c->K, batch);
    CK(cudaGetLastError());
    return FSLIC_OK;
}

static int launch_lab(fslic_ctx* c, const uint8_t* d_images, uint32_t* quad, int batch, int convert_to_lab,
                      cudaStream_t st) {
    const long npix = (long)batch * c->N;
    long blocks = (npix / 4 + 255) / 256;
    const long cap = (long)c->num_sms * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    if (convert_to_lab && ((reinterpret_cast<uintptr_t>(d_images) | reinterpret_cast<uintptr_t>(quad)) & 15) == 0 && npix >= 4096) {
        // persistent CTAs: the 48 KB of tables are filled once per CTA
        long nb = (npix / 16 + 255) / 256;
        if (nb > (long)c->num_sms * 4) nb = (long)c->num_sms * 4;
        if (nb < 1) nb = 1;
        k_rgb_to_lab16<<<(int)nb, 256, LAB16_SMEM, st>>>(d_images, quad, npix, c->d_gamma, c->d_labtbl, c->lc);
    } else {
        k_rgb_to_quad<<<(int)blocks, 256, 0, st>>>(d_images, quad, npix, c->d_gamma, c->d_labtbl, c->lc, convert_to_lab);
    }
    CK(cudaGetLastError());
    return FSLIC_OK;
}

extern "C" int fslic_b200_rgb_to_quad(fslic_ctx* c, const uint8_t* d_images, uint8_t* d_quad_out, int batch,
                                      int convert_to_lab, void* stream) {
    int rc = check_batch(c, batch);
    if (rc) return rc;
    USE_DEVICE(c->device);
    return launch_lab(c, d_images, reinterpret_cast<uint32_t*>(d_quad_out), batch, convert_to_lab, (cudaStream_t)stream);
}

// ---- connectivity enforcement over `batch` images, chunked by cca_batch -------------------------
// Host-output hook of run_cca (iterate_host only): label maps are copied to the host as soon as they are final --
// for the images k_cca_threshold settled that is while the std::partial_sort replay of the others still runs.
struct HostOut {
    uint16_t* h_labels;      // destination of image 0 of this call
    cudaStream_t out_stream;
    bool done;               // set when run_cca issued the label copies itself
};

// `slot` / `lane`: the blocking host path runs the two halves of a batch as two independent calls that overlap on the
// device; each gets its own window of the scratch arrays (images slot .. slot + batch) and its own side stream / events.
static int run_cca(fslic_ctx* c, const uint16_t* d_in, uint16_t* d_out, int batch, int K, int thres, cudaStream_t st,
                   int* launches, HostOut* ho = nullptr, int slot = 0, int lane = 0) {
    const int N = c->N;
    if (slot != 0 && slot + batch > c->cca_batch) return set_err(FSLIC_EINVAL, "scratch window out of range");
    const size_t so = (size_t)slot;
    const int nblk_all = ceil_div(N, CCA_BLOCK);
    int* const x_par = c->par + so * N;
    uint32_t* const x_aux = c->aux + so * N;
    int* const x_cleader = c->cleader + so * N;
    uint32_t* const x_carea = c->carea + so * N;
    uint16_t* const x_cnew = c->cnew + so * N;
    uint16_t* const x_fin = c->fin + so * N;
    int* const x_rootbuf = c->rootbuf + so * N;
    int* const x_blkcnt = c->blkcnt + so * nblk_all;
    int* const x_blkoff = c->blkoff + so * nblk_all;
    CcaCounters* const x_counters = c->counters + so;
    unsigned int* const x_ahist = c->ahist + so * CCA_HIST;
    unsigned long long* const x_heap = c->heap + so * (size_t)c->heap_K;
    long long* const x_selprof = c->selprof ? c->selprof + 8 * so : nullptr;
    CcaCounters* const x_hcnt = c->h_counters + so;
    cudaStream_t const x_side = lane ? c->side_stream2 : c->side_stream;
    cudaEvent_t const x_fork = lane ? c->side_fork2 : c->side_fork, x_join = lane ? c->side_join2 : c->side_join,
                      x_tail = lane ? c->tail_done2 : c->tail_done;
    CcaParams cp;
    cp.H = c->H; cp.W = c->W; cp.N = N; cp.K = K; cp.thres = thres; cp.which = -1;
    cp.nblk = ceil_div(N, CCA_BLOCK);
    const size_t heap_bytes = (size_t)(2 * K + 4) * 8;  // live slots + the +infinity padding of the replay loop
    cp.heap_in_smem = heap_bytes + SEL_CHUNK * 8 <= (size_t)(c->max_smem_optin - 8 * 1024);
    static const int sel_sync = (getenv("FSLIC_SELSYNC") && atoi(getenv("FSLIC_SELSYNC")) == 0) ? 0 : 1;
    cp.sel_sync = sel_sync;
    if (K + 2 > c->heap_K) return set_err(FSLIC_EINVAL, "K too large for the selection heap");
    for (int b0 = 0; b0 < batch; b0 += c->cca_batch) {
        const int nb = (batch - b0 < c->cca_batch) ? (batch - b0) : c->cca_batch;
        const uint16_t* in = d_in + (size_t)b0 * N;
        uint16_t* out = d_out + (size_t)b0 * N;
        const bool timed = c->cca_timing && nb < 4 && batch <= c->cca_batch;  // one stream, one sub-batch
        c->cca_timed = timed;
        if (timed) CK(cudaEventRecord(c->cev[0], st));
        CK(cudaMemsetAsync(x_counters, 0, sizeof(CcaCounters) * nb, st));
        CK(cudaMemsetAsync(x_ahist, 0, sizeof(unsigned int) * CCA_HIST * nb, st));
        dim3 g(cp.nblk, nb);
        {
            const int ttx = ceil_div(c->W, CCL_T), tty = ceil_div(c->H, CCL_T);
            const long ntt = (long)ttx * tty * nb;
            k_ccl_tile<<<(int)((ntt + CCL_TW - 1) / CCL_TW), 32 * CCL_TW, 0, st>>>(cp, in, x_par, x_aux, ttx, tty, ntt);
        }
        {
            const int seam_px = ((c->W - 1) / CCL_T) * c->H + ((c->H - 1) / CCL_T) * c->W;
            if (seam_px > 0) {
                dim3 gs(ceil_div(seam_px, 256), nb);
                k_ccl_seams<<<gs, 256, 0, st>>>(cp, in, x_par);
            }
        }
        if (timed) CK(cudaEventRecord(c->cev[1], st));
        k_ccl_flatten<<<g, 256, 0, st>>>(cp, in, x_par, x_aux, x_blkcnt, x_rootbuf);
        k_scan_blocks<<<nb, 1024, 0, st>>>(x_blkcnt, x_blkoff, cp.nblk, cp.nblk, nullptr, 0, 1,
                                           &x_counters[0].ncomp, (int)(sizeof(CcaCounters) / sizeof(int)), nullptr, -1);
        // grids of the per-component walks: sized for full batches (a few CTAs per image); a small batch gets more
        // CTAs per image instead, it is all dependent-load latency there
        const int number_grid = nb >= 8 ? CCA_NUMBER_GRID : std::min(std::max(ceil_div(cp.nblk, 32), CCA_NUMBER_GRID), 64);
        k_ccl_number<<<dim3(number_grid, nb), CCA_BLOCK, 0, st>>>(cp, x_rootbuf, x_aux, x_blkcnt, x_blkoff, x_cleader, x_carea,
                                                                      x_counters, x_ahist);
        if (timed) CK(cudaEventRecord(c->cev[2], st));
        k_cca_threshold<<<nb, 1024, 0, st>>>(cp, x_carea, x_counters, x_ahist);
        if (timed) CK(cudaEventRecord(c->cev[3], st));
        // Everything after the threshold decision depends on the kept set.  For images k_cca_threshold settled
        // that is known now; for the (few) images whose ties need the sequential std::partial_sort replay it
        // is known only after k_cca_select, which keeps a handful of SMs busy for ~1 ms.  So for batches the
        // tail runs twice: for the settled images on a side stream concurrently with the replay, and for the
        // replayed images afterwards.
        auto tail = [&](int which, cudaStream_t ts) {
            CcaParams cq = cp;
            cq.which = which;
            const dim3 gk(std::min(cp.nblk, std::max(CCA_KEPT_GRID, 256 / nb)), nb);
            k_kept_count<<<gk, CCA_BLOCK, 0, ts>>>(cq, x_carea, x_counters, x_blkcnt);
            k_scan_blocks<<<nb, 1024, 0, ts>>>(x_blkcnt, x_blkoff, cp.nblk, 0, &x_counters[0].ncomp,
                                               (int)(sizeof(CcaCounters) / sizeof(int)), CCA_BLOCK,
                                               &x_counters[0].nkept, (int)(sizeof(CcaCounters) / sizeof(int)),
                                               x_counters, which);
            k_kept_label<<<gk, CCA_BLOCK, 0, ts>>>(cq, x_carea, x_counters, x_blkoff, x_cnew);
            int ab = ceil_div(N, 256 * (nb < 4 ? 2 : 8));
            if (ab > c->num_sms * 8) ab = c->num_sms * 8;
            dim3 ga(ab, nb);
            if (timed) cudaEventRecord(c->cev[4], ts);
            k_cca_absorb<<<ga, 256, 0, ts>>>(cq, x_par, x_aux, x_cleader, x_cnew, x_counters, x_fin);
            if (timed) cudaEventRecord(c->cev[5], ts);
            int ob = ceil_div(ceil_div(N, 8), 256);  // 8 pixels per thread on the vector path (any N works: grid-stride)
            if (ob > c->num_sms * 32) ob = c->num_sms * 32;
            dim3 go(ob, nb);
            k_cca_output<<<go, 256, 0, ts>>>(cq, x_par, x_fin, out, x_counters);
            if (timed) cudaEventRecord(c->cev[6], ts);
        };
        const bool split = nb >= 4;
        const bool early = split && ho && batch <= c->cca_batch && nb <= 64;
        if (early) {
            // the host path is synchronous anyway: wait for the threshold decision and read the per-image flags
            CK(cudaMemcpyAsync(x_hcnt, x_counters, sizeof(CcaCounters) * nb, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        }
        if (split) {
            CK(cudaEventRecord(x_fork, st));
            CK(cudaStreamWaitEvent(x_side, x_fork, 0));
            tail(0, x_side);
            CK(cudaEventRecord(x_join, x_side));
        }
        auto copy_runs = [&](int want) -> int {  // D2H of maximal runs of images whose need_sim flag == want
            int b = 0;
            while (b < nb) {
                if ((x_hcnt[b].need_sim != 0) != (want != 0)) { b++; continue; }
                int e = b;
                while (e < nb && (x_hcnt[e].need_sim != 0) == (want != 0)) e++;
                CK(cudaMemcpyAsync(ho->h_labels + (size_t)b * N, out + (size_t)b * N, (size_t)(e - b) * N * 2,
                                   cudaMemcpyDeviceToHost, ho->out_stream));
                b = e;
            }
            return FSLIC_OK;
        };
        if (early) {
            CK(cudaStreamWaitEvent(ho->out_stream, x_join, 0));
            int rc2 = copy_runs(0);
            if (rc2) return rc2;
        }
        k_cca_select<<<nb, 1024, SEL_CHUNK * 8 + (cp.heap_in_smem ? heap_bytes : 0), st>>>(cp, x_carea, x_counters, x_heap, x_selprof);
        tail(split ? 1 : -1, st);
        if (early) {
            CK(cudaEventRecord(x_tail, st));
            CK(cudaStreamWaitEvent(ho->out_stream, x_tail, 0));
            int rc2 = copy_runs(1);
            if (rc2) return rc2;
            ho->done = true;
        }
        if (split) {
            CK(cudaStreamWaitEvent(st, x_join, 0));
            if (launches) *launches += 5;
        }
        CK(cudaGetLastError());
        if (launches) *launches += 12;
    }
    return FSLIC_OK;
}

extern "C" int fslic_b200_enforce_connectivity(fslic_ctx* c, uint16_t* d_labels, int batch, int K, int min_threshold,
                                               void* stream) {
    int rc = check_batch(c, batch, false);
    if (rc) return rc;
    if (K <= 0) return FSLIC_OK;  // context.cpp:17
    if (K > 65535) return set_err(FSLIC_EINVAL, "K must fit the u16 label type");
    USE_DEVICE(c->device);
    return run_cca(c, d_labels, d_labels, batch, K, min_threshold, (cudaStream_t)stream, nullptr);
}

extern "C" int fslic_b200_debug_heap_select(fslic_ctx* c, const int32_t* d_area, int n, int middle, uint8_t* d_kept,
                                            void* stream) {
    if (!c) return set_err(FSLIC_EINVAL, "ctx is NULL");
    if (middle + 2 > c->heap_K || middle < 1 || n < 1) return set_err(FSLIC_EINVAL, "bad n/middle");
    USE_DEVICE(c->device);
    CK(cudaMemsetAsync(d_kept, 0, n, (cudaStream_t)stream));
    const size_t hb = (size_t)(2 * middle + 4) * 8;
    const int use_smem = hb + SEL_CHUNK * 8 <= (size_t)(c->max_smem_optin - 8 * 1024);
    k_debug_heap_select<<<1, 1024, SEL_CHUNK * 8 + (use_smem ? hb : 0), (cudaStream_t)stream>>>(reinterpret_cast<const uint32_t*>(d_area), n,
                                                                              middle, d_kept, c->heap, use_smem);
    CK(cudaGetLastError());
    return FSLIC_OK;
}

// per-slice views of the batched buffers (c->slice = first image of the slice)
#define SL_QUAD(c) ((c)->quad + (size_t)(c)->slice * (c)->N)
#define SL_LABELS(c) ((c)->labels + (size_t)(c)->slice * (c)->N)
#define SL_CINFO(c) ((c)->cinfo + (size_t)(c)->slice * (c)->K)
#define SL_CELLS(c) ((c)->cell_start + (size_t)(c)->slice * ((c)->ncell + 1))
#define SL_ACC(c) ((c)->acc + (size_t)(c)->slice * (c)->K * 4)

// ---- one assign pass (warp kernel, or the generic kernel when the patch cannot live in shared memory) ----
struct PassGeom {
    int R;
    bool fast;
    int OY, OX, TS, tbl_elems;
    size_t smem;
};

static PassGeom pass_geometry(const fslic_ctx* c, int stride) {
    PassGeom g;
    const int S = c->S;
    g.R = AS_R;
    g.OX = S + 31;
    g.OY = S + stride * (g.R - 1);
    // row pitch from a fixed menu so it is a compile-time constant of the kernel (immediate LDS offsets)
    const int need = 2 * g.OX + 1;
    g.TS = need <= 128 ? 128 : need <= 192 ? 192 : need <= 256 ? 256 : need <= 384 ? 384 : 0;
    const long elems = (long)(2 * g.OY + 1) * (g.TS ? g.TS : need);
    g.tbl_elems = (int)(elems < (1L << 30) ? elems : (1L << 30));
    g.smem = align_up((size_t)g.tbl_elems * 2, 16) + AS_STAGE_BYTES;
    g.fast = g.TS != 0 && elems <= SPT_MAX_ELEMS && g.smem <= (size_t)(c->max_smem_optin - 2 * 1024);
    return g;
}

// kernel menu: TS in {128,192,256,384} x (STRIDE 3 + update | STRIDE 1 no update | runtime stride)
template <int TS>
static assign_fn pick_assign_ts(int stride, bool update) {
    if (update) return stride == 3 ? k_assign_warp<TS, 3, true> : k_assign_warp<TS, 0, true>;
    return stride == 1 ? k_assign_warp<TS, 1, false> : k_assign_warp<TS, 0, false>;
}
static assign_fn pick_assign(int TS, int stride, bool update) {
    switch (TS) {
        case 128: return pick_assign_ts<128>(stride, update);
        case 192: return pick_assign_ts<192>(stride, update);
        case 256: return pick_assign_ts<256>(stride, update);
        default: return pick_assign_ts<384>(stride, update);
    }
}

// kernel menu of the TMA-staged kernel: TS in {128,192,256} x (stride 3 + update | stride 1, no update) x TPS in {1,4}
template <int TS>
static assign5_fn pick_assign5_ts(bool update, int tps, bool fuse) {
    if (update && fuse) return tps == 4 ? k_assign5<TS, 3, true, 4, true> : k_assign5<TS, 3, true, 1, true>;
    if (update) return tps == 4 ? k_assign5<TS, 3, true, 4> : k_assign5<TS, 3, true, 1>;
    return tps == 4 ? k_assign5<TS, 1, false, 4> : k_assign5<TS, 1, false, 1>;
}
static assign5_fn pick_assign5(int TS, bool update, int tps, bool fuse) {
    switch (TS) {
        case 128: return pick_assign5_ts<128>(update, tps, fuse);
        case 192: return pick_assign5_ts<192>(update, tps, fuse);
        default: return pick_assign5_ts<256>(update, tps, fuse);
    }
}

// cuTensorMapEncodeTiled through the runtime's driver entry point table (no link against libcuda)
typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static encode_tiled_fn tensor_map_encoder() {
    static encode_tiled_fn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<encode_tiled_fn>(p);
        cudaGetLastError();
    }
    return fn;
}

// 3-D view (x, sub-row, image) of the rows i = rem + sr * stride of a [B][H][W] array of `esize`-byte pixels;
// box = box_w columns x 4 sub-rows x 1 image.  Out-of-range parts of a box read as zero and are not written.
static bool make_subrow_map(CUtensorMap* m, CUtensorMapDataType dt, int esize, void* base, int H, int W, int B, int stride,
                            int rem, int nsub, int box_w) {
    encode_tiled_fn enc = tensor_map_encoder();
    if (!enc) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)nsub, (cuuint64_t)B};
    const cuuint64_t strides[2] = {(cuuint64_t)stride * W * esize, (cuuint64_t)H * W * esize};
    const cuuint32_t box[3] = {(cuuint32_t)box_w, 4u, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    unsigned char* p = static_cast<unsigned char*>(base) + (size_t)rem * W * esize;
    return enc(m, dt, 3, p, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static int build_patches(fslic_ctx* c, int stride, bool need_sub, float coef, cudaStream_t st, int* launches) {
    // The two patches depend on (S, stride, coef, metric) only: consecutive calls with the same parameters reuse them (two
    // launches less per call, four on the sliced host path).  Inside a stream capture they are always rebuilt, so a
    // replayed graph never depends on what an unrelated call left in the buffers.
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    uint32_t coef_bits;
    memcpy(&coef_bits, &coef, 4);
    const bool warm = cap == cudaStreamCaptureStatusNone && c->spt_valid && c->spt_stream == st && c->spt_stride == stride &&
                      c->spt_coef_bits == coef_bits && c->spt_manhattan == c->manhattan && (c->spt_has_sub || !need_sub);
    if (warm) return FSLIC_OK;
    c->spt_valid = true;
    c->spt_stream = st;  // a call on another stream is not ordered after this build: it rebuilds
    c->spt_stride = stride;
    c->spt_coef_bits = coef_bits;
    c->spt_manhattan = c->manhattan;
    c->spt_has_sub = need_sub;
    if (need_sub) {
        const PassGeom g = pass_geometry(c, stride);
        if (g.fast) {
            k_build_sptable<<<64, 256, 0, st>>>(c->sptable, c->S, g.OY, g.OX, g.TS, coef, !c->manhattan);
            if (launches) *launches += 1;
        }
    }
    const PassGeom gf = pass_geometry(c, 1);
    if (gf.fast) {
        k_build_sptable<<<64, 256, 0, st>>>(c->sptable + SPT_MAX_ELEMS, c->S, gf.OY, gf.OX, gf.TS, coef, !c->manhattan);
        if (launches) *launches += 1;
    }
    CK(cudaGetLastError());
    return FSLIC_OK;
}

// fuse_clusters / fused_out: when the TMA kernel takes an update pass of a small batch, its last CTA also does the
// bookkeeping for the NEXT pass (prepare_in_tail) on these cluster records; *fused_out tells the caller to skip k_prepare.
static int run_assign_pass(fslic_ctx* c, int batch, int stride, int rem, int cfg_stride, int fresh_from, bool update,
                           float coef, cudaStream_t st, int* launches, int variant = -1,
                           const fslic_cluster* d_clusters = nullptr, fslic_cluster* fuse_clusters = nullptr,
                           bool* fused_out = nullptr) {
    if (fused_out) *fused_out = false;
    if (variant == 3 && update) {  // the `preemptive` option (preempt.cuh); its full assign is the ordinary one
        AssignParams ap;
        memset(&ap, 0, sizeof(ap));
        ap.H = c->H; ap.W = c->W; ap.K = c->K; ap.S = c->S; ap.B = batch;
        ap.stride = stride; ap.rem = rem;
        ap.nsub = (c->H - rem + stride - 1) / stride;
        if (ap.nsub <= 0) return FSLIC_OK;
        ap.cfg_stride = cfg_stride; ap.fresh_from = fresh_from;
        ap.G = c->G; ap.cellW = c->cellW; ap.cellH = c->cellH; ap.ncell = c->ncell;
        ap.coef = coef;
        ap.euclid = !c->manhattan;
        const long px = (long)ap.nsub * c->W * batch;
        long grid = (px + 255) / 256;
        if (grid > (long)c->num_sms * 32) grid = (long)c->num_sms * 32;
        const int CW2 = ceil_div(c->W, 2 * c->S), ncell2 = CW2 * ceil_div(c->H, 2 * c->S);
        k_assign_preempt<true><<<(int)grid, 256, 0, st>>>(ap, SL_QUAD(c), SL_LABELS(c), SL_CINFO(c), SL_CELLS(c), d_clusters,
                                                          SL_ACC(c), c->pre_cellmap + (size_t)c->slice * ncell2, CW2, ncell2,
                                                          c->pre_nactive + c->slice);
        c->last_assign_impl = 0;
        if (launches) *launches += 1;
        CK(cudaGetLastError());
        return FSLIC_OK;
    }
    if (variant == 3) variant = -1;
    if (variant >= 0) {  // float-distance variants (realdist.cuh): one thread per pixel over the cell grid
        AssignParams ap;
        memset(&ap, 0, sizeof(ap));
        ap.H = c->H; ap.W = c->W; ap.K = c->K; ap.S = c->S; ap.B = batch;
        ap.stride = stride; ap.rem = rem;
        ap.nsub = (c->H - rem + stride - 1) / stride;
        if (ap.nsub <= 0) return FSLIC_OK;
        ap.cfg_stride = cfg_stride; ap.fresh_from = fresh_from;
        ap.G = c->G; ap.cellW = c->cellW; ap.cellH = c->cellH; ap.ncell = c->ncell;
        ap.coef = coef;
        ap.euclid = !c->manhattan;
        const long px = (long)ap.nsub * c->W * batch;
        long grid = (px + 255) / 256;
        if (grid > (long)c->num_sms * 32) grid = (long)c->num_sms * 32;
        const fslic_cluster* cl = d_clusters;
#define REAL_LAUNCH(V)                                                                                             \
    if (update)                                                                                                    \
        k_assign_real<V, true><<<(int)grid, 256, 0, st>>>(ap, SL_QUAD(c), SL_LABELS(c), SL_CINFO(c), SL_CELLS(c), cl, SL_ACC(c)); \
    else                                                                                                           \
        k_assign_real<V, false><<<(int)grid, 256, 0, st>>>(ap, SL_QUAD(c), SL_LABELS(c), SL_CINFO(c), SL_CELLS(c), cl, SL_ACC(c));
        if (variant == 0) { REAL_LAUNCH(0) } else if (variant == 1) { REAL_LAUNCH(1) } else { REAL_LAUNCH(2) }
#undef REAL_LAUNCH
        c->last_assign_impl = 0;
        if (launches) *launches += 1;
        CK(cudaGetLastError());
        return FSLIC_OK;
    }
    const PassGeom g = pass_geometry(c, stride);
    AssignParams ap;
    ap.H = c->H; ap.W = c->W; ap.K = c->K; ap.S = c->S; ap.B = batch;
    ap.stride = stride; ap.rem = rem;
    ap.nsub = (c->H - rem + stride - 1) / stride;
    if (ap.nsub <= 0) return FSLIC_OK;
    ap.cfg_stride = cfg_stride; ap.fresh_from = fresh_from;
    ap.G = c->G; ap.cellW = c->cellW; ap.cellH = c->cellH; ap.ncell = c->ncell;
    ap.Ginv = (uint32_t)(((1ull << 32) + (unsigned)c->G - 1) / (unsigned)c->G);
    ap.OY = g.OY; ap.OX = g.OX; ap.TS = g.TS; ap.tbl_elems = g.tbl_elems;
    ap.tiles_x = ceil_div(c->W, 32);
    ap.tiles_y = ceil_div(ap.nsub, g.R);
    ap.ntiles = ap.tiles_x * ap.tiles_y;
    ap.coef = coef;
    ap.euclid = !c->manhattan;
    ap.tps = AS_T;
    ap.fuse_prepare = 0;
    // The TMA-staged kernel: row strides of the tensor maps must be multiples of 16 bytes (W % 8 == 0 for the u16
    // labels), the sub-row pitch is an immediate of its patch loads (stride 3 with the update, 1 without), and its
    // per-warp shared blocks must fit beside the patch.  Everything else takes the LDG kernel below.
    bool use5 = g.fast && c->assign_impl == 5 && (c->W % 8) == 0 && g.TS <= 256 && (update ? stride == 3 : stride == 1) &&
                (long)ceil_div(c->W, 32) * ap.tiles_y * batch < (1L << 30) && tensor_map_encoder() != nullptr;
    int warps5 = 0;
    size_t smem5 = 0;
    if (use5) {
        const size_t tblb = align_up((size_t)g.tbl_elems * 2, 128);
        for (int w : {32, 16, 8}) {
            smem5 = tblb + (size_t)w * A5_WBLK;
            if (smem5 <= (size_t)(c->max_smem_optin - 1024)) {
                warps5 = w;
                break;
            }
        }
        if (!warps5) use5 = false;
    }
    if (use5) {
        // super tiles of 4 tiles when that still gives every warp of the grid work and the union list stays well below
        // its 32 slots; single tiles otherwise (single images, small S)
        const double est4 = (double)(2 * c->S + stride * 3 + 1) * (2 * c->S + 128) / ((double)c->S * c->S);
        const long supers4 = (long)ceil_div(ap.tiles_x, 4) * ap.tiles_y * batch;
        const int tps = (est4 <= 24.0 && supers4 >= (long)c->num_sms * warps5) ? 4 : 1;
        ap.tps = tps;
        CUtensorMap tmq, tml;
        uint32_t* qbase = SL_QUAD(c);
        uint16_t* lbase = SL_LABELS(c);
        if (!make_subrow_map(&tmq, CU_TENSOR_MAP_DATA_TYPE_UINT32, 4, qbase, c->H, c->W, batch, stride, rem, ap.nsub, 32 * tps) ||
            !make_subrow_map(&tml, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, lbase, c->H, c->W, batch, stride, rem, ap.nsub, 32 * tps)) {
            use5 = false;
        } else {
            const uint16_t* tbl = c->sptable + (update ? 0 : SPT_MAX_ELEMS);
            const long supers = (long)ceil_div(ap.tiles_x, tps) * ap.tiles_y * batch;
            // Super tiles are handed out statically, so a launch lasts ceil(supers / warps) rounds: with ~4 rounds (720p x 32)
            // a full grid of 32-warp CTAs idles a fifth of the time in the last round.  The kernel is issue bound and
            // saturates an SM with fewer warps, so take the warp count (>= 3/4 of the maximum) that wastes the least.
            if (supers > (long)c->num_sms * warps5) {
                int best_w = warps5;
                double best_cost = 1e30;
                for (int w = warps5; w >= (warps5 * 3) / 4; w--) {
                    const long workers = (long)c->num_sms * w;
                    const double cost = (double)((supers + workers - 1) / workers) * w;  // rounds x warps sharing an SM
                    if (cost < best_cost * 0.995) {
                        best_cost = cost;
                        best_w = w;
                    }
                }
                warps5 = best_w;
                smem5 = align_up((size_t)g.tbl_elems * 2, 128) + (size_t)warps5 * A5_WBLK;
            }
            else if (supers < (long)c->num_sms * warps5) {
                // not even one super tile per warp (single images): spread them over all SMs instead of filling a few
                const int w = std::max(4, (int)ceil_div((int)supers, c->num_sms));
                if (w < warps5) {
                    warps5 = w;
                    smem5 = align_up((size_t)g.tbl_elems * 2, 128) + (size_t)warps5 * A5_WBLK;
                }
            }
            static const bool fuse_allowed = !(getenv("FSLIC_FUSE") && atoi(getenv("FSLIC_FUSE")) == 0);
            const size_t tail_smem = prepare_tail_smem_bytes(c->K, c->ncell);
            if (update && fuse_clusters && fused_out && fuse_allowed && batch <= 2 && c->K <= 4096 &&
                tail_smem <= (size_t)(c->max_smem_optin - 1024)) {
                ap.fuse_prepare = 1;
                if (smem5 < tail_smem) smem5 = tail_smem;
                *fused_out = true;
            }
            const assign5_fn fn = pick_assign5(g.TS, update, tps, ap.fuse_prepare != 0);
            long grid = (supers + warps5 - 1) / warps5;
            if (grid > c->num_sms) grid = c->num_sms;
            // the warp-uniform walk constants (constant bank; see the note on code generation in assign5.cuh)
            ap.stx = ceil_div(ap.tiles_x, tps);
            ap.per_img = ap.stx * ap.tiles_y;
            ap.total = (int)supers;
            ap.wstride = (int)grid * warps5;
            ap.db = ap.wstride / ap.per_img;
            ap.dty = (ap.wstride % ap.per_img) / ap.stx;
            ap.dsx = (ap.wstride % ap.per_img) % ap.stx;
            ap.tbl_bytes = (uint32_t)align_up((size_t)g.tbl_elems * 2, 128);
            ap.cinfo_img_bytes = (uint32_t)c->K * (uint32_t)sizeof(CInfo);
            ap.cells_img_bytes = (uint32_t)(c->ncell + 1) * 4u;
            ap.acc_img_bytes = (uint32_t)c->K * 32u;
            cudaEvent_t e0 = nullptr, e1 = nullptr;
            if (c->kev_on && update) {
                while ((int)c->kev.size() < c->kev_used + 2) {
                    cudaEvent_t e;
                    CK(cudaEventCreate(&e));
                    c->kev.push_back(e);
                }
                e0 = c->kev[c->kev_used++];
                e1 = c->kev[c->kev_used++];
                CK(cudaEventRecord(e0, st));
            }
            fn<<<(int)grid, 32 * warps5, smem5, st>>>(ap, tmq, tml, qbase, lbase, SL_CINFO(c), SL_CELLS(c), SL_ACC(c), tbl,
                                                      fuse_clusters, SL_CINFO(c), SL_CELLS(c), c->prep_tickets + c->slice);
            if (e1) CK(cudaEventRecord(e1, st));
            c->last_assign_impl = 5;
        }
    }
    if (use5) {
        // launched above
    } else if (g.fast) {
        c->last_assign_impl = 4;
        const uint16_t* tbl = c->sptable + (update ? 0 : SPT_MAX_ELEMS);
        const assign_fn fn = pick_assign(g.TS, stride, update);
        int occ = 1;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, AS_THREADS, g.smem);
        if (occ < 1) occ = 1;
        long grid = (long)c->num_sms * occ;
        // small launches (single images): one tile per warp step so that every SM gets work
        ap.tps = ((long)ap.ntiles * batch < (long)c->num_sms * occ * AS_WARPS * AS_T) ? 1 : AS_T;
        const long supers = (long)ceil_div(ap.tiles_x, ap.tps) * ap.tiles_y * batch;
        const long need = (supers + AS_WARPS - 1) / AS_WARPS;
        if (grid > need) grid = need;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (c->kev_on && update) {
            while ((int)c->kev.size() < c->kev_used + 2) {
                cudaEvent_t e;
                CK(cudaEventCreate(&e));
                c->kev.push_back(e);
            }
            e0 = c->kev[c->kev_used++];
            e1 = c->kev[c->kev_used++];
            CK(cudaEventRecord(e0, st));
        }
        fn<<<(int)grid, AS_THREADS, g.smem, st>>>(ap, SL_QUAD(c), SL_LABELS(c), SL_CINFO(c), SL_CELLS(c), SL_ACC(c), tbl);
        if (e1) CK(cudaEventRecord(e1, st));
    } else {
        c->last_assign_impl = 0;
        const long px = (long)ap.nsub * c->W * batch;
        long grid = (px + 255) / 256;
        if (grid > (long)c->num_sms * 64) grid = (long)c->num_sms * 64;
        if (update)
            k_assign_generic<true><<<(int)grid, 256, 0, st>>>(ap, SL_QUAD(c), SL_LABELS(c), SL_CINFO(c), SL_CELLS(c),
                                                              SL_ACC(c));
        else
            k_assign_generic<false><<<(int)grid, 256, 0, st>>>(ap, SL_QUAD(c), SL_LABELS(c), SL_CINFO(c), SL_CELLS(c),
                                                               SL_ACC(c));
    }
    if (launches) *launches += 1;
    CK(cudaGetLastError());
    return FSLIC_OK;
}

static int run_prepare(fslic_ctx* c, fslic_cluster* d_clusters, int batch, int first, int finalize, cudaStream_t st,
                       int* launches, int noq = 0, int preempt = 0, int last = 0) {
    PrepParams pp;
    pp.H = c->H; pp.W = c->W; pp.K = c->K; pp.S = c->S; pp.T = 2 * c->S + 32;
    pp.G = c->G; pp.cellW = c->cellW; pp.cellH = c->cellH; pp.ncell = c->ncell;
    pp.first = first; pp.finalize = finalize; pp.last = last; pp.noq = noq;
    pp.preempt = preempt; pp.l1_thres = c->preempt_l1; pp.nactive = preempt ? c->pre_nactive + c->slice : nullptr;
    const size_t smem = (size_t)(c->ncell + 2) * sizeof(int);
    if (preempt) {  // k_prepare carries the option's bookkeeping; after an update k_preempt_mark derives the active set
        k_prepare<<<batch, 1024, smem, st>>>(pp, d_clusters, SL_ACC(c), SL_QUAD(c), SL_CINFO(c), SL_CELLS(c),
                                             c->cinfo_tmp + (size_t)c->slice * c->K);
        if (launches) *launches += 1;
        if (finalize && !last) {
            const int CW2 = ceil_div(c->W, 2 * c->S), ncell2 = CW2 * ceil_div(c->H, 2 * c->S);
            k_preempt_mark<<<batch, 1024, 0, st>>>(c->K, c->S, c->H, c->W, c->G, c->cellW, c->cellH, c->ncell, d_clusters, SL_CINFO(c),
                                                   SL_CELLS(c), c->pre_cellmap + (size_t)c->slice * ncell2, CW2, ncell2,
                                                   c->pre_nactive + c->slice);
            if (launches) *launches += 1;
        }
        CK(cudaGetLastError());
        return FSLIC_OK;
    }
    // k_prepare2 (one thread per cluster, several CTAs per image) is quicker for a handful of images (single image:
    // 0.412 vs 0.431 ms per blocking call); with a full batch its extra CTAs only contend (18 vs 13 us at 32 images)
    static const int forced = getenv("FSLIC_PREPARE") ? atoi(getenv("FSLIC_PREPARE")) : 0;
    const bool old_prepare = forced == 1 || (forced != 2 && batch >= 8);
    if (forced != 1 && forced != 2 && c->K <= 1024 * PREP3_PER)
        k_prepare3<<<batch, 1024, smem, st>>>(pp, d_clusters, SL_ACC(c), SL_QUAD(c), SL_CINFO(c), SL_CELLS(c));
    else if (old_prepare)
        k_prepare<<<batch, 1024, smem, st>>>(pp, d_clusters, SL_ACC(c), SL_QUAD(c), SL_CINFO(c), SL_CELLS(c),
                                             c->cinfo_tmp + (size_t)c->slice * c->K);
    else
        k_prepare2<<<dim3(ceil_div(c->K, 256), batch), 256, smem, st>>>(
            pp, d_clusters, SL_ACC(c), SL_QUAD(c), SL_CINFO(c), SL_CELLS(c), c->cinfo_tmp + (size_t)c->slice * c->K,
            c->cell_cnt + (size_t)c->slice * (c->ncell + 1), c->prep_tickets + c->slice);
    CK(cudaGetLastError());
    if (launches) *launches += 1;
    return FSLIC_OK;
}

// variant: as in iterate_front (-1 the default integer path); ContextRealDistL2 (1) keeps its squared term whatever the flag
static int check_params(const fslic_ctx* c, const fslic_params* p, float* coef_out, int variant = -1) {
    if (!p) return set_err(FSLIC_EINVAL, "params is NULL");
    if (p->subsample_stride <= 0 || p->subsample_stride > 255) return set_err(FSLIC_EINVAL, "subsample_stride must be in 1..255");
    if (p->max_iter < 0) return set_err(FSLIC_EINVAL, "max_iter must be >= 0");
    if (!(p->compactness >= 0.f)) return set_err(FSLIC_EINVAL, "compactness must be >= 0");
    const int S = c->S;
    const int color_shift = p->convert_to_lab ? 1 : 0;  // cielab.h:25,352 / context.cpp:127
    // BaseContext::set_spatial_patch, context.cpp:25-26 (same float operations, same order)
    float coef = 1.0f / ((float)S / p->compactness);
    coef *= (float)(1 << color_shift);
    // the largest patch value: coef * 2S (Manhattan), coef * hypotf(S, S) (Euclidean, context.cpp:36)
    const float reach = (!c->manhattan && variant != 1) ? (float)sqrt(2.0 * (double)S * (double)S) : (float)(2 * S);
    if (S > 0 && !(coef * reach < (float)(FSLIC_BIGSP - 766)))
        return set_err(FSLIC_ERANGE, "compactness too large: the u16 distance of the reference would overflow");
    if (S == 0) coef = 0.f;  // 1/(0/compactness) = inf in the reference; with S == 0 only m = 0 is ever used -> inf*0 = NaN -> (u16) UB; use 0
    *coef_out = coef;
    return FSLIC_OK;
}

// Front half of iterate (context.cpp:114-181): Lab LUT, max_iter x (assign + update), full assign, for the
// `batch` images starting at image `b0` of the context's buffers.  Leaves the pre-CCA labels in c->labels.
static int iterate_front(fslic_ctx* c, int b0, const uint8_t* d_images, fslic_cluster* d_clusters, int batch,
                         const fslic_params* p, float coef, cudaStream_t st, int* launches, bool timing,
                         bool lab_done = false, int variant = -1) {
    c->slice = b0;
    int rc = FSLIC_OK;
    if (!lab_done) rc = launch_lab(c, d_images, SL_QUAD(c), batch, p->convert_to_lab, st);  // else: the caller ran it
    if (rc) return rc;
    (*launches)++;
    if (timing) CK(cudaEventRecord(c->ev[1], st));
    const int stride = p->subsample_stride;
    const int noq = variant == 2 ? 1 : 0;
    const int preempt = variant == 3 ? 1 : 0;
    if (variant < 0 || preempt) {
        rc = build_patches(c, stride, p->max_iter > 0, coef, st, launches);
        if (rc) return rc;
    }
    const fslic_cluster* cl = d_clusters;  // the NoQ variant reads its float centroids from the cluster records themselves
    int rem = 0;
    bool prepared = false;  // the previous assign+update launch already did the bookkeeping in its tail
    for (int it = 0; it < p->max_iter; it++) {
        if (!prepared) {
            rc = run_prepare(c, d_clusters, batch, it == 0, it > 0, st, launches, noq, preempt, 0);
            if (rc) return rc;
        }
        rc = run_assign_pass(c, batch, stride, rem, stride, it, true, coef, st, launches, variant, cl,
                             variant < 0 ? d_clusters : nullptr, &prepared);
        if (rc) return rc;
        rem = (rem + 1) % stride;
    }
    if (timing) CK(cudaEventRecord(c->ev[2], st));
    if (!prepared) {
        rc = run_prepare(c, d_clusters, batch, p->max_iter == 0, p->max_iter > 0, st, launches, noq, preempt, 1);
        if (rc) return rc;
    }
    rc = run_assign_pass(c, batch, 1, 0, stride, p->max_iter < stride ? p->max_iter : stride, false, coef, st, launches,
                         variant, cl);
    c->slice = 0;
    return rc;
}

// Back half (context.cpp:191-194): connectivity enforcement of images [0, batch) of c->labels into d_labels.
static int iterate_back(fslic_ctx* c, uint16_t* d_labels, int batch, const fslic_params* p, cudaStream_t st, int* launches,
                        HostOut* ho = nullptr, int slot = 0, int lane = 0) {
    const int thres = (int)round((double)(c->S * c->S) * (double)p->min_size_factor);  // context.cpp:16
    return run_cca(c, c->labels + (size_t)slot * c->N, d_labels, batch, c->K, thres, st, launches, ho, slot, lane);
}

static int iterate_graphed(fslic_ctx* c, const uint8_t* d_images, fslic_cluster* d_clusters, uint16_t* d_labels, int batch,
                           const fslic_params* p, cudaStream_t st);

static int iterate_plain(fslic_ctx* c, const uint8_t* d_images, fslic_cluster* d_clusters, uint16_t* d_labels,
                         int batch, const fslic_params* p, void* stream, bool lab_done = false, int variant = -1) {
    int rc = check_batch(c, batch);
    if (rc) return rc;
    float coef;
    rc = check_params(c, p, &coef, variant);
    if (rc) return rc;
    USE_DEVICE(c->device);
    cudaStream_t st = (cudaStream_t)stream;
    int launches = 0;
    const bool timing = p->collect_timing != 0;
    c->kev_on = p->collect_timing >= 2;
    c->kev_used = 0;
    c->cca_timing = timing;
    c->cca_timed = false;
    if (timing) CK(cudaEventRecord(c->ev[0], st));
    rc = iterate_front(c, 0, d_images, d_clusters, batch, p, coef, st, &launches, timing, lab_done, variant);
    if (rc) return rc;
    if (timing) CK(cudaEventRecord(c->ev[3], st));
    rc = iterate_back(c, d_labels, batch, p, st, &launches);
    if (rc) return rc;
    if (timing) {
        CK(cudaEventRecord(c->ev[4], st));
        CK(cudaEventSynchronize(c->ev[4]));
        float ms;
        CK(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1])); c->stage_ms[FSLIC_T_CIELAB] = ms;
        CK(cudaEventElapsedTime(&ms, c->ev[1], c->ev[2])); c->stage_ms[FSLIC_T_ASSIGN] = ms;
        c->stage_ms[FSLIC_T_UPDATE] = 0.f;  // fused into assign
        CK(cudaEventElapsedTime(&ms, c->ev[2], c->ev[3])); c->stage_ms[FSLIC_T_FULL_ASSIGN] = ms;
        CK(cudaEventElapsedTime(&ms, c->ev[3], c->ev[4])); c->stage_ms[FSLIC_T_CCA] = ms;
        CK(cudaEventElapsedTime(&ms, c->ev[0], c->ev[4])); c->stage_ms[FSLIC_T_TOTAL] = ms;
        for (int i = 0; i < 6; i++) {
            c->cca_ms[i] = 0.f;
            if (c->cca_timed && cudaEventElapsedTime(&ms, c->cev[i], c->cev[i + 1]) == cudaSuccess) c->cca_ms[i] = ms;
        }
        cudaGetLastError();
        c->assign_kernel_ms = 0.f;
        c->assign_kernel_launches = 0;
        for (int i = 0; i + 1 < c->kev_used; i += 2) {
            CK(cudaEventElapsedTime(&ms, c->kev[i], c->kev[i + 1]));
            c->assign_kernel_ms += ms;
            c->assign_kernel_launches++;
        }
    }
    c->last_launches = launches;
    c->cca_timing = false;
    return FSLIC_OK;
}

extern "C" int fslic_b200_cca_stage_ms(fslic_ctx* c, float* out_ms, int count) {
    if (!c || !out_ms) return set_err(FSLIC_EINVAL, "NULL argument");
    for (int i = 0; i < count && i < 6; i++) out_ms[i] = c->cca_ms[i];
    return FSLIC_OK;
}

// Public entry.  A small batch is ~45 launches of kernels that each run a few microseconds: when the same buffers,
// batch and parameters come back (second consecutive call) the call is captured into a CUDA graph once and replayed
// from then on.  Needs a capturable stream (not the legacy default stream) and no timing; anything else launches plainly.
extern "C" int fslic_b200_iterate(fslic_ctx* c, const uint8_t* d_images, fslic_cluster* d_clusters, uint16_t* d_labels,
                                  int batch, const fslic_params* p, void* stream) {
    if (c && p && c->graphs_enabled && batch > 0 && batch < 4 && p->collect_timing == 0 && stream != nullptr) {
        fslic_ctx::GraphKey k;
        memset(&k, 0, sizeof(k));
        k.img = nullptr; k.cl = d_clusters; k.lab = d_labels; k.batch = batch; k.p = *p; k.manhattan = c->manhattan;
        const bool have = c->gexec && memcmp(&k, &c->gkey, sizeof(k)) == 0;
        const bool again = memcmp(&k, &c->gkey_seen, sizeof(k)) == 0;
        memcpy(&c->gkey_seen, &k, sizeof(k));
        if (have || again) return iterate_graphed(c, d_images, d_clusters, d_labels, batch, p, (cudaStream_t)stream);
    }
    return iterate_plain(c, d_images, d_clusters, d_labels, batch, p, stream);
}

// The float-distance contexts of the reference (context.h:100-125; cfast_slic.pyx:198-252): variant 0 = ContextRealDist
// ("standard"), 1 = ContextRealDistL2, 2 = ContextRealDistNoQ; the spatial metric is the context's manhattan flag.
extern "C" int fslic_b200_iterate_real(fslic_ctx* c, int variant, const uint8_t* d_images, fslic_cluster* d_clusters,
                                       uint16_t* d_labels, int batch, const fslic_params* p, void* stream) {
    if (variant < 0 || variant > 2) return set_err(FSLIC_EINVAL, "variant must be 0 (standard), 1 (l2) or 2 (noq)");
    return iterate_plain(c, d_images, d_clusters, d_labels, batch, p, stream, false, variant);
}

extern "C" int fslic_b200_iterate_preemptive(fslic_ctx* c, const uint8_t* d_images, fslic_cluster* d_clusters, uint16_t* d_labels,
                                             int batch, const fslic_params* p, float preemptive_thres, void* stream) {
    int rc = check_batch(c, batch);
    if (rc) return rc;
    if (c->S <= 0) return set_err(FSLIC_EINVAL, "preemptive needs S >= 1 (the reference divides by 2 S, preemptive.h:37-38)");
    if (!(preemptive_thres >= 0.f)) return set_err(FSLIC_EINVAL, "preemptive_thres must be >= 0");
    USE_DEVICE(c->device);
    if (!c->pre_cellmap) {
        const size_t ncell2 = (size_t)ceil_div(c->W, 2 * c->S) * ceil_div(c->H, 2 * c->S);
        uint8_t* cm = nullptr;
        int* na = nullptr;
        if (cudaMalloc(reinterpret_cast<void**>(&cm), ncell2 * c->maxB) != cudaSuccess ||
            cudaMalloc(reinterpret_cast<void**>(&na), sizeof(int) * c->maxB) != cudaSuccess) {
            if (cm) cudaFree(cm);
            cudaGetLastError();
            return set_err(FSLIC_ENOMEM, "out of device memory (preemptive scratch)");
        }
        c->pre_cellmap = cm;
        c->pre_nactive = na;
    }
    c->preempt_l1 = fmaxf(roundf((float)(2 * c->S) * preemptive_thres), 1.0f);  // preemptive.h:126
    return iterate_plain(c, d_images, d_clusters, d_labels, batch, p, stream, false, 3);
}

extern "C" int fslic_b200_assign_kernel_time(fslic_ctx* c, float* total_ms, int* launches) {
    if (!c || !total_ms || !launches) return set_err(FSLIC_EINVAL, "NULL argument");
    *total_ms = c->assign_kernel_ms;
    *launches = c->assign_kernel_launches;
    return FSLIC_OK;
}

extern "C" int fslic_b200_debug_cca_counters(fslic_ctx* c, int32_t* out8, int image) {
    if (!c || !out8 || image < 0 || image >= c->cca_batch) return set_err(FSLIC_EINVAL, "bad argument");
    USE_DEVICE(c->device);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(out8, c->counters + image, sizeof(CcaCounters), cudaMemcpyDeviceToHost));
    return FSLIC_OK;
}

extern "C" int fslic_b200_debug_select_profile(fslic_ctx* c, long long* out8, int image) {
    if (!c || !out8 || image < 0 || image >= c->cca_batch) return set_err(FSLIC_EINVAL, "bad argument");
    if (!c->selprof) return set_err(FSLIC_EINVAL, "the context was created without FSLIC_SELPROF=1");
    USE_DEVICE(c->device);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(out8, c->selprof + 8 * image, 8 * sizeof(long long), cudaMemcpyDeviceToHost));
    return FSLIC_OK;
}

extern "C" int fslic_b200_stage_ms(fslic_ctx* c, float* out_ms, int count) {
    if (!c || !out_ms) return set_err(FSLIC_EINVAL, "NULL argument");
    for (int i = 0; i < count && i < FSLIC_T_COUNT; i++) out_ms[i] = c->stage_ms[i];
    return FSLIC_OK;
}

extern "C" int fslic_b200_debug_stages(fslic_ctx* c, uint8_t* d_quad_out, uint16_t* d_precca_out, int batch,
                                       void* stream) {
    int rc = check_batch(c, batch);
    if (rc) return rc;
    USE_DEVICE(c->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (d_quad_out) CK(cudaMemcpyAsync(d_quad_out, c->quad, (size_t)batch * c->N * 4, cudaMemcpyDeviceToDevice, st));
    if (d_precca_out) CK(cudaMemcpyAsync(d_precca_out, c->labels, (size_t)batch * c->N * 2, cudaMemcpyDeviceToDevice, st));
    return FSLIC_OK;
}

// ---- host-buffer entry points (what the reference-facing plugin calls) --------------------------
static int ensure_staging(fslic_ctx* c) {
    if (c->d_img && c->d_cl && c->d_lab) return FSLIC_OK;
    const size_t B = (size_t)c->maxB, N = (size_t)c->N;
    // allocate into temporaries and commit all three together: a failed second or third allocation must not
    // leave a half-initialised staging set behind for the next call to trip over
    uint8_t* img = nullptr;
    fslic_cluster* cl = nullptr;
    uint16_t* lab = nullptr;
    cudaError_t e = dalloc(&img, B * N * 3);
    if (e == cudaSuccess) e = dalloc(&cl, B * c->K);
    if (e == cudaSuccess) e = dalloc(&lab, B * N);
    if (e != cudaSuccess) {
        if (img) cudaFree(img);
        if (cl) cudaFree(cl);
        if (lab) cudaFree(lab);
        cudaGetLastError();
        return set_err(e == cudaErrorMemoryAllocation ? FSLIC_ENOMEM : FSLIC_ECUDA,
                       std::string("staging buffers: ") + cudaGetErrorString(e));
    }
    c->d_img = img; c->d_cl = cl; c->d_lab = lab;
    return FSLIC_OK;
}

extern "C" int fslic_b200_initialize_clusters_host(fslic_ctx* c, const uint8_t* h_images, fslic_cluster* h_clusters,
                                                   int batch) {
    int rc = check_batch(c, batch);
    if (rc) return rc;
    USE_DEVICE(c->device);
    rc = ensure_staging(c);
    if (rc) return rc;
    cudaStream_t st = c->own_stream;
    const size_t ib = (size_t)batch * c->N * 3, cb = (size_t)batch * c->K * sizeof(fslic_cluster);
    CK(cudaMemcpyAsync(c->d_img, h_images, ib, cudaMemcpyHostToDevice, st));
    rc = fslic_b200_initialize_clusters(c, c->d_img, c->d_cl, batch, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(h_clusters, c->d_cl, cb, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return FSLIC_OK;
}

// One iterate() of a small batch on the context's own stream, replayed from a captured CUDA graph when the same
// buffers, batch and parameters come back (the host entry points always use the context's staging buffers, so
// that is every call after the first).  Falls back to plain launches if the capture fails.
static int iterate_graphed(fslic_ctx* c, const uint8_t* d_images, fslic_cluster* d_clusters, uint16_t* d_labels, int batch,
                           const fslic_params* p, cudaStream_t st) {
    // Only the Lab kernel reads the images: it is launched plainly, everything after it is the graph, so a caller that
    // feeds a new image buffer every call (a video stream) with the same cluster / label buffers still replays.
    int rc = check_batch(c, batch);
    if (rc) return rc;
    float coef;
    rc = check_params(c, p, &coef);
    if (rc) return rc;
    fslic_ctx::GraphKey k;
    memset(&k, 0, sizeof(k));
    k.img = nullptr; k.cl = d_clusters; k.lab = d_labels; k.batch = batch; k.p = *p; k.manhattan = c->manhattan;
    {
        USE_DEVICE(c->device);
        c->slice = 0;
        rc = launch_lab(c, d_images, c->quad, batch, p->convert_to_lab, st);
        if (rc) return rc;
    }
    if (c->gexec && memcmp(&k, &c->gkey, sizeof(k)) == 0) {
        CK(cudaGraphLaunch(c->gexec, st));
        c->last_launches = c->glaunches;
        return FSLIC_OK;
    }
    if (c->gexec) {
        cudaGraphExecDestroy(c->gexec);
        c->gexec = nullptr;
    }
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        cudaGetLastError();
        return iterate_plain(c, d_images, d_clusters, d_labels, batch, p, st, true);
    }
    rc = iterate_plain(c, d_images, d_clusters, d_labels, batch, p, st, true);
    cudaGraph_t g = nullptr;
    const cudaError_t e = cudaStreamEndCapture(st, &g);
    if (rc != FSLIC_OK || e != cudaSuccess || !g) {
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        if (rc != FSLIC_OK) return rc;  // a parameter error: nothing was launched
        return iterate_plain(c, d_images, d_clusters, d_labels, batch, p, st, true);
    }
    const cudaError_t ei = cudaGraphInstantiate(&c->gexec, g, 0);
    cudaGraphDestroy(g);
    if (ei != cudaSuccess) {
        c->gexec = nullptr;
        cudaGetLastError();
        return iterate_plain(c, d_images, d_clusters, d_labels, batch, p, st, true);
    }
    memcpy(&c->gkey, &k, sizeof(k));
    c->glaunches = c->last_launches;
    CK(cudaGraphLaunch(c->gexec, st));
    return FSLIC_OK;
}

// Enqueues H2D -> kernels -> D2H for one host batch on the context's three streams.  With may_sync the caller is
// going to block anyway, so the connectivity stage may read its per-image decisions back mid-way and start the
// label download of settled images early; without it nothing here waits for the device.
static int iterate_host_enqueue_body(fslic_ctx* c, const uint8_t* h_images, fslic_cluster* h_clusters,
                                     uint16_t* h_labels, int batch, const fslic_params* p, bool may_sync) {
    int rc = check_batch(c, batch);
    if (rc) return rc;
    USE_DEVICE(c->device);
    rc = ensure_staging(c);
    if (rc) return rc;
    if (c->pending) {  // one batch in flight per context: its staging buffers are about to be overwritten
        CK(cudaStreamSynchronize(c->out_stream));
        CK(cudaStreamSynchronize(c->own_stream));
        c->pending = false;
    }
    // Software pipeline over chunks of the batch: H2D(chunk i+1) | compute(chunk i) | D2H(chunk i-1) on three
    // streams, so for batches the PCIe copies hide behind the kernels (and vice versa).  With pinned host
    // buffers the copies are truly asynchronous; pageable buffers still work, just without overlap.
    const size_t N = (size_t)c->N;
    // chunks of 32: smaller chunks would pay the fixed latencies of the pipeline (notably the sequential
    // std::partial_sort replay of ambiguous images) once per chunk, which costs more than the overlap wins
    int chunk = batch < 32 ? batch : 32;
    if (const char* e = getenv("FSLIC_HOST_CHUNK")) {  // test hook: force the multi-chunk pipeline
        const int v = atoi(e);
        if (v >= 1 && v < chunk) chunk = v;
    }
    const int nchunks = (batch + chunk - 1) / chunk;
    while ((int)c->pipe_ev.size() < 3 * nchunks) {
        cudaEvent_t e;
        CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->pipe_ev.push_back(e);
    }
    fslic_params pp = *p;
    if (nchunks > 1) pp.collect_timing = 0;  // per-stage timings are only meaningful for an unchunked run
    const bool trace = may_sync && getenv("FSLIC_TRACE") != nullptr;
    std::vector<cudaEvent_t> tev;
    if (trace) {
        tev.resize(1 + 4 * nchunks);
        for (auto& e : tev) cudaEventCreate(&e);
        cudaEventRecord(tev[0], c->in_stream);
    }
    for (int k = 0; k < nchunks; k++) {
        const int b0 = k * chunk, nb = (batch - b0 < chunk) ? (batch - b0) : chunk;
        // Upload in two halves: the front half of the pipeline (Lab + passes) of the first half runs while the
        // second half is still on the wire; the back half (connectivity enforcement, whose replay latency is per
        // launch, not per image) then runs once over the whole chunk.
        bool labels_copied = false;
        static const bool no_split = getenv("FSLIC_HOST_SPLIT") && atoi(getenv("FSLIC_HOST_SPLIT")) == 0;
        if (nb >= 8 && !no_split) {
            float coef;
            rc = check_params(c, &pp, &coef);
            if (rc) return rc;
            int launches = 0;
            c->kev_on = false;  // per-launch kernel timing belongs to fslic_b200_iterate(collect_timing >= 2) only
            c->kev_used = 0;
            const int h0 = nb / 2;
            static const bool no_lanes = getenv("FSLIC_HOST_LANES") && atoi(getenv("FSLIC_HOST_LANES")) == 0;
            if (may_sync && !no_lanes && nchunks == 1 && nb >= 16 && nb <= c->cca_batch && nb <= 64) {
                // Blocking call: the caller waits anyway, so the two halves run as two independent pipelines that overlap
                // on the device -- half A's connectivity stage (incl. the ~0.7 ms std::partial_sort replay of its ambiguous
                // images, a handful of SMs) and its label download run while half B is still on the wire / in its assign
                // passes.  Each half has its own compute + side stream and its own window of the scratch arrays.
                for (int hpart = 0; hpart < 2; hpart++) {
                    const int s0 = b0 + (hpart ? h0 : 0), sn = hpart ? nb - h0 : h0;
                    CK(cudaMemcpyAsync(c->d_img + (size_t)s0 * N * 3, h_images + (size_t)s0 * N * 3, (size_t)sn * N * 3,
                                       cudaMemcpyHostToDevice, c->in_stream));
                    CK(cudaMemcpyAsync(c->d_cl + (size_t)s0 * c->K, h_clusters + (size_t)s0 * c->K,
                                       (size_t)sn * c->K * sizeof(fslic_cluster), cudaMemcpyHostToDevice, c->in_stream));
                    CK(cudaEventRecord(hpart ? c->pipe_ev[3 * k] : c->pipe_ev[3 * k + 2], c->in_stream));
                }
                for (int hpart = 0; hpart < 2; hpart++) {  // both front halves first: nothing in them waits for the host
                    const int s0 = b0 + (hpart ? h0 : 0), sn = hpart ? nb - h0 : h0;
                    cudaStream_t cs = hpart ? c->own_stream2 : c->own_stream;
                    CK(cudaStreamWaitEvent(cs, hpart ? c->pipe_ev[3 * k] : c->pipe_ev[3 * k + 2], 0));
                    // (the second front half starts behind the first: they share the cached spatial patches, which the first
                    //  call may still be building, and the first half's data is there earlier anyway)
                    if (hpart) CK(cudaStreamWaitEvent(cs, c->front_done, 0));
                    rc = iterate_front(c, s0 - b0, c->d_img + (size_t)s0 * N * 3, c->d_cl + (size_t)s0 * c->K, sn, &pp, coef, cs,
                                       &launches, false);
                    if (rc) return rc;
                    if (!hpart) CK(cudaEventRecord(c->front_done, cs));
                }
                for (int hpart = 0; hpart < 2; hpart++) {  // back halves: each reads its per-image decisions back mid-way
                    const int s0 = b0 + (hpart ? h0 : 0), sn = hpart ? nb - h0 : h0;
                    cudaStream_t cs = hpart ? c->own_stream2 : c->own_stream;
                    HostOut ho;
                    ho.h_labels = h_labels + (size_t)s0 * N;
                    ho.out_stream = c->out_stream;
                    ho.done = false;
                    rc = iterate_back(c, c->d_lab + (size_t)s0 * N, sn, &pp, cs, &launches, &ho, s0 - b0, hpart);
                    if (rc) return rc;
                    // clusters of this half (and its labels if run_cca did not download them itself)
                    CK(cudaEventRecord(c->pipe_ev[3 * k + 1], cs));
                    CK(cudaStreamWaitEvent(c->out_stream, c->pipe_ev[3 * k + 1], 0));
                    if (!ho.done)
                        CK(cudaMemcpyAsync(h_labels + (size_t)s0 * N, c->d_lab + (size_t)s0 * N, (size_t)sn * N * 2,
                                           cudaMemcpyDeviceToHost, c->out_stream));
                    CK(cudaMemcpyAsync(h_clusters + (size_t)s0 * c->K, c->d_cl + (size_t)s0 * c->K,
                                       (size_t)sn * c->K * sizeof(fslic_cluster), cudaMemcpyDeviceToHost, c->out_stream));
                }
                c->last_launches = launches;
                c->pending = true;
                CK(cudaStreamSynchronize(c->out_stream));
                CK(cudaStreamSynchronize(c->own_stream));
                CK(cudaStreamSynchronize(c->own_stream2));
                c->pending = false;
                return FSLIC_OK;
            }
            for (int hpart = 0; hpart < 2; hpart++) {
                const int s0 = b0 + (hpart ? h0 : 0), sn = hpart ? nb - h0 : h0;
                CK(cudaMemcpyAsync(c->d_img + (size_t)s0 * N * 3, h_images + (size_t)s0 * N * 3, (size_t)sn * N * 3,
                                   cudaMemcpyHostToDevice, c->in_stream));
                CK(cudaMemcpyAsync(c->d_cl + (size_t)s0 * c->K, h_clusters + (size_t)s0 * c->K,
                                   (size_t)sn * c->K * sizeof(fslic_cluster), cudaMemcpyHostToDevice, c->in_stream));
                cudaEvent_t ev = hpart ? c->pipe_ev[3 * k] : c->pipe_ev[3 * k + 2];
                CK(cudaEventRecord(ev, c->in_stream));
                if (trace && hpart == 1) cudaEventRecord(tev[1 + 4 * k], c->in_stream);
                CK(cudaStreamWaitEvent(c->own_stream, ev, 0));
                if (trace && hpart == 0) cudaEventRecord(tev[2 + 4 * k], c->own_stream);
                // slice s0 - b0 of the context buffers <-> images s0 .. s0+sn of this chunk
                rc = iterate_front(c, s0 - b0, c->d_img + (size_t)s0 * N * 3, c->d_cl + (size_t)s0 * c->K, sn, &pp, coef,
                                   c->own_stream, &launches, false);
                if (rc) return rc;
            }
            HostOut ho;
            ho.h_labels = h_labels + (size_t)b0 * N;
            ho.out_stream = c->out_stream;
            ho.done = false;
            rc = iterate_back(c, c->d_lab + (size_t)b0 * N, nb, &pp, c->own_stream, &launches, may_sync ? &ho : nullptr);
            if (rc) return rc;
            labels_copied = ho.done;
            c->last_launches = launches;
        } else {
        CK(cudaMemcpyAsync(c->d_img + (size_t)b0 * N * 3, h_images + (size_t)b0 * N * 3, (size_t)nb * N * 3,
                           cudaMemcpyHostToDevice, c->in_stream));
        CK(cudaMemcpyAsync(c->d_cl + (size_t)b0 * c->K, h_clusters + (size_t)b0 * c->K,
                           (size_t)nb * c->K * sizeof(fslic_cluster), cudaMemcpyHostToDevice, c->in_stream));
        CK(cudaEventRecord(c->pipe_ev[3 * k], c->in_stream));
        if (trace) cudaEventRecord(tev[1 + 4 * k], c->in_stream);
        CK(cudaStreamWaitEvent(c->own_stream, c->pipe_ev[3 * k], 0));
        if (trace) cudaEventRecord(tev[2 + 4 * k], c->own_stream);
        if (c->graphs_enabled && nb < 4 && nchunks == 1 && pp.collect_timing == 0)  // nb < 4: one stream, no host sync inside
            rc = iterate_graphed(c, c->d_img, c->d_cl, c->d_lab, nb, &pp, c->own_stream);
        else
            rc = iterate_plain(c, c->d_img + (size_t)b0 * N * 3, c->d_cl + (size_t)b0 * c->K, c->d_lab + (size_t)b0 * N, nb,
                                    &pp, c->own_stream);
        if (rc) return rc;
        }
        CK(cudaEventRecord(c->pipe_ev[3 * k + 1], c->own_stream));
        if (trace) cudaEventRecord(tev[3 + 4 * k], c->own_stream);
        CK(cudaStreamWaitEvent(c->out_stream, c->pipe_ev[3 * k + 1], 0));
        if (!labels_copied)
            CK(cudaMemcpyAsync(h_labels + (size_t)b0 * N, c->d_lab + (size_t)b0 * N, (size_t)nb * N * 2, cudaMemcpyDeviceToHost,
                               c->out_stream));
        CK(cudaMemcpyAsync(h_clusters + (size_t)b0 * c->K, c->d_cl + (size_t)b0 * c->K,
                           (size_t)nb * c->K * sizeof(fslic_cluster), cudaMemcpyDeviceToHost, c->out_stream));
        if (trace) cudaEventRecord(tev[4 + 4 * k], c->out_stream);
    }
    c->pending = true;
    if (!may_sync) return FSLIC_OK;
    CK(cudaStreamSynchronize(c->out_stream));
    CK(cudaStreamSynchronize(c->own_stream));
    c->pending = false;
    if (trace) {
        float ms;
        for (int k = 0; k < nchunks; k++) {
            float a, b2, c2, d2;
            cudaEventElapsedTime(&a, tev[0], tev[1 + 4 * k]);
            cudaEventElapsedTime(&b2, tev[0], tev[2 + 4 * k]);
            cudaEventElapsedTime(&c2, tev[0], tev[3 + 4 * k]);
            cudaEventElapsedTime(&d2, tev[0], tev[4 + 4 * k]);
            fprintf(stderr, "[fslic trace] chunk %d: h2d done %.3f | compute %.3f..%.3f | d2h done %.3f ms\n", k, a, b2, c2, d2);
        }
        (void)ms;
        for (auto e : tev) cudaEventDestroy(e);
    }
    return FSLIC_OK;
}

static int iterate_host_enqueue(fslic_ctx* c, const uint8_t* h_images, fslic_cluster* h_clusters, uint16_t* h_labels,
                                int batch, const fslic_params* p, bool may_sync) {
    const int rc = iterate_host_enqueue_body(c, h_images, h_clusters, h_labels, batch, p, may_sync);
    if (rc != FSLIC_OK && c && c->in_stream) {
        // an error after copies / kernels were enqueued: nothing may stay in flight on the staging buffers or the
        // caller's host buffers once the error is reported
        const std::string keep = g_err;
        DeviceGuard g(c->device);
        cudaStreamSynchronize(c->in_stream);
        cudaStreamSynchronize(c->own_stream);
        cudaStreamSynchronize(c->side_stream);
        if (c->own_stream2) cudaStreamSynchronize(c->own_stream2);
        if (c->side_stream2) cudaStreamSynchronize(c->side_stream2);
        cudaStreamSynchronize(c->out_stream);
        cudaGetLastError();
        c->pending = false;
        g_err = keep;
    }
    return rc;
}

extern "C" int fslic_b200_iterate_host(fslic_ctx* c, const uint8_t* h_images, fslic_cluster* h_clusters,
                                       uint16_t* h_labels, int batch, const fslic_params* p) {
    return iterate_host_enqueue(c, h_images, h_clusters, h_labels, batch, p, true);
}

extern "C" int fslic_b200_iterate_host_async(fslic_ctx* c, const uint8_t* h_images, fslic_cluster* h_clusters,
                                             uint16_t* h_labels, int batch, const fslic_params* p) {
    return iterate_host_enqueue(c, h_images, h_clusters, h_labels, batch, p, false);
}

extern "C" int fslic_b200_wait(fslic_ctx* c) {
    if (!c) return set_err(FSLIC_EINVAL, "ctx is NULL");
    if (!c->pending) return FSLIC_OK;
    USE_DEVICE(c->device);
    CK(cudaStreamSynchronize(c->out_stream));
    CK(cudaStreamSynchronize(c->own_stream));
    c->pending = false;
    return FSLIC_OK;
}

// ---- consumers of the label map (SURVEY.md 8(f) rows 1-2): stateless, device pointers, caller-provided scratch ------
static uint32_t conn_table_size(int K) {
    uint32_t t = 4096;
    while (t < 32u * (uint32_t)K) t <<= 1;  // a superpixel map has ~3 distinct adjacent pairs per label
    return t;
}
static size_t conn_sort_temp_bytes(uint32_t T) {
    size_t bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                    (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)T);
    return bytes;
}

extern "C" size_t fslic_b200_connectivity_scratch_bytes(int K) {
    if (K <= 0) return 256;
    const size_t T = conn_table_size(K);
    return align_up(T * 4, 256) * 2 + align_up(T * 8, 256) * 2 + align_up(conn_sort_temp_bytes((uint32_t)T), 256) + 256;
}

extern "C" int fslic_b200_get_connectivity(int device, int H, int W, int K, const uint16_t* d_labels, int32_t* d_counts,
                                           uint32_t* d_neighbors, void* d_scratch, size_t scratch_bytes, void* stream) {
    if (H <= 0 || W <= 0 || K <= 0 || K > 65535) return set_err(FSLIC_EINVAL, "bad H, W or K");
    if (!d_labels || !d_counts || !d_neighbors || !d_scratch) return set_err(FSLIC_EINVAL, "NULL argument");
    if (scratch_bytes < fslic_b200_connectivity_scratch_bytes(K)) return set_err(FSLIC_EINVAL, "scratch too small");
    USE_DEVICE(device);
    cudaStream_t st = (cudaStream_t)stream;
    const uint32_t T = conn_table_size(K);
    unsigned char* p = static_cast<unsigned char*>(d_scratch);
    uint32_t* tkey = reinterpret_cast<uint32_t*>(p); p += align_up((size_t)T * 4, 256);
    uint32_t* skey = reinterpret_cast<uint32_t*>(p); p += align_up((size_t)T * 4, 256);
    unsigned long long* tord = reinterpret_cast<unsigned long long*>(p); p += align_up((size_t)T * 8, 256);
    unsigned long long* sord = reinterpret_cast<unsigned long long*>(p); p += align_up((size_t)T * 8, 256);
    size_t temp_bytes = conn_sort_temp_bytes(T);
    void* temp = p; p += align_up(temp_bytes, 256);
    int* overflow = reinterpret_cast<int*>(p);
    CK(cudaMemsetAsync(tkey, 0xff, (size_t)T * 4, st));
    CK(cudaMemsetAsync(tord, 0xff, (size_t)T * 8, st));
    CK(cudaMemsetAsync(overflow, 0, 4, st));
    CK(cudaMemsetAsync(d_counts, 0, (size_t)K * 4, st));
    CK(cudaMemsetAsync(d_neighbors, 0, (size_t)K * CONN_MAX * 4, st));
    if (H > 1 && W > 1) {
        const long n = (long)(H - 1) * (W - 1);
        long blocks = (n + 255) / 256;
        if (blocks > 148 * 16) blocks = 148 * 16;
        k_conn_discover<<<(int)blocks, 256, 0, st>>>(d_labels, H, W, K, tkey, tord, T - 1, overflow);
        int h_overflow = 0;
        CK(cudaMemcpyAsync(&h_overflow, overflow, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (h_overflow) {
            k_conn_scan<<<1, 32, 0, st>>>(d_labels, H, W, K, d_counts, d_neighbors);
        } else {
            if (cub::DeviceRadixSort::SortPairs(temp, temp_bytes, tord, sord, tkey, skey, (int)T, 0, 64, st) != cudaSuccess)
                return set_err(FSLIC_ECUDA, "radix sort of the pair table failed");
            k_conn_walk<<<1, 32, 0, st>>>(sord, skey, T, K, d_counts, d_neighbors);
        }
    }
    CK(cudaGetLastError());
    return FSLIC_OK;
}

extern "C" int fslic_b200_get_mask_density(int device, int H, int W, int K, const fslic_cluster* d_clusters,
                                           const uint16_t* d_labels, const uint8_t* d_mask, uint8_t* d_densities,
                                           int32_t* d_scratch, void* stream) {
    if (H <= 0 || W <= 0 || K <= 0 || K > 65535) return set_err(FSLIC_EINVAL, "bad H, W or K");
    if (!d_clusters || !d_labels || !d_mask || !d_densities || !d_scratch) return set_err(FSLIC_EINVAL, "NULL argument");
    USE_DEVICE(device);
    cudaStream_t st = (cudaStream_t)stream;
    const long n = (long)H * W;
    CK(cudaMemsetAsync(d_scratch, 0, (size_t)K * 4, st));
    long blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    k_mask_sum<<<(int)blocks, 256, 0, st>>>(d_labels, d_mask, n, K, d_scratch);
    k_density_final<<<ceil_div(K, 256), 256, 0, st>>>(d_scratch, d_clusters, K, d_densities);
    CK(cudaGetLastError());
    return FSLIC_OK;
}

extern "C" int fslic_b200_cluster_density_to_mask(int device, int H, int W, int K, const uint16_t* d_labels,
                                                  const uint8_t* d_densities, uint8_t* d_result, void* stream) {
    if (H <= 0 || W <= 0 || K <= 0 || K > 65535) return set_err(FSLIC_EINVAL, "bad H, W or K");
    if (!d_labels || !d_densities || !d_result) return set_err(FSLIC_EINVAL, "NULL argument");
    USE_DEVICE(device);
    const long n = (long)H * W;
    long blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    k_density_broadcast<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(d_labels, d_densities, n, K, d_result);
    CK(cudaGetLastError());
    return FSLIC_OK;
}
