// fast_slic_b200/csrc/assign.cuh -- the assign + update hot loop.
//
// Replaces BaseContext::assign / assign_clusters / update of the reference
// (/root/reference/src/context.cpp:200-243, 259-298, 302-387; AVX2 form arch/x64/avx2.h:11-185).
//
// The reference is cluster-centric: every cluster scatters into its (2S+1)^2 window with a strict
// `<` against a per-pixel running minimum; ties are therefore won by the cluster visited first,
// i.e. by the smaller (phase, k) where phase = 2*((cy/T)&1) + ((cx/T)&1), T = 2S+32
// (context.cpp:214-242).  On the GPU the loop is turned inside out: every pixel gathers over the
// clusters whose window covers it and minimises the packed key  d << 16 | rank,  rank being the
// candidate's position in the (phase, k)-sorted candidate list of its CTA tile.  Pixels no window
// covers keep their previous label (context.cpp:289-294 never fires for them).
#pragma once
#include "common.cuh"

// ---------------------------------------------------------------------------------------------
// k_prepare: per-image bookkeeping between two assign passes (one CTA per image).
//   1. finalise the previous update: integer round-divide of the accumulated sums
//      (context.cpp:356-374, round_int fast-slic-common.h:63-65) and clear the accumulators;
//   2. first pass only: re-seed the cluster colour from the quad image (context.cpp:128-135);
//   3. clamp centres into the image (context.cpp:209-212), truncate to int16 (context.cpp:266-267),
//      derive the visiting-order key, write the 16-byte CInfo record;
//   4. counting-sort the CInfo records into a uniform cell grid of pitch G >= S, so a tile can collect
//      the clusters whose window may touch it from a few contiguous ranges of the sorted array.
// ---------------------------------------------------------------------------------------------
struct PrepParams {
    int H, W, K, S, T;
    int G, cellW, cellH, ncell;
    int first;     // 1: re-seed colours, no update to finalise
    int finalize;  // 1: fold `acc` into the clusters
    int last;      // 1: after the final update: set is_active / is_updatable like the reference leaves them
    int noq;       // 1: ContextRealDistNoQ -- centroids are float quotients, not rounded integers (context.cpp:375-381)
    // k_prepare only: the `preemptive` option (preempt.cuh; preemptive.h:113-141, context.cpp:360)
    int preempt;       // 1: only updatable clusters take their new centre; the movement test counts is_updatable down
    float l1_thres;    // max(roundf(2 S thres), 1)
    int* nactive;      // [B] number of active clusters (first pass: K = everything active)
};

__global__ void __launch_bounds__(1024) k_prepare(PrepParams pp, fslic_cluster* __restrict__ clusters,
                                                   unsigned long long* __restrict__ acc,
                                                   const uint32_t* __restrict__ quad, CInfo* __restrict__ cinfo,
                                                   int* __restrict__ cell_start,
                                                   CInfo* __restrict__ cinfo_tmp) {
    extern __shared__ int s_cnt[];  // ncell + 1 counters, then 1024/32 warp sums
    const int b = blockIdx.x;
    const int tid = threadIdx.x, nt = blockDim.x;
    fslic_cluster* cl = clusters + (size_t)b * pp.K;
    unsigned long long* ac = acc + (size_t)b * pp.K * 4;
    const uint32_t* qd = quad + (size_t)b * pp.H * pp.W;
    CInfo* ci = cinfo_tmp + (size_t)b * pp.K;          // by cluster index (scratch)
    CInfo* ci_sorted = cinfo + (size_t)b * pp.K;       // by cell, what the assign kernels read
    int* cs = cell_start + (size_t)b * (pp.ncell + 1);

    for (int c = tid; c <= pp.ncell; c += nt) s_cnt[c] = 0;
    if (pp.preempt && pp.first && tid == 0) pp.nactive[b] = pp.K;  // b_all_active = true (preemptive.h:63)
    __syncthreads();

    for (int k = tid; k < pp.K; k += nt) {
        fslic_cluster c = cl[k];
        if (pp.finalize) {
            // packed sums: [0] = n | sum_y << 32, [1] = sum_x | sum_L << 32, [2] = sum_a | sum_b << 32
            const unsigned long long w0 = ac[k * 4 + 0], w1 = ac[k * 4 + 1], w2 = ac[k * 4 + 2];
            const float old_y = c.y, old_x = c.x;  // set_old_clusters (context.cpp:303): the centres the assign used
            const bool frozen = pp.preempt && !c.is_updatable;  // context.cpp:360: keeps centre AND member count
            const uint32_t n = frozen ? 0u : (uint32_t)w0;
            if (!frozen) c.num_members = n;  // written even when n == 0 (context.cpp:360-362)
            if (n > 0 && pp.noq) {  // (float)sum / n: int -> float conversion, IEEE division
                const float fn = __int2float_rn((int32_t)n);
                c.y = __fdiv_rn(__int2float_rn((int32_t)(w0 >> 32)), fn);
                c.x = __fdiv_rn(__int2float_rn((int32_t)(uint32_t)w1), fn);
                c.r = __fdiv_rn(__int2float_rn((int32_t)(w1 >> 32)), fn);
                c.g = __fdiv_rn(__int2float_rn((int32_t)(uint32_t)w2), fn);
                c.b = __fdiv_rn(__int2float_rn((int32_t)(w2 >> 32)), fn);
            } else if (n > 0) {
                const int32_t in = (int32_t)n, half = in / 2;
                c.y = (float)(((int32_t)(w0 >> 32) + half) / in);
                c.x = (float)(((int32_t)(uint32_t)w1 + half) / in);
                c.r = (float)(((int32_t)(w1 >> 32) + half) / in);
                c.g = (float)(((int32_t)(uint32_t)w2 + half) / in);
                c.b = (float)(((int32_t)(w2 >> 32) + half) / in);
            }
            ac[k * 4 + 0] = 0; ac[k * 4 + 1] = 0; ac[k * 4 + 2] = 0;
            if (pp.preempt && c.is_updatable) {  // PreemptiveGrid::set_new_clusters, first loop (preemptive.h:132-141)
                const float l1 = __fadd_rn(fabsf(__fsub_rn(old_x, c.x)), fabsf(__fsub_rn(old_y, c.y)));
                c.is_updatable = l1 < pp.l1_thres ? (uint8_t)(c.is_updatable - 1) : (uint8_t)2;
            }
        }
        if (pp.first) {
            int y = min(max((int)c.y, 0), pp.H - 1), x = min(max((int)c.x, 0), pp.W - 1);
            const uint32_t q = qd[(size_t)y * pp.W + x];
            c.r = (float)(q & 0xff);
            c.g = (float)((q >> 8) & 0xff);
            c.b = (float)((q >> 16) & 0xff);
        }
        // safeguard clamp, stored back like the reference does
        c.x = fminf(fmaxf(c.x, 0.f), (float)(pp.W - 1));
        c.y = fminf(fmaxf(c.y, 0.f), (float)(pp.H - 1));
        c.number = (uint16_t)k;
        if (!pp.preempt || pp.first) {
            c.is_active = 1;
            c.is_updatable = 2;  // PreemptiveGrid::initialize (preemptive.h:59-67)
        } else if (pp.last) {
            c.is_active = 1;     // PreemptiveGrid::finalize (preemptive.h:69-74); is_updatable stays where it got to
        }                        // else: k_preempt_mark decides is_active from the new centres
        cl[k] = c;

        const int cy = (int16_t)c.y, cx = (int16_t)c.x;
        const int cr = (int16_t)c.r, cg = (int16_t)c.g, cb = (int16_t)c.b;
        const int phase = 2 * ((cy / pp.T) & 1) + ((cx / pp.T) & 1);
        CInfo r;
        r.cyx = (cy & 0xffff) | (cx << 16);
        r.color = (uint32_t)(cr & 0xff) | ((uint32_t)(cg & 0xff) << 8) | ((uint32_t)(cb & 0xff) << 16);
        r.sortkey = ((uint32_t)phase << 16) | (uint32_t)k;
        r.pad = 0;
        ci[k] = r;
        const int cell = (cy / pp.G) * pp.cellW + (cx / pp.G);
        atomicAdd(&s_cnt[cell], 1);
    }
    __syncthreads();
    // exclusive scan of the cell histogram (ncell <= ~16K): every thread owns a run of consecutive cells,
    // one block-wide scan of the run totals (two barriers in all)
    __shared__ int s_warp[32];
    {
        const int ncnt = pp.ncell + 1;
        const int per = (ncnt + nt - 1) / nt;
        const int c0 = tid * per;
        int local = 0;
        for (int u = 0; u < per; u++) {
            const int c = c0 + u;
            if (c < ncnt) local += s_cnt[c];
        }
        int x = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int y = __shfl_up_sync(FSLIC_FULL, x, o);
            if ((tid & 31) >= o) x += y;
        }
        if ((tid & 31) == 31) s_warp[tid >> 5] = x;
        __syncthreads();
        if (tid < 32) {
            int w = (tid < (nt >> 5)) ? s_warp[tid] : 0;
            int z = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int y = __shfl_up_sync(FSLIC_FULL, z, o);
                if (tid >= o) z += y;
            }
            s_warp[tid] = z - w;
        }
        __syncthreads();
        int run = s_warp[tid >> 5] + x - local;  // exclusive prefix of this thread's first cell
        for (int u = 0; u < per; u++) {
            const int c = c0 + u;
            if (c < ncnt) {
                const int v = s_cnt[c];
                s_cnt[c] = run;  // becomes the running fill pointer
                cs[c] = run;
                run += v;
            }
        }
    }
    __syncthreads();
    for (int k = tid; k < pp.K; k += nt) {
        const CInfo r = ci[k];
        const int cy = (int16_t)(r.cyx & 0xffff), cx = r.cyx >> 16;
        const int cell = (cy / pp.G) * pp.cellW + (cx / pp.G);
        const int slot = atomicAdd(&s_cnt[cell], 1);
        ci_sorted[slot] = r;  // order inside a cell is arbitrary: consumers rank by sortkey
    }
}

// ---------------------------------------------------------------------------------------------
// k_prepare3: k_prepare for K <= 4096 with the latency taken out (round 2).  k_prepare goes to global memory four
// times in a row per cluster (load record, store the unsorted CInfo, load it back after the scan, store it sorted) and
// handles its two clusters per thread one after the other.  Here every thread loads all its clusters up front, keeps
// the CInfo records in registers, and the shared-memory atomicAdd that counts a cell also hands out the record's rank
// inside the cell -- so after ONE scan the records go straight to their sorted slots: one global load round trip, one
// store, four barriers.  Same results (order inside a cell is arbitrary for both; consumers rank by sort key).
// ---------------------------------------------------------------------------------------------
#define PREP3_PER 4  // clusters per thread at most (K <= 4096 with 1024 threads)
__global__ void __launch_bounds__(1024) k_prepare3(PrepParams pp, fslic_cluster* __restrict__ clusters,
                                                   unsigned long long* __restrict__ acc, const uint32_t* __restrict__ quad,
                                                   CInfo* __restrict__ cinfo, int* __restrict__ cell_start) {
    extern __shared__ int s_cnt[];  // ncell + 1 counters
    __shared__ int s_warp[32];
    const int b = blockIdx.x;
    const int tid = threadIdx.x, nt = blockDim.x;
    fslic_cluster* cl = clusters + (size_t)b * pp.K;
    unsigned long long* ac = acc + (size_t)b * pp.K * 4;
    const uint32_t* qd = quad + (size_t)b * pp.H * pp.W;
    CInfo* ci_sorted = cinfo + (size_t)b * pp.K;
    int* cs = cell_start + (size_t)b * (pp.ncell + 1);
    const int ncnt = pp.ncell + 1;
    for (int c = tid; c < ncnt; c += nt) s_cnt[c] = 0;

    // all global loads of this thread's clusters in flight together
    uint4 ca[PREP3_PER], cb[PREP3_PER];
    ulonglong2 a01[PREP3_PER];
    unsigned long long a2[PREP3_PER];
#pragma unroll
    for (int u = 0; u < PREP3_PER; u++) {
        const int k = tid + u * nt;
        if (k < pp.K) {
            const uint4* p = reinterpret_cast<const uint4*>(cl + k);
            ca[u] = p[0];
            cb[u] = p[1];
            if (pp.finalize) {
                a01[u] = *reinterpret_cast<const ulonglong2*>(ac + (size_t)k * 4);
                a2[u] = ac[(size_t)k * 4 + 2];
            }
        }
    }
    __syncthreads();  // histogram zeroed
    CInfo rec[PREP3_PER];
    int cell[PREP3_PER], rank[PREP3_PER];
#pragma unroll
    for (int u = 0; u < PREP3_PER; u++) {
        const int k = tid + u * nt;
        cell[u] = -1;
        if (k < pp.K) {
            fslic_cluster c;
            memcpy(&c, &ca[u], 16);
            memcpy(reinterpret_cast<char*>(&c) + 16, &cb[u], 16);
            if (pp.finalize) {
                // packed sums: [0] = n | sum_y << 32, [1] = sum_x | sum_L << 32, [2] = sum_a | sum_b << 32
                const unsigned long long w0 = a01[u].x, w1 = a01[u].y, w2 = a2[u];
                const uint32_t n = (uint32_t)w0;
                c.num_members = n;  // written even when n == 0 (context.cpp:360-362)
                if (n > 0 && pp.noq) {
                    const float fn = __int2float_rn((int32_t)n);
                    c.y = __fdiv_rn(__int2float_rn((int32_t)(w0 >> 32)), fn);
                    c.x = __fdiv_rn(__int2float_rn((int32_t)(uint32_t)w1), fn);
                    c.r = __fdiv_rn(__int2float_rn((int32_t)(w1 >> 32)), fn);
                    c.g = __fdiv_rn(__int2float_rn((int32_t)(uint32_t)w2), fn);
                    c.b = __fdiv_rn(__int2float_rn((int32_t)(w2 >> 32)), fn);
                } else if (n > 0) {
                    const int32_t in = (int32_t)n, half = in / 2;
                    c.y = (float)(((int32_t)(w0 >> 32) + half) / in);
                    c.x = (float)(((int32_t)(uint32_t)w1 + half) / in);
                    c.r = (float)(((int32_t)(w1 >> 32) + half) / in);
                    c.g = (float)(((int32_t)(uint32_t)w2 + half) / in);
                    c.b = (float)(((int32_t)(w2 >> 32) + half) / in);
                }
                *reinterpret_cast<ulonglong2*>(ac + (size_t)k * 4) = make_ulonglong2(0ull, 0ull);
                ac[(size_t)k * 4 + 2] = 0ull;
            }
            if (pp.first) {
                int y = min(max((int)c.y, 0), pp.H - 1), x = min(max((int)c.x, 0), pp.W - 1);
                const uint32_t q = qd[(size_t)y * pp.W + x];
                c.r = (float)(q & 0xff);
                c.g = (float)((q >> 8) & 0xff);
                c.b = (float)((q >> 16) & 0xff);
            }
            // safeguard clamp, stored back like the reference does
            c.x = fminf(fmaxf(c.x, 0.f), (float)(pp.W - 1));
            c.y = fminf(fmaxf(c.y, 0.f), (float)(pp.H - 1));
            c.number = (uint16_t)k;
            c.is_active = 1;
            c.is_updatable = 2;
            uint4 o0, o1;
            memcpy(&o0, &c, 16);
            memcpy(&o1, reinterpret_cast<char*>(&c) + 16, 16);
            uint4* p = reinterpret_cast<uint4*>(cl + k);
            p[0] = o0;
            p[1] = o1;

            const int cy = (int16_t)c.y, cx = (int16_t)c.x;
            const int cr = (int16_t)c.r, cg = (int16_t)c.g, cbl = (int16_t)c.b;
            const int phase = 2 * ((cy / pp.T) & 1) + ((cx / pp.T) & 1);
            rec[u].cyx = (cy & 0xffff) | (cx << 16);
            rec[u].color = (uint32_t)(cr & 0xff) | ((uint32_t)(cg & 0xff) << 8) | ((uint32_t)(cbl & 0xff) << 16);
            rec[u].sortkey = ((uint32_t)phase << 16) | (uint32_t)k;
            rec[u].pad = 0;
            cell[u] = (cy / pp.G) * pp.cellW + (cx / pp.G);
            rank[u] = atomicAdd(&s_cnt[cell[u]], 1);  // count the cell and take a slot inside it
        }
    }
    __syncthreads();
    {   // exclusive scan of the cell histogram: every thread owns a run of consecutive cells
        const int per = (ncnt + nt - 1) / nt;
        const int c0 = tid * per;
        int local = 0;
        for (int u = 0; u < per; u++) {
            const int c = c0 + u;
            if (c < ncnt) local += s_cnt[c];
        }
        int x = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int y = __shfl_up_sync(FSLIC_FULL, x, o);
            if ((tid & 31) >= o) x += y;
        }
        if ((tid & 31) == 31) s_warp[tid >> 5] = x;
        __syncthreads();
        if (tid < 32) {
            int w = (tid < (nt >> 5)) ? s_warp[tid] : 0;
            int z = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int y = __shfl_up_sync(FSLIC_FULL, z, o);
                if (tid >= o) z += y;
            }
            s_warp[tid] = z - w;
        }
        __syncthreads();
        int run = s_warp[tid >> 5] + x - local;
        for (int u = 0; u < per; u++) {
            const int c = c0 + u;
            if (c < ncnt) {
                const int v = s_cnt[c];
                s_cnt[c] = run;
                cs[c] = run;
                run += v;
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < PREP3_PER; u++)
        if (cell[u] >= 0) ci_sorted[s_cnt[cell[u]] + rank[u]] = rec[u];
}

// ---------------------------------------------------------------------------------------------
// prepare_in_tail: the finalize / record / counting-sort work of k_prepare3 (no colour re-seed) as a device function
// for the TAIL of an assign+update launch: the last CTA of k_assign5 to finish (ticket counter) calls it, so that a
// single image's ten passes do not pay a kernel boundary between "update" and "next assign" (the eleven k_prepare
// launches were a third of a single image's device time).  The caller's registers are capped at 64 per thread, so the
// records wait in shared memory instead of registers: `smem` needs prepare_tail_smem_bytes(K, ncell) bytes.  The
// accumulators were written by RED.64 from other SMs: they are read with ld.global.cg (L2).  K <= 4096.
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ size_t prepare_tail_smem_bytes(int K, int ncell) {
    return (size_t)((ncell + 1 + 3) & ~3) * 4 + 32 * 4 + (size_t)K * 16 + (size_t)K * 4;
}

__device__ __forceinline__ void prepare_in_tail(const PrepParams& pp, fslic_cluster* __restrict__ cl,
                                                unsigned long long* __restrict__ ac, CInfo* __restrict__ ci_sorted,
                                                int* __restrict__ cs, unsigned char* smem, int tid, int nt) {
    const int ncnt = pp.ncell + 1;
    int* s_cnt = reinterpret_cast<int*>(smem);
    int* s_warp = s_cnt + ((ncnt + 3) & ~3);
    uint4* s_rec = reinterpret_cast<uint4*>(s_warp + 32);
    int* s_slot = reinterpret_cast<int*>(s_rec + pp.K);  // cell << 12 | rank inside the cell
    for (int c = tid; c < ncnt; c += nt) s_cnt[c] = 0;
    __syncthreads();
    for (int k = tid; k < pp.K; k += nt) {
        uint4* gp = reinterpret_cast<uint4*>(cl + k);
        const uint4 g0 = gp[0], g1 = gp[1];
        fslic_cluster c;
        memcpy(&c, &g0, 16);
        memcpy(reinterpret_cast<char*>(&c) + 16, &g1, 16);
        {
            const uint4 a01 = __ldcg(reinterpret_cast<const uint4*>(ac + (size_t)k * 4));
            const uint2 a2 = __ldcg(reinterpret_cast<const uint2*>(ac + (size_t)k * 4 + 2));
            // packed sums: [0] = n | sum_y << 32, [1] = sum_x | sum_L << 32, [2] = sum_a | sum_b << 32
            const uint32_t n = a01.x;
            c.num_members = n;  // written even when n == 0 (context.cpp:360-362)
            if (n > 0) {
                const int32_t in = (int32_t)n, half = in / 2;
                c.y = (float)(((int32_t)a01.y + half) / in);
                c.x = (float)(((int32_t)a01.z + half) / in);
                c.r = (float)(((int32_t)a01.w + half) / in);
                c.g = (float)(((int32_t)a2.x + half) / in);
                c.b = (float)(((int32_t)a2.y + half) / in);
            }
            *reinterpret_cast<ulonglong2*>(ac + (size_t)k * 4) = make_ulonglong2(0ull, 0ull);
            ac[(size_t)k * 4 + 2] = 0ull;
        }
        c.x = fminf(fmaxf(c.x, 0.f), (float)(pp.W - 1));
        c.y = fminf(fmaxf(c.y, 0.f), (float)(pp.H - 1));
        c.number = (uint16_t)k;
        c.is_active = 1;
        c.is_updatable = 2;
        uint4 o0, o1;
        memcpy(&o0, &c, 16);
        memcpy(&o1, reinterpret_cast<char*>(&c) + 16, 16);
        gp[0] = o0;
        gp[1] = o1;
        const int cy = (int16_t)c.y, cx = (int16_t)c.x;
        const int cr = (int16_t)c.r, cg = (int16_t)c.g, cbl = (int16_t)c.b;
        const int phase = 2 * ((cy / pp.T) & 1) + ((cx / pp.T) & 1);
        uint4 rec;
        rec.x = (uint32_t)((cy & 0xffff) | (cx << 16));
        rec.y = (uint32_t)(cr & 0xff) | ((uint32_t)(cg & 0xff) << 8) | ((uint32_t)(cbl & 0xff) << 16);
        rec.z = ((uint32_t)phase << 16) | (uint32_t)k;
        rec.w = 0;
        s_rec[k] = rec;
        const int cell = (cy / pp.G) * pp.cellW + (cx / pp.G);
        s_slot[k] = (cell << 12) | atomicAdd(&s_cnt[cell], 1);
    }
    __syncthreads();
    {   // exclusive scan of the cell histogram: every thread owns a run of consecutive cells
        const int per = (ncnt + nt - 1) / nt;
        const int c0 = tid * per;
        int local = 0;
        for (int u = 0; u < per; u++) {
            const int c = c0 + u;
            if (c < ncnt) local += s_cnt[c];
        }
        int x = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int y = __shfl_up_sync(FSLIC_FULL, x, o);
            if ((tid & 31) >= o) x += y;
        }
        if ((tid & 31) == 31) s_warp[tid >> 5] = x;
        __syncthreads();
        if (tid < 32) {
            int w = (tid < (nt >> 5)) ? s_warp[tid] : 0;
            int z = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int y = __shfl_up_sync(FSLIC_FULL, z, o);
                if (tid >= o) z += y;
            }
            s_warp[tid] = z - w;
        }
        __syncthreads();
        int run = s_warp[tid >> 5] + x - local;
        for (int u = 0; u < per; u++) {
            const int c = c0 + u;
            if (c < ncnt) {
                const int v = s_cnt[c];
                s_cnt[c] = run;
                cs[c] = run;
                run += v;
            }
        }
    }
    __syncthreads();
    uint4* out = reinterpret_cast<uint4*>(ci_sorted);
    for (int k = tid; k < pp.K; k += nt) {
        const int sl = s_slot[k];
        out[s_cnt[sl >> 12] + (sl & 4095)] = s_rec[k];
    }
    __syncthreads();  // the shared buffers are reused by the next image
}

// ---------------------------------------------------------------------------------------------
// k_prepare2: the same bookkeeping spread over ceil(K / 256) CTAs per image (round 2).  k_prepare is one CTA per image
// and latency bound -- two clusters per thread one after the other, five block barriers -- 13 us per launch, eleven
// launches per iterate: a third of a single image's device time.  Here every cluster has its own thread (steps 1-3 of
// k_prepare: finalise, re-seed, clamp, CInfo record, cell histogram through global atomics), and the LAST CTA of an
// image to finish (ticket counter) runs step 4 for the whole image: cell histogram -> shared memory, exclusive scan,
// scatter of the records.  The histogram and the ticket are left zeroed for the next launch.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_prepare2(PrepParams pp, fslic_cluster* __restrict__ clusters,
                                                  unsigned long long* __restrict__ acc, const uint32_t* __restrict__ quad,
                                                  CInfo* __restrict__ cinfo, int* __restrict__ cell_start,
                                                  CInfo* __restrict__ cinfo_tmp, int* __restrict__ cell_cnt,
                                                  unsigned int* __restrict__ tickets) {
    extern __shared__ int s_cnt[];  // last CTA only: ncell + 1 counters
    __shared__ int s_warp[8];
    __shared__ bool s_last;
    const int b = blockIdx.y;
    const int tid = threadIdx.x, nt = blockDim.x;
    fslic_cluster* cl = clusters + (size_t)b * pp.K;
    unsigned long long* ac = acc + (size_t)b * pp.K * 4;
    const uint32_t* qd = quad + (size_t)b * pp.H * pp.W;
    CInfo* ci = cinfo_tmp + (size_t)b * pp.K;          // by cluster index (scratch)
    CInfo* ci_sorted = cinfo + (size_t)b * pp.K;       // by cell, what the assign kernels read
    int* cs = cell_start + (size_t)b * (pp.ncell + 1);
    int* gcnt = cell_cnt + (size_t)b * (pp.ncell + 1);

    const int k = blockIdx.x * nt + tid;
    if (k < pp.K) {
        fslic_cluster c = cl[k];
        if (pp.finalize) {
            // packed sums: [0] = n | sum_y << 32, [1] = sum_x | sum_L << 32, [2] = sum_a | sum_b << 32
            const unsigned long long w0 = ac[k * 4 + 0], w1 = ac[k * 4 + 1], w2 = ac[k * 4 + 2];
            const uint32_t n = (uint32_t)w0;
            c.num_members = n;  // written even when n == 0 (context.cpp:360-362)
            if (n > 0 && pp.noq) {  // (float)sum / n: int -> float conversion, IEEE division
                const float fn = __int2float_rn((int32_t)n);
                c.y = __fdiv_rn(__int2float_rn((int32_t)(w0 >> 32)), fn);
                c.x = __fdiv_rn(__int2float_rn((int32_t)(uint32_t)w1), fn);
                c.r = __fdiv_rn(__int2float_rn((int32_t)(w1 >> 32)), fn);
                c.g = __fdiv_rn(__int2float_rn((int32_t)(uint32_t)w2), fn);
                c.b = __fdiv_rn(__int2float_rn((int32_t)(w2 >> 32)), fn);
            } else if (n > 0) {
                const int32_t in = (int32_t)n, half = in / 2;
                c.y = (float)(((int32_t)(w0 >> 32) + half) / in);
                c.x = (float)(((int32_t)(uint32_t)w1 + half) / in);
                c.r = (float)(((int32_t)(w1 >> 32) + half) / in);
                c.g = (float)(((int32_t)(uint32_t)w2 + half) / in);
                c.b = (float)(((int32_t)(w2 >> 32) + half) / in);
            }
            ac[k * 4 + 0] = 0; ac[k * 4 + 1] = 0; ac[k * 4 + 2] = 0;
        }
        if (pp.first) {
            int y = min(max((int)c.y, 0), pp.H - 1), x = min(max((int)c.x, 0), pp.W - 1);
            const uint32_t q = qd[(size_t)y * pp.W + x];
            c.r = (float)(q & 0xff);
            c.g = (float)((q >> 8) & 0xff);
            c.b = (float)((q >> 16) & 0xff);
        }
        // safeguard clamp, stored back like the reference does
        c.x = fminf(fmaxf(c.x, 0.f), (float)(pp.W - 1));
        c.y = fminf(fmaxf(c.y, 0.f), (float)(pp.H - 1));
        c.number = (uint16_t)k;
        c.is_active = 1;
        c.is_updatable = 2;
        cl[k] = c;

        const int cy = (int16_t)c.y, cx = (int16_t)c.x;
        const int cr = (int16_t)c.r, cg = (int16_t)c.g, cb = (int16_t)c.b;
        const int phase = 2 * ((cy / pp.T) & 1) + ((cx / pp.T) & 1);
        CInfo r;
        r.cyx = (cy & 0xffff) | (cx << 16);
        r.color = (uint32_t)(cr & 0xff) | ((uint32_t)(cg & 0xff) << 8) | ((uint32_t)(cb & 0xff) << 16);
        r.sortkey = ((uint32_t)phase << 16) | (uint32_t)k;
        r.pad = 0;
        ci[k] = r;
        atomicAdd(&gcnt[(cy / pp.G) * pp.cellW + (cx / pp.G)], 1);
    }
    // the last CTA of this image to get here sorts the records into the cell grid
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&tickets[b], 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int ncnt = pp.ncell + 1;
    for (int c = tid; c < ncnt; c += nt) {
        s_cnt[c] = __ldcg(&gcnt[c]);
        gcnt[c] = 0;  // ready for the next launch
    }
    if (tid == 0) tickets[b] = 0;
    __syncthreads();
    {   // exclusive scan: every thread owns a run of consecutive cells, one block-wide scan of the run totals
        const int per = (ncnt + nt - 1) / nt;
        const int c0 = tid * per;
        int local = 0;
        for (int u = 0; u < per; u++) {
            const int c = c0 + u;
            if (c < ncnt) local += s_cnt[c];
        }
        int x = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int y = __shfl_up_sync(FSLIC_FULL, x, o);
            if ((tid & 31) >= o) x += y;
        }
        if ((tid & 31) == 31) s_warp[tid >> 5] = x;
        __syncthreads();
        int woff = 0;
        for (int w = 0; w < (tid >> 5); w++) woff += s_warp[w];
        int run = woff + x - local;  // exclusive prefix of this thread's first cell
        for (int u = 0; u < per; u++) {
            const int c = c0 + u;
            if (c < ncnt) {
                const int v = s_cnt[c];
                s_cnt[c] = run;  // becomes the running fill pointer
                cs[c] = run;
                run += v;
            }
        }
    }
    __syncthreads();
    for (int kk = tid; kk < pp.K; kk += nt) {
        const uint4 r = __ldcg(reinterpret_cast<const uint4*>(&ci[kk]));  // written by other CTAs: read through L2
        const int cy = (int16_t)(r.x & 0xffff), cx = (int)r.x >> 16;
        const int slot = atomicAdd(&s_cnt[(cy / pp.G) * pp.cellW + (cx / pp.G)], 1);
        *reinterpret_cast<uint4*>(&ci_sorted[slot]) = r;  // order inside a cell is arbitrary: consumers rank by sortkey
    }
}

// ---------------------------------------------------------------------------------------------
// Spatial patch (BaseContext::set_spatial_patch, context.cpp:23-40), laid out for LINEAR addressing:
//   tbl[(di + OY) * TS + (dj + OX)] = (u16)(coef * (float)(|di| + |dj|))  inside the (2S+1)^2 window,
//                                   = FSLIC_BIGSP                         outside it,
// for di in [-OY, OY], dj in [-OX, OX].  A pixel's entry for candidate c is then at
//   (i*TS + j) + ((OY - cy)*TS + (OX - cx)):  a per-thread constant plus a per-candidate constant,
// so the window predicate and both abs() disappear from the inner loop.
// With manhattan_spatial_dist = false (context.cpp:34-38) the entry is (u16)(coef * hypotf(di, dj)) on the same
// square window; the kernels that read the table do not change.
// ---------------------------------------------------------------------------------------------

// glibc's hypotf on integer arguments: it rounds the exact sqrt(a^2 + b^2) once to float, which is what the double
// square root of the exact double sum gives (a^2 + b^2 < 2^53).  CUDA's hypotf and a float sqrt both differ from it.
__device__ __forceinline__ float ref_hypotf(int a, int b) {
    return __double2float_rn(__dsqrt_rn((double)a * (double)a + (double)b * (double)b));
}

// the reference's u16 spatial term for offsets (di, dj) of the window (context.cpp:30 / :36)
__device__ __forceinline__ uint32_t spatial_u16(float coef, int di, int dj, int euclid) {
    const float m = euclid ? ref_hypotf(di, dj) : (float)(abs(di) + abs(dj));
    return (uint16_t)__float2uint_rz(__fmul_rn(coef, m));
}

__global__ void k_build_sptable(uint16_t* __restrict__ tbl, int S, int OY, int OX, int TS, float coef, int euclid) {
    const int n = (2 * OY + 1) * TS;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
        const int r = t / TS, c = t - r * TS;
        const int di = abs(r - OY), dj = abs(c - OX);
        uint16_t v = (uint16_t)FSLIC_BIGSP;
        if (di <= S && dj <= S && c <= 2 * OX) v = (uint16_t)spatial_u16(coef, di, dj, euclid);
        tbl[t] = v;
    }
}

struct AssignParams {
    int H, W, K, S, B;
    int stride, rem;   // rows i with i % stride == rem are processed; sub-row sr <-> i = rem + sr*stride
    int nsub;          // number of such rows
    int cfg_stride;    // the configured subsample stride (freshness test)
    int fresh_from;    // rows with (i % cfg_stride) >= fresh_from were never assigned before
    int G, cellW, cellH, ncell;
    uint32_t Ginv;     // ceil(2^32 / G): x / G == __umulhi(x, Ginv) for 0 <= x < 65536 (x * G < 2^32)
    int OY, OX, TS, tbl_elems;
    int tiles_x, tiles_y, ntiles;  // warp tiles (32 columns x R sub-rows) per image
    int tps;           // warp tiles per super tile: AS_T, or 1 when the launch is too small to fill the GPU otherwise
    float coef;        // generic path only
    // k_assign5 only: everything warp uniform that the host can precompute lives in the constant bank, so the kernel
    // neither keeps it in registers nor re-derives it (the compiler rematerialised the divisions per super tile)
    int stx, per_img, total;        // super tiles per tile row / per image / in all
    int wstride, db, dty, dsx;      // a warp's step through the super tiles, decomposed into (image, tile row, column) carries
    uint32_t tbl_bytes;             // patch size in shared memory, padded to 128 bytes
    uint32_t cinfo_img_bytes, cells_img_bytes, acc_img_bytes;  // per-image pitches of cinfo / cell_start / acc
    int fuse_prepare;               // 1: the last CTA to finish runs prepare_in_tail for the next pass (small batches)
    int euclid;                     // manhattan_spatial_dist = false: kernels that compute the spatial term inline use hypotf
};

#define AS_WARPS 16
#define AS_THREADS (AS_WARPS * 32)
#define AS_LIST 32  // candidate capacity of one warp tile; beyond it the tile takes the brute-force path

__device__ __forceinline__ int div_g(int x, uint32_t ginv) { return (int)__umulhi((uint32_t)x, ginv); }

// Packed per-cluster accumulators, 3 x u64 (+1 pad) so one update is 3 RED.64 instead of 6 RED.32:
//   [0] = n | sum_y << 32      [1] = sum_x | sum_L << 32      [2] = sum_a | sum_b << 32
// Every half stays far below 2^32 (sum_y <= n*H), so the halves never carry into each other.
__device__ __forceinline__ void acc_add_pixel(unsigned long long* ac, uint32_t label, int i, int j, uint32_t q) {
    atomicAdd(&ac[label * 4 + 0], 1ull | ((unsigned long long)(uint32_t)i << 32));
    atomicAdd(&ac[label * 4 + 1], (unsigned long long)(uint32_t)j | ((unsigned long long)(q & 0xff) << 32));
    atomicAdd(&ac[label * 4 + 2], (unsigned long long)((q >> 8) & 0xff) | ((unsigned long long)((q >> 16) & 0xff) << 32));
}

// Brute-force assignment of one pixel straight from the cell grid: lexicographic minimum of
// (d, phase, k) over the clusters whose window covers (i, j).  Returns the new label (or the kept
// one) and stores it.  Used by the generic kernel and by warp tiles whose candidate list overflowed.
// spatial(|di|, |dj|) is the u16 spatial term: computed by the generic kernel, read from the shared patch by the
// table-driven kernels (which then need neither coef nor the metric in registers).
template <typename Spatial>
__device__ __forceinline__ uint32_t assign_pixel_generic(const AssignParams& ap, int i, int j, uint32_t q,
                                                          const CInfo* __restrict__ ci, const int* __restrict__ cs,
                                                          uint16_t* __restrict__ lb, Spatial spatial) {
    const int S = ap.S, W = ap.W, H = ap.H;
    unsigned long long best = ~0ull;
    const int cr0 = max(i - S, 0) / ap.G, cr1 = min(i + S, H - 1) / ap.G;
    const int cc0 = max(j - S, 0) / ap.G, cc1 = min(j + S, W - 1) / ap.G;
    for (int cr = cr0; cr <= cr1; cr++) {
        const int s = cs[cr * ap.cellW + cc0], e = cs[cr * ap.cellW + cc1 + 1];
        for (int u = s; u < e; u++) {
            const CInfo r = ci[u];
            const int cy = (int16_t)(r.cyx & 0xffff), cx = r.cyx >> 16;
            const int di = abs(i - cy), dj = abs(j - cx);
            if (di > S || dj > S) continue;
            const uint32_t sp = spatial(di, dj);
            const uint32_t d = sad4_acc(q, r.color, sp) & 0xffffu;  // u16 arithmetic like the scalar reference
            const unsigned long long key = ((unsigned long long)d << 32) | r.sortkey;
            best = key < best ? key : best;
        }
    }
    uint32_t label;
    if (best != ~0ull && (uint32_t)(best >> 32) < 0xFFFFu) {
        label = (uint32_t)(best & 0xffff);
        lb[(size_t)i * W + j] = (uint16_t)label;
    } else if ((i % ap.cfg_stride) >= ap.fresh_from) {
        lb[(size_t)i * W + j] = 0xFFFF;
        label = 0xFFFF;
    } else {
        label = lb[(size_t)i * W + j];  // keep the label of an earlier pass (context.cpp:289-294 never fires)
    }
    return label;
}

__device__ __forceinline__ uint32_t lds_u16(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}

// exact per-byte equality -> 0x80 in every byte of w that equals the corresponding byte of m
__device__ __forceinline__ uint32_t eq80(uint32_t w, uint32_t m) {
    const uint32_t t = w ^ m;
    const uint32_t a = (t & 0x7f7f7f7fu) + 0x7f7f7f7fu;
    return ~(a | t) & 0x80808080u;
}

__device__ __forceinline__ void mma_u8_16x8x32(int (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                               uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// ---------------------------------------------------------------------------------------------
// k_assign_warp<TS, STRIDE, UPDATE>: the hot kernel.  Persistent CTAs (the spatial patch is loaded
// into shared memory once per CTA); inside a CTA every WARP is autonomous -- no block barrier
// after the patch load.  A warp walks "super tiles" of 4 horizontally adjacent warp tiles
// (each 32 columns x 4 sub-rows):
//   L. candidate lists for the 4 tiles at once, 8 lanes per tile: the clusters whose (2S+1)^2
//      window can touch the tile are collected from the cell grid (exact filter, ballot
//      compaction, <= 32 per tile), ranked by (phase, k) -- the reference's visiting order
//      (context.cpp:214-242) -- and staged {colour, patch offset} by rank in per-warp shared memory;
//   then per tile:
//   1. 4 quad loads per lane (LDG.32, 128 B per warp row);
//   2. per candidate and pixel:  LDS.U16 patch entry [immediate row offsets: TS and STRIDE are
//      compile-time] -> VABSDIFF4.U8.ACC (colour SAD + spatial) -> IMAD (d << 16 | rank) -> VIMNMX;
//   3. labels out (STG.U16, 64 B per warp row);
//   4. update sums (context.cpp:316-327) as an exact int8 tensor-core product
//        one-hot(rank)^T (candidates x pixels)  x  [1, row, lane, L, a, b] (pixels x features)
//      (mma.sync m16n8k32 u8 x u8 -> s32, 4 MMAs per 128 pixels and 16 candidates); the D fragment of lane
//      (g, tig) is accumulator word tig of candidates g and g+8, flushed as RED.64 if they received pixels.
//      Integer sums are order independent => exact.
// HBM per processed pixel: 4 B quad read + 2 B label written.
// ---------------------------------------------------------------------------------------------
#ifndef FSLIC_UPDATE_MATCH
#define FSLIC_UPDATE_MATCH 0  // 0: int8 tensor-core one-hot product; 1: MATCH.ANY + REDUX per row (measured 1.4x slower, kept for comparison)
#endif
#ifndef AS_RG
#define AS_RG 1  // row groups of 4 sub-rows per lane (R = 4 * AS_RG rows per warp tile)
#endif
#ifndef AS_MINB
#define AS_MINB 2  // resident CTAs per SM the register budget is sized for
#endif
#define AS_R (4 * AS_RG)
#define AS_T 4   // warp tiles per super tile
#define AS_STAGE_BYTES (AS_WARPS * AS_T * AS_LIST * 22)

template <int TS, int STRIDE, bool UPDATE>
__global__ void __launch_bounds__(AS_THREADS, AS_MINB) k_assign_warp(AssignParams ap, const uint32_t* __restrict__ quad,
                                                               uint16_t* __restrict__ labels,
                                                               const CInfo* __restrict__ cinfo,
                                                               const int* __restrict__ cell_start,
                                                               unsigned long long* __restrict__ acc,
                                                               const uint16_t* __restrict__ g_tbl) {
    constexpr int R = AS_R;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint16_t* s_tbl = reinterpret_cast<uint16_t*>(smem_raw);
    // per-warp private staging block behind the patch in dynamic shared memory (AS_STAGE_BYTES in total):
    //   [ent: AS_T x 32 x uint2][ukey: AS_T x 32 x u32][ucol: same][ucyx: same][k: AS_T x 32 x u16]
    // the MMA A staging [32 pixel lanes][8 features] x u32 aliases ukey+ucol of the SAME warp (dead once ranked)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned char* wst = smem_raw + ((ap.tbl_elems * 2 + 15) & ~15) + warp * (AS_T * AS_LIST * 22);
    uint2 (*s_ent)[AS_LIST] = reinterpret_cast<uint2 (*)[AS_LIST]>(wst);
    uint32_t (*s_ukey)[AS_LIST] = reinterpret_cast<uint32_t (*)[AS_LIST]>(wst + AS_T * AS_LIST * 8);
    uint32_t (*s_ucol)[AS_LIST] = reinterpret_cast<uint32_t (*)[AS_LIST]>(wst + AS_T * AS_LIST * 12);
    int32_t (*s_ucyx)[AS_LIST] = reinterpret_cast<int32_t (*)[AS_LIST]>(wst + AS_T * AS_LIST * 16);
    uint16_t (*s_k)[AS_LIST] = reinterpret_cast<uint16_t (*)[AS_LIST]>(wst + AS_T * AS_LIST * 20);
    uint32_t (*s_feat)[8] = reinterpret_cast<uint32_t (*)[8]>(wst + AS_T * AS_LIST * 8);
    static_assert(32 * 8 * 4 <= AS_T * AS_LIST * 8, "the MMA staging must fit in ukey + ucol");
    static_assert(AS_R <= 16, "row index feature is a byte and the sums are scaled by 128 in s32");

    for (int t = tid; t < (ap.tbl_elems + 1) / 2; t += AS_THREADS)
        reinterpret_cast<uint32_t*>(s_tbl)[t] = reinterpret_cast<const uint32_t*>(g_tbl)[t];
    __syncthreads();

    const int S = ap.S, W = ap.W, H = ap.H;
    const int stride = STRIDE ? STRIDE : ap.stride;
    const int g = lane >> 2, tig = lane & 3;   // MMA fragment coordinates
    const int grp = lane >> 3, gl = lane & 7;  // list building: 8 lanes per tile
    const int rowpix = stride * W;

    // super-tile walk without divisions: (b, ty, sx) advance by a fixed (db, dty, dsx) with carries
    const int tps = ap.tps;
    const int stx = (ap.tiles_x + tps - 1) / tps;  // super tiles per tile row
    const long per_img = (long)stx * ap.tiles_y;
    const long total = per_img * ap.B;
    const long wstride = (long)gridDim.x * AS_WARPS;
    const long first = (long)blockIdx.x * AS_WARPS + warp;
    int b = (int)(first / per_img);
    const int tl0 = (int)(first - (long)b * per_img);
    int ty = tl0 / stx, sx = tl0 - ty * stx;
    const int db = (int)(wstride / per_img);
    const int dtl = (int)(wstride - (long)db * per_img);
    const int dty = dtl / stx, dsx = dtl - dty * stx;
    for (long st = first; st < total; st += wstride, b += db, ty += dty, sx += dsx) {
        if (sx >= stx) { sx -= stx; ty += 1; }
        if (ty >= ap.tiles_y) { ty -= ap.tiles_y; b += 1; }
        const int wsr0 = ty * R;
        const int nrow = min(R, ap.nsub - wsr0);  // valid sub-rows of this tile row (>= 1)
        const int wi0 = ap.rem + wsr0 * stride, wi1 = wi0 + (nrow - 1) * stride;
        const size_t img_off = (size_t)b * H * W;
        const CInfo* ci = cinfo + (size_t)b * ap.K;
        const int* cs = cell_start + (size_t)b * (ap.ncell + 1);
        unsigned long long* ac = acc + (size_t)b * ap.K * 4;

        // ---- L. candidate lists of the 4 tiles, 8 lanes each ----
        // tile of this lane group: columns [gj0, gj0+31]; wanted clusters: cy in [wi0-S, wi1+S], cx in [gj0-S, gj0+31+S]
        const int gtx = sx * tps + grp;
        const bool gvalid = grp < tps && gtx < ap.tiles_x;
        const int gj0 = gtx * 32;
        int n_g = 0;  // candidates found for this group's tile (same value in its 8 lanes)
        {
            const int cr0 = div_g(max(wi0 - S, 0), ap.Ginv), cr1 = div_g(min(wi1 + S, H - 1), ap.Ginv);
            const int cc0 = div_g(max(gj0 - S, 0), ap.Ginv), cc1 = div_g(min(gj0 + 31 + S, W - 1), ap.Ginv);
            for (int crb = cr0; crb <= cr1; crb += 8) {
                const int cr = crb + gl;
                int rs = 0, cnt = 0;
                if (gvalid && cr <= cr1) {
                    rs = cs[cr * ap.cellW + cc0];
                    cnt = cs[cr * ap.cellW + cc1 + 1] - rs;
                }
                int incl = cnt;  // inclusive scan inside the 8-lane group
#pragma unroll
                for (int o = 1; o < 8; o <<= 1) {
                    const int y = __shfl_up_sync(FSLIC_FULL, incl, o, 8);
                    if (gl >= o) incl += y;
                }
                const int T = __shfl_sync(FSLIC_FULL, incl, 7, 8);
                const int Tmax = __reduce_max_sync(FSLIC_FULL, T);
                const int nr = min(8, cr1 - crb + 1);  // cell rows in this chunk (same for every lane group)
                for (int t0 = 0; t0 < Tmax; t0 += 8) {
                    const int t = t0 + gl;
                    int row = 0;
                    for (int r = 0; r < nr - 1; r++) row += (t >= __shfl_sync(FSLIC_FULL, incl, r, 8));
                    const int rincl = __shfl_sync(FSLIC_FULL, incl, row, 8);
                    const int rcnt = __shfl_sync(FSLIC_FULL, cnt, row, 8);
                    const int rstart = __shfl_sync(FSLIC_FULL, rs, row, 8);
                    bool hit = false;
                    CInfo r;
                    if (t < T) {
                        r = ci[rstart + (t - (rincl - rcnt))];
                        const int cy = (int16_t)(r.cyx & 0xffff), cx = r.cyx >> 16;
                        hit = (cy >= wi0 - S) && (cy <= wi1 + S) && (cx >= gj0 - S) && (cx <= gj0 + 31 + S);
                    }
                    const unsigned gb = (__ballot_sync(FSLIC_FULL, hit) >> (grp * 8)) & 0xffu;
                    const int slot = n_g + __popc(gb & ((1u << gl) - 1));
                    if (hit && slot < AS_LIST) {
                        s_ukey[grp][slot] = r.sortkey;
                        s_ucol[grp][slot] = r.color;
                        s_ucyx[grp][slot] = r.cyx;
                    }
                    n_g += __popc(gb);
                }
            }
        }
        __syncwarp();
        {   // rank by (phase, k) (keys are unique) and stage by rank
            const int nmax = __reduce_max_sync(FSLIC_FULL, min(n_g, AS_LIST));
            for (int a0 = 0; a0 < nmax; a0 += 8) {
                const int a = a0 + gl;
                const bool mine = a < n_g && n_g <= AS_LIST;
                const uint32_t key = mine ? s_ukey[grp][a] : 0u;
                int rank = 0;
                for (int u = 0; u < nmax; u++) rank += (u < n_g) && (s_ukey[grp][u] < key);
                if (mine) {
                    const int32_t cyx = s_ucyx[grp][a];
                    const int cy = (int16_t)(cyx & 0xffff), cx = cyx >> 16;
                    s_ent[grp][rank] =
                        make_uint2(s_ucol[grp][a], (uint32_t)(2 * ((ap.OY - cy) * TS + (ap.OX - cx))));
                    s_k[grp][rank] = (uint16_t)(key & 0xffff);
                }
            }
        }
        __syncwarp();
        // ---- the 4 tiles, one after the other ----
#pragma unroll 1
        for (int tq = 0; tq < tps; tq++) {
            const int tx = sx * tps + tq;
            if (tx >= ap.tiles_x) break;  // warp uniform
            const int n = __shfl_sync(FSLIC_FULL, n_g, tq * 8);
            const int wj0 = tx * 32;
            const int j = wj0 + lane;
            const bool colok = j < W;
            const uint32_t* qrow = quad + img_off + (size_t)wi0 * W + j;  // this lane's pixel in row 0 of the tile
            uint16_t* lrow = labels + img_off + (size_t)wi0 * W + j;

            // ---- 1. pixels ----
            uint32_t q[R];
#pragma unroll
            for (int rr = 0; rr < R; rr++) {
                const bool ok = colok && rr < nrow;
                q[rr] = ok ? ld_nc_u32(qrow + rr * rowpix) : 0u;
            }

            if (n > AS_LIST) {
                // ---- overflow (clusters piled on one spot): brute force, direct atomics ----
#pragma unroll
                for (int rr = 0; rr < R; rr++) {
                    if (colok && rr < nrow) {
                        const int i = wi0 + rr * stride;
                        const uint32_t label = assign_pixel_generic(ap, i, j, q[rr], ci, cs, labels + img_off, [&](int di, int dj) {
                            return (uint32_t)s_tbl[(di + ap.OY) * TS + (dj + ap.OX)];
                        });
                        if (UPDATE && label != 0xFFFF) acc_add_pixel(ac, label, i, j, q[rr]);
                    }
                }
                continue;
            }

            // ---- 2. distances ----
            // every (row, column) of the footprint is inside the patch for every listed candidate, valid or not.
            // patch entry of (row rr, candidate c) at shared byte address row0 + c.offset + rr * 2*stride*TS
            const unsigned char* rowp = smem_raw + 2 * (wi0 * TS + j);
            uint32_t best[R];
#pragma unroll
            for (int rr = 0; rr < R; rr++) best[rr] = 0xffffffffu;
            for (int c = 0; c < n; c++) {
                const uint2 e = s_ent[tq][c];
                const unsigned char* pc = rowp + (int)e.y;
#pragma unroll
                for (int rr = 0; rr < R; rr++) {
                    const uint32_t sp = *reinterpret_cast<const uint16_t*>(pc + rr * (2 * stride * TS));
                    const uint32_t d = sad4_acc(q[rr], e.x, sp);
                    best[rr] = min(best[rr], d * 65536u + (uint32_t)c);
                }
            }

            // ---- 3. labels + update sums (context.cpp:316-327) ----
#if FSLIC_UPDATE_MATCH
            // Per row: lanes are grouped by their winning cluster with one MATCH.ANY; each group reduces its packed
            // sums with two REDUX (every group under its own member mask) and its leader issues 3 RED.64.
            // Integer sums are order independent => exact.
#pragma unroll
            for (int rr = 0; rr < R; rr++) {
                const bool ok = colok && rr < nrow;
                const bool covered = ok && ((best[rr] >> 16) < FSLIC_BIGSP);
                uint32_t kk = 0xFFFFu;  // cluster this pixel contributes to (0xFFFF: none)
                if (covered) {
                    kk = s_k[tq][best[rr] & 0xff];
                    lrow[rr * rowpix] = (uint16_t)kk;
                } else if (ok) {
                    const int i = wi0 + rr * stride;
                    if ((i % ap.cfg_stride) >= ap.fresh_from) {
                        lrow[rr * rowpix] = 0xFFFF;
                    } else if (UPDATE) {  // a stale label from an earlier pass still counts (context.cpp:318-319)
                        kk = lrow[rr * rowpix];
                    }
                }
                if (UPDATE) {
                    const unsigned grp_mask = __match_any_sync(FSLIC_FULL, kk);
                    if (kk != 0xFFFFu) {
                        const uint32_t qv = q[rr];
                        // w0 = count | lane << 8 | L << 17 ; w1 = a | b << 16   (sums over <= 32 lanes cannot carry)
                        const uint32_t s0 = __reduce_add_sync(grp_mask, 1u | ((uint32_t)lane << 8) | ((qv & 0xffu) << 17));
                        const uint32_t s1 = __reduce_add_sync(grp_mask, ((qv >> 8) & 0xffu) | ((qv & 0xff0000u)));
                        if (lane == __ffs(grp_mask) - 1) {
                            const uint32_t cnt = s0 & 0xffu, sl = (s0 >> 8) & 0x1ffu, sL = s0 >> 17;
                            const uint32_t i = (uint32_t)(wi0 + rr * stride);
                            unsigned long long* a3 = ac + (size_t)kk * 4;
                            atomicAdd(a3 + 0, (unsigned long long)cnt | ((unsigned long long)(cnt * i) << 32));
                            atomicAdd(a3 + 1, (unsigned long long)(cnt * (uint32_t)wj0 + sl) | ((unsigned long long)sL << 32));
                            atomicAdd(a3 + 2, (unsigned long long)(s1 & 0xffffu) | ((unsigned long long)(s1 >> 16) << 32));
                        }
                    }
                }
            }
            {
#else
            // ---- 3. labels ----
            uint32_t rw[AS_RG];  // local rank bytes, 4 rows per word (0xFF = contributes to no candidate)
#pragma unroll
            for (int gq = 0; gq < AS_RG; gq++) rw[gq] = 0;
#pragma unroll
            for (int rr = 0; rr < R; rr++) {
                const bool ok = colok && rr < nrow;
                const bool covered = ok && ((best[rr] >> 16) < FSLIC_BIGSP);
                uint32_t rb = 0xff;
                if (covered) {
                    rb = best[rr] & 0xff;
                    lrow[rr * rowpix] = s_k[tq][rb];
                } else if (ok) {
                    const int i = wi0 + rr * stride;
                    if ((i % ap.cfg_stride) >= ap.fresh_from) {
                        lrow[rr * rowpix] = 0xFFFF;
                    } else if (UPDATE) {  // a stale label from an earlier pass still counts (context.cpp:318-319)
                        const uint16_t old = lrow[rr * rowpix];
                        if (old != 0xFFFF) acc_add_pixel(ac, old, i, j, q[rr]);
                    }
                }
                rw[rr >> 2] |= rb << (8 * (rr & 3));
            }

            // ---- 4. update sums on the tensor cores ----
            if (UPDATE) {
                // D[candidate][feature] += OneHot[candidate][pixel] * F[pixel][feature]   (m16n8k32, u8 x u8 -> s32)
                //   A = one-hot of the winning rank, built in registers (16 candidates per pass: one pass unless
                //       the list is longer than 16);  B = [1, row, lane, L, a, b, 0, 0] per pixel, staged in smem.
                // Lane (g, tig) ends up with features (2 tig, 2 tig + 1) of candidates g and g + 8: exactly the two
                // halves of packed accumulator word tig -- no compaction of the winners, no shuffles of D.
                const int n16 = (n + 15) >> 4;
                for (int nt = 0; nt < n16; nt++) {
                    int d[4] = {0, 0, 0, 0};
                    const uint32_t mg0 = (uint32_t)(nt * 16 + g) * 0x01010101u, mg1 = mg0 + 0x08080808u;
#pragma unroll
                    for (int gq = 0; gq < AS_RG; gq++) {
                        // stage this row group's features: [count 1, row index, lane index, L, a, b, 0, 0] per pixel lane
                        const uint32_t q0 = q[4 * gq], q1 = q[4 * gq + 1], q2 = q[4 * gq + 2], q3 = q[4 * gq + 3];
                        const uint32_t lo01 = __byte_perm(q0, q1, 0x5140), lo23 = __byte_perm(q2, q3, 0x5140);
                        const uint32_t hi01 = __byte_perm(q0, q1, 0x0062), hi23 = __byte_perm(q2, q3, 0x0062);
                        __syncwarp();  // the previous group's fragments have been read
                        *reinterpret_cast<uint4*>(&s_feat[lane][0]) =
                            make_uint4(0x01010101u, 0x03020100u + 0x04040404u * gq, (uint32_t)lane * 0x01010101u,
                                       __byte_perm(lo01, lo23, 0x5410));
                        *reinterpret_cast<uint4*>(&s_feat[lane][4]) =
                            make_uint4(__byte_perm(lo01, lo23, 0x7632), __byte_perm(hi01, hi23, 0x5410), 0u, 0u);
                        __syncwarp();
#pragma unroll
                        for (int s4 = 0; s4 < 4; s4++) {
                            const uint32_t w0 = __shfl_sync(FSLIC_FULL, rw[gq], 8 * s4 + tig);
                            const uint32_t w1 = __shfl_sync(FSLIC_FULL, rw[gq], 8 * s4 + 4 + tig);
                            mma_u8_16x8x32(d, eq80(w0, mg0), eq80(w0, mg1), eq80(w1, mg0), eq80(w1, mg1),
                                           s_feat[8 * s4 + tig][g], s_feat[8 * s4 + 4 + tig][g]);
                        }
                    }
                    // sums are scaled by 128 (the one-hot byte is 0x80)
#pragma unroll
                    for (int hh = 0; hh < 2; hh++) {
                        const int c = nt * 16 + g + 8 * hh;
                        const uint32_t v0 = (uint32_t)d[2 * hh] >> 7, v1 = (uint32_t)d[2 * hh + 1] >> 7;
                        const uint32_t cnt = __shfl_sync(FSLIC_FULL, v0, lane & ~3);  // feature 0 lives in the tig = 0 lane
                        if (c < n && tig < 3 && cnt != 0) {
                            unsigned long long word;
                            if (tig == 0)
                                word = (unsigned long long)cnt |
                                       ((unsigned long long)(cnt * (uint32_t)wi0 + (uint32_t)stride * v1) << 32);
                            else if (tig == 1)
                                word = (unsigned long long)(cnt * (uint32_t)wj0 + v0) | ((unsigned long long)v1 << 32);
                            else
                                word = (unsigned long long)v0 | ((unsigned long long)v1 << 32);
                            atomicAdd(&ac[(uint32_t)s_k[tq][c] * 4 + tig], word);
                        }
                    }
                }
                __syncwarp();  // s_feat is rewritten by the next tile
            }
#endif
#if FSLIC_UPDATE_MATCH
            }
#endif
        }
        __syncwarp();  // the list staging is rewritten by the next super tile
    }
}

// ---------------------------------------------------------------------------------------------
// k_assign_generic<UPDATE>: correctness-first path without the shared-memory patch, for S so large
// that the linear patch does not fit in shared memory.  One thread per pixel.
// ---------------------------------------------------------------------------------------------
template <bool UPDATE>
__global__ void __launch_bounds__(256) k_assign_generic(AssignParams ap, const uint32_t* __restrict__ quad,
                                                         uint16_t* __restrict__ labels,
                                                         const CInfo* __restrict__ cinfo,
                                                         const int* __restrict__ cell_start,
                                                         unsigned long long* __restrict__ acc) {
    const long per_img = (long)ap.nsub * ap.W;
    const long total = per_img * ap.B;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const int b = (int)(t / per_img);
        const long r = t - (long)b * per_img;
        const int sr = (int)(r / ap.W), j = (int)(r - (long)sr * ap.W);
        const int i = ap.rem + sr * ap.stride;
        const uint32_t q = quad[(size_t)b * ap.H * ap.W + (size_t)i * ap.W + j];
        const uint32_t label = assign_pixel_generic(ap, i, j, q, cinfo + (size_t)b * ap.K,
                                                    cell_start + (size_t)b * (ap.ncell + 1),
                                                    labels + (size_t)b * ap.H * ap.W,
                                                    [&](int di, int dj) { return spatial_u16(ap.coef, di, dj, ap.euclid); });
        if (UPDATE && label != 0xFFFF) acc_add_pixel(acc + (size_t)b * ap.K * 4, label, i, j, q);
    }
}
