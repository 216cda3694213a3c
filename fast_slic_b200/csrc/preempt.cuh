// fast_slic_b200/csrc/preempt.cuh -- the `preemptive` option of the reference (SURVEY.md section 8(f) row 4).
//
// Replaces PreemptiveGrid (/root/reference/src/preemptive.h) and the branches of BaseContext::assign / ::update that
// consult it (context.cpp:218, :307-345, :360, :385).  With preemptive = true a cluster that moved less than
// max(round(2 S thres), 1) pixels (L1) in an update counts its is_updatable down (2 -> 1 -> 0, 0 is final); every cluster
// within a Chebyshev distance of 2S of a still-updatable one stays ACTIVE, so does its 2S x 2S pixel cell.  Inactive
// clusters are not visited by the next assign (their pixels keep their labels unless an active cluster's window takes
// them), pixels of inactive cells do not count in the next update, clusters that are not updatable keep their centre.
//
// It is an option that is off in every BASELINE configuration, so this is a correctness-first path (one thread per
// pixel over the cell grid, like k_assign_generic); the bookkeeping rides on k_prepare (PrepParams.preempt) plus
// k_preempt_mark below.  Results are bit-identical to the compiled reference (tests/test_parity_gpu.py).
#pragma once
#include "assign.cuh"

// per image: is_active of every cluster, the active-cell map and the number of active clusters.  One CTA per image.
// cinfo / cell_start: the FULL cell grid k_prepare just built (all clusters, new centres).
__global__ void __launch_bounds__(1024) k_preempt_mark(int K, int S, int H, int W, int G, int cellW, int cellH, int ncell,
                                                       fslic_cluster* __restrict__ clusters, const CInfo* __restrict__ cinfo,
                                                       const int* __restrict__ cell_start, uint8_t* __restrict__ cellmap,
                                                       int CW2, int ncell2, int* __restrict__ nactive) {
    const int b = blockIdx.x;
    fslic_cluster* cl = clusters + (size_t)b * K;
    const CInfo* ci = cinfo + (size_t)b * K;
    const int* cs = cell_start + (size_t)b * (ncell + 1);
    uint8_t* cm = cellmap + (size_t)b * ncell2;
    __shared__ int s_count;
    if (threadIdx.x == 0) s_count = 0;
    for (int t = threadIdx.x; t < ncell2; t += blockDim.x) cm[t] = 0;
    __syncthreads();
    const int R = 2 * S;
    int mine = 0;
    for (int n = threadIdx.x; n < K; n += blockDim.x) {
        // (int) of the clamped centre == the int16 the records hold (H, W <= 32767)
        const int y = (int)cl[n].y, x = (int)cl[n].x;
        const int cr0 = max(y - R, 0) / G, cr1 = min(y + R, H - 1) / G;
        const int cc0 = max(x - R, 0) / G, cc1 = min(x + R, W - 1) / G;
        bool active = false;
        for (int cr = cr0; cr <= cr1 && !active; cr++) {
            const int s = cs[cr * cellW + cc0], e = cs[cr * cellW + cc1 + 1];
            for (int u = s; u < e; u++) {
                const CInfo r = ci[u];
                const int uy = (int16_t)(r.cyx & 0xffff), ux = r.cyx >> 16;
                if (abs(uy - y) > R || abs(ux - x) > R) continue;  // preemptive.h:160-161
                // (a pair within 2S of each other always sits in adjacent 2S cells: the 3 x 3 walk of :150-156 adds nothing)
                if (cl[r.sortkey & 0xffffu].is_updatable) {         // preemptive.h:145
                    active = true;
                    break;
                }
            }
        }
        cl[n].is_active = active ? 1 : 0;
        if (active) {
            cm[(y / R) * CW2 + (x / R)] = 1;  // get_active_cell(neighbor_y, neighbor_x), preemptive.h:163
            mine++;
        }
    }
    if (mine) atomicAdd(&s_count, mine);
    __syncthreads();
    if (threadIdx.x == 0) nactive[b] = s_count;  // b_all_active <=> == K (preemptive.h:170-176)
}

// assign (+ update sums) of one row subsample with inactive clusters left out and, unless every cluster is active,
// only the pixels of active cells counted (context.cpp:218, :314-345).  One thread per pixel.
template <bool UPDATE>
__global__ void __launch_bounds__(256) k_assign_preempt(AssignParams ap, const uint32_t* __restrict__ quad,
                                                        uint16_t* __restrict__ labels, const CInfo* __restrict__ cinfo,
                                                        const int* __restrict__ cell_start,
                                                        const fslic_cluster* __restrict__ clusters,
                                                        unsigned long long* __restrict__ acc,
                                                        const uint8_t* __restrict__ cellmap, int CW2, int ncell2,
                                                        const int* __restrict__ nactive) {
    const long per_img = (long)ap.nsub * ap.W;
    const long total = per_img * ap.B;
    const int S = ap.S, W = ap.W, H = ap.H;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const int b = (int)(t / per_img);
        const long r = t - (long)b * per_img;
        const int sr = (int)(r / W), j = (int)(r - (long)sr * W);
        const int i = ap.rem + sr * ap.stride;
        const CInfo* ci = cinfo + (size_t)b * ap.K;
        const int* cs = cell_start + (size_t)b * (ap.ncell + 1);
        const fslic_cluster* cl = clusters + (size_t)b * ap.K;
        uint16_t* lb = labels + (size_t)b * H * W;
        const uint32_t q = quad[(size_t)b * H * W + (size_t)i * W + j];
        unsigned long long best = ~0ull;
        const int cr0 = max(i - S, 0) / ap.G, cr1 = min(i + S, H - 1) / ap.G;
        const int cc0 = max(j - S, 0) / ap.G, cc1 = min(j + S, W - 1) / ap.G;
        for (int cr = cr0; cr <= cr1; cr++) {
            const int s = cs[cr * ap.cellW + cc0], e = cs[cr * ap.cellW + cc1 + 1];
            for (int u = s; u < e; u++) {
                const CInfo rec = ci[u];
                const int cy = (int16_t)(rec.cyx & 0xffff), cx = rec.cyx >> 16;
                const int di = abs(i - cy), dj = abs(j - cx);
                if (di > S || dj > S) continue;
                if (!cl[rec.sortkey & 0xffffu].is_active) continue;  // context.cpp:218
                const uint32_t sp = spatial_u16(ap.coef, di, dj, ap.euclid);
                const uint32_t d = sad4_acc(q, rec.color, sp) & 0xffffu;
                const unsigned long long key = ((unsigned long long)d << 32) | rec.sortkey;
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
            label = lb[(size_t)i * W + j];  // keeps the label of an earlier pass; still counts in the update (context.cpp:318-319)
        }
        if (UPDATE && label != 0xFFFF) {
            const bool counted = nactive[b] == ap.K || cellmap[(size_t)b * ncell2 + (i / (2 * S)) * CW2 + (j / (2 * S))] != 0;
            if (counted) acc_add_pixel(acc + (size_t)b * ap.K * 4, label, i, j, q);
        }
    }
}
