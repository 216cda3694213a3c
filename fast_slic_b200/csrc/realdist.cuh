// fast_slic_b200/csrc/realdist.cuh -- the float-distance variants of the assign step (SURVEY.md section 8(f) row 3).
//
// Replaces ContextRealDist (BaseContext<float>::assign_clusters, /root/reference/src/context.cpp:259-298 with the float
// patch of :23-33), ContextRealDistL2::assign_clusters / set_spatial_patch (:394-445) and
// ContextRealDistNoQ::assign_clusters_proto<true> (:462-499).  The scheduler (assign(), :200-243) and the update's integer
// sums (:302-357) are the default path's; only the distance, the window of the NoQ variant and its float centroids
// (:375-381) differ.  Correctness first: one thread per pixel gathers over the cell grid (the structure of
// assign_pixel_generic); every float operation is written with an explicit rounding intrinsic in the order of the
// reference's object code, so labels and clusters are bit-identical (tests/test_parity_gpu.py::test_real_dist_variants).
//   VARIANT 0  d = coef * (|di| + |dj|)  +  (|dr| + |dg| + |db|)                     one multiply, one add
//   VARIANT 1  d = fma(dj', dj', di' * di')  +  (dr^2 + dg^2 + db^2),  di' = coef * di   (GCC fuses the patch like this)
//   VARIANT 2  d = |r - cr| + |g - cg| + |b - cb| + |coef (j - cx)| + |coef (i - cy)|  on float centroids, left to right
// With manhattan_spatial_dist = false (AssignParams.euclid; context.cpp:34-38, :488-491):
//   VARIANT 0  the patch is coef * hypotf(di, dj)
//   VARIANT 1  unchanged: ContextRealDistL2::set_spatial_patch ignores the flag
//   VARIANT 2  d = fma(dx, dx, fma(db, db, fma(dr, dr, dg * dg))) + dy * dy   (the -mfma object code: dy^2 once per row)
// Ties: strict '>' against the running minimum in visiting order => minimum of (d, phase, k); non-negative floats
// order like their bit patterns, so the key is  float_bits(d) << 32 | phase << 16 | k.
#pragma once
#include "assign.cuh"

template <int VARIANT, bool UPDATE>
__global__ void __launch_bounds__(256) k_assign_real(AssignParams ap, const uint32_t* __restrict__ quad,
                                                      uint16_t* __restrict__ labels, const CInfo* __restrict__ cinfo,
                                                      const int* __restrict__ cell_start,
                                                      const fslic_cluster* __restrict__ clusters,
                                                      unsigned long long* __restrict__ acc) {
    const long per_img = (long)ap.nsub * ap.W;
    const long total = per_img * ap.B;
    const int S = ap.S, W = ap.W, H = ap.H;
    const float coef = ap.coef, fS = (float)S;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const int b = (int)(t / per_img);
        const long rr = t - (long)b * per_img;
        const int sr = (int)(rr / W), j = (int)(rr - (long)sr * W);
        const int i = ap.rem + sr * ap.stride;
        const size_t img_off = (size_t)b * H * W;
        const uint32_t q = quad[img_off + (size_t)i * W + j];
        const int qr = q & 0xff, qg = (q >> 8) & 0xff, qb = (q >> 16) & 0xff;
        const CInfo* ci = cinfo + (size_t)b * ap.K;
        const int* cs = cell_start + (size_t)b * (ap.ncell + 1);
        const fslic_cluster* cl = clusters + (size_t)b * ap.K;
        unsigned long long best = ~0ull;
        const int m = S + (VARIANT == 2 ? 1 : 0);  // the NoQ window is cut from float centres: one more row / column to look at
        const int cr0 = max(i - m, 0) / ap.G, cr1 = min(i + m, H - 1) / ap.G;
        const int cc0 = max(j - m, 0) / ap.G, cc1 = min(j + m, W - 1) / ap.G;
        for (int cr = cr0; cr <= cr1; cr++) {
            const int s = cs[cr * ap.cellW + cc0], e = cs[cr * ap.cellW + cc1 + 1];
            for (int u = s; u < e; u++) {
                const CInfo r = ci[u];
                float d;
                if (VARIANT == 2) {
                    const fslic_cluster c = cl[r.sortkey & 0xffffu];
                    // context.cpp:472-473: my_max<int>(cy - S, 0) .. my_min<int>(cy + S + 1, H), float arithmetic truncated
                    const int i0 = max((int)__fsub_rn(c.y, fS), 0), i1 = min((int)__fadd_rn(__fadd_rn(c.y, fS), 1.0f), H);
                    const int j0 = max((int)__fsub_rn(c.x, fS), 0), j1 = min((int)__fadd_rn(__fadd_rn(c.x, fS), 1.0f), W);
                    if (i < i0 || i >= i1 || j < j0 || j >= j1) continue;
                    const float dr = __fsub_rn((float)qr, c.r), dg = __fsub_rn((float)qg, c.g), db = __fsub_rn((float)qb, c.b);
                    const float dy = __fmul_rn(coef, __fsub_rn((float)i, c.y)), dx = __fmul_rn(coef, __fsub_rn((float)j, c.x));
                    if (ap.euclid) {  // assign_clusters_proto<false>, context.cpp:490, as its -mfma object code evaluates it
                        float t = __fmul_rn(dg, dg);
                        t = __fmaf_rn(dr, dr, t);
                        t = __fmaf_rn(db, db, t);
                        t = __fmaf_rn(dx, dx, t);
                        d = __fadd_rn(t, __fmul_rn(dy, dy));
                    } else {
                        d = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(fabsf(dr), fabsf(dg)), fabsf(db)), fabsf(dx)), fabsf(dy));
                    }
                } else {
                    const int cy = (int16_t)(r.cyx & 0xffff), cx = r.cyx >> 16;
                    const int di = i - cy, dj = j - cx;
                    if (abs(di) > S || abs(dj) > S) continue;
                    const int cr_ = r.color & 0xff, cg_ = (r.color >> 8) & 0xff, cb_ = (r.color >> 16) & 0xff;
                    if (VARIANT == 0) {
                        const float patch = __fmul_rn(coef, ap.euclid ? ref_hypotf(di, dj) : (float)(abs(di) + abs(dj)));
                        d = __fadd_rn(patch, (float)(abs(qr - cr_) + abs(qg - cg_) + abs(qb - cb_)));
                    } else {
                        const float fdi = __fmul_rn(coef, (float)di), fdj = __fmul_rn(coef, (float)dj);
                        const float patch = __fmaf_rn(fdj, fdj, __fmul_rn(fdi, fdi));
                        const int er = qr - cr_, eg = qg - cg_, eb = qb - cb_;
                        d = __fadd_rn(patch, (float)(er * er + eg * eg + eb * eb));  // < 2^24: exact in float
                    }
                }
                const unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | r.sortkey;
                best = key < best ? key : best;
            }
        }
        uint16_t* lp = labels + img_off + (size_t)i * W + j;
        uint32_t label;
        if (best != ~0ull) {
            label = (uint32_t)(best & 0xffff);
            *lp = (uint16_t)label;
        } else if ((i % ap.cfg_stride) >= ap.fresh_from) {
            *lp = 0xFFFF;
            label = 0xFFFF;
        } else {
            label = *lp;  // no window covers the pixel: it keeps the label of an earlier pass
        }
        if (UPDATE && label != 0xFFFF) acc_add_pixel(acc + (size_t)b * ap.K * 4, label, i, j, q);
    }
}
