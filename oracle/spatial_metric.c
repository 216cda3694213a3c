/*
 * oracle/spatial_metric.c -- TEST INFRASTRUCTURE ONLY.
 *
 * The Euclidean spatial term of the reference (`manhattan_spatial_dist = false`, context.h:35) restated on top of
 * oracle/slic_oracle.c, which is included whole: scheduler order, update, preemptive bookkeeping and connectivity
 * enforcement are the very code the Manhattan restatement is checked with; only the distance differs.
 *
 *   integer path (BaseContext<uint16_t>)  patch(di, dj) = (u16)(coef * hypotf(di, dj))          context.cpp:34-38
 *   ContextRealDist (variant 0)           patch(di, dj) = coef * hypotf(di, dj), kept as float  context.cpp:34-38
 *   ContextRealDistL2 (variant 1)         unchanged: its set_spatial_patch ignores the flag     context.cpp:435-445
 *   ContextRealDistNoQ (variant 2)        dr^2 + dg^2 + db^2 + dx^2 + dy^2                      context.cpp:488-491
 *
 * hypotf: glibc's hypotf rounds the exact sqrt(a^2 + b^2) once to float.  For integer arguments that is the double
 * square root of the exact double sum, rounded to float; written that way here so that the restatement gives the same
 * answer whatever libm the machine has (tests/test_spatial_metric_cpu.py checks it against the local hypotf).
 *
 * NoQ: the reference's -O3 -mavx2 -mfma object code (objdump -d of context.o, assign_clusters_proto<false>) squares
 * dy once per row (vmulss) and per pixel computes
 *     t = dg*dg (vmulss); t = fma(dr, dr, t); t = fma(db, db, t); t = fma(dx, dx, t); d = t + dy*dy (vaddss),
 * with dr, dg, db the quad bytes 0, 1, 2 minus the centroid's r, g, b.  Restated with fmaf in that order.
 */
#include "slic_oracle.c"

float orc_ref_hypotf(int a, int b) { return (float)sqrt((double)a * (double)a + (double)b * (double)b); }

/* BaseContext<uint16_t>::set_spatial_patch, Euclidean branch (context.cpp:24-26, :34-38): (2S+1)^2, row-major */
void orc_spatial_patch_euclid(int S, float compactness, int color_shift, uint16_t* patch) {
    float coef = 1.0f / ((float)S / compactness);
    coef *= (float)(1 << color_shift);
    for (int i = 0; i <= 2 * S; i++)
        for (int j = 0; j <= 2 * S; j++) patch[i * (2 * S + 1) + j] = (uint16_t)(coef * orc_ref_hypotf(i - S, j - S));
}

/* One assign pass with the Euclidean term: the bucketed scheduler of assign_pass_bucketed / assign_pass_real
 * (context.cpp:200-243), strict '>' against min_dists.  variant -1: the u16 integer path (min_dists start at
 * 0xFFFF, numeric_limits<uint16_t>::max), 0: ContextRealDist, 2: ContextRealDistNoQ (float min_dists). */
static void assign_pass_euclid(int variant, int H, int W, int K, int S, OrcCluster* clusters, const uint8_t* quad,
                               float coef, const uint16_t* patch16, uint16_t* assignment, float* min_dists, int stride,
                               int rem) {
    const float init = variant < 0 ? 65535.0f : 3.402823466e+38f;
    for (long p = 0; p < (long)H * W; p++) min_dists[p] = init;
    for (int k = 0; k < K; k++) { /* :209-212 */
        float x = clusters[k].x, y = clusters[k].y;
        clusters[k].x = x < 0 ? 0 : (x > (float)(W - 1) ? (float)(W - 1) : x);
        clusters[k].y = y < 0 ? 0 : (y > (float)(H - 1) ? (float)(H - 1) : y);
    }
    int T = 2 * S + 32;
    int cell_W = ceil_int(W, T), cell_H = ceil_int(H, T);
    int ncell = cell_W * cell_H;
    int* start = (int*)calloc((size_t)ncell + 1, sizeof(int));
    int* items = (int*)malloc(sizeof(int) * (size_t)(K > 0 ? K : 1));
    for (int k = 0; k < K; k++) {
        if (!clusters[k].is_active) continue;
        start[cell_W * ((int)clusters[k].y / T) + ((int)clusters[k].x / T) + 1]++;
    }
    for (int c = 0; c < ncell; c++) start[c + 1] += start[c];
    int* fill = (int*)malloc(sizeof(int) * (size_t)(ncell > 0 ? ncell : 1));
    memcpy(fill, start, sizeof(int) * (size_t)ncell);
    for (int k = 0; k < K; k++) {
        if (!clusters[k].is_active) continue;
        items[fill[cell_W * ((int)clusters[k].y / T) + ((int)clusters[k].x / T)]++] = k;
    }
    const int P = 2 * S + 1;
    for (int phase = 0; phase < 4; phase++)
        for (int ci = phase / 2; ci < cell_H; ci += 2)
            for (int cj = phase % 2; cj < cell_W; cj += 2) {
                int cell = ci * cell_W + cj;
                for (int t = start[cell]; t < start[cell + 1]; t++) {
                    const OrcCluster* c = &clusters[items[t]];
                    int i0, i1, j0, j1;
                    int16_t cy = (int16_t)c->y, cx = (int16_t)c->x;
                    int16_t cr = (int16_t)c->r, cg = (int16_t)c->g, cb = (int16_t)c->b;
                    if (variant == 2) { /* :471-472 */
                        i0 = (int)(c->y - (float)S); if (i0 < 0) i0 = 0;
                        i1 = (int)(c->y + (float)S + 1.0f); if (i1 > H) i1 = H;
                        j0 = (int)(c->x - (float)S); if (j0 < 0) j0 = 0;
                        j1 = (int)(c->x + (float)S + 1.0f); if (j1 > W) j1 = W;
                        i1--; j1--;
                    } else {
                        i0 = cy - S < 0 ? 0 : cy - S; i1 = cy + S >= H ? H - 1 : cy + S;
                        j0 = cx - S < 0 ? 0 : cx - S; j1 = cx + S >= W ? W - 1 : cx + S;
                    }
                    for (int i = i0; i <= i1; i++) {
                        if (i % stride != rem) continue;
                        const float dy = coef * ((float)i - c->y), dy2 = dy * dy; /* NoQ: once per row */
                        for (int j = j0; j <= j1; j++) {
                            long p = (long)i * W + j;
                            int r = quad[4 * p], g = quad[4 * p + 1], b = quad[4 * p + 2];
                            float d;
                            if (variant < 0) { /* context.cpp:276-287 with the u16 patch */
                                d = (float)(uint16_t)(abs(r - cr) + abs(g - cg) + abs(b - cb) +
                                                      patch16[(i - cy + S) * P + (j - cx + S)]);
                            } else if (variant == 0) { /* the float patch, untruncated */
                                float patch = coef * orc_ref_hypotf(i - cy, j - cx);
                                d = patch + (float)(abs(r - cr) + abs(g - cg) + abs(b - cb));
                            } else {
                                float dr = (float)r - c->r, dg = (float)g - c->g, db = (float)b - c->b;
                                float dx = coef * ((float)j - c->x);
                                float s = dg * dg;
                                s = fmaf(dr, dr, s);
                                s = fmaf(db, db, s);
                                s = fmaf(dx, dx, s);
                                d = s + dy2;
                            }
                            if (min_dists[p] > d) {
                                min_dists[p] = d;
                                assignment[p] = c->number;
                            }
                        }
                    }
                }
            }
    free(start); free(items); free(fill);
}

/* orc_iterate_preemptive (context.cpp:109-197) with the Euclidean patch; manhattan != 0 is the original restatement */
void orc_iterate_metric(int H, int W, int K, const uint8_t* image, OrcCluster* clusters, uint16_t* out, int max_iter,
                        float compactness, float min_size_factor, int stride, int convert_to_lab, int preemptive,
                        float preemptive_thres, int manhattan, uint16_t* precca_out) {
    if (manhattan) {
        orc_iterate_preemptive(H, W, K, image, clusters, out, max_iter, compactness, min_size_factor, stride, convert_to_lab,
                               preemptive, preemptive_thres, NULL, precca_out);
        return;
    }
    if (H <= 0 || W <= 0 || K <= 0) return;
    int S = (int16_t)sqrt((double)(H * W / K)); /* context.h:60 */
    long N = (long)H * W;
    uint8_t* quad = (uint8_t*)malloc((size_t)N * 4);
    uint16_t* assignment = (uint16_t*)malloc(sizeof(uint16_t) * (size_t)N);
    float* min_dists = (float*)malloc(sizeof(float) * (size_t)N);
    uint16_t* patch = (uint16_t*)malloc(sizeof(uint16_t) * (size_t)(2 * S + 1) * (2 * S + 1));
    int color_shift = convert_to_lab ? OUTPUT_SHIFT : 0;
    orc_rgb_to_quad(image, H, W, convert_to_lab, quad); /* :114-127 */
    for (int k = 0; k < K; k++) {                       /* :128-135 */
        int y = clampi((int)clusters[k].y, 0, H - 1), x = clampi((int)clusters[k].x, 0, W - 1);
        clusters[k].r = quad[4 * ((long)y * W + x)];
        clusters[k].g = quad[4 * ((long)y * W + x) + 1];
        clusters[k].b = quad[4 * ((long)y * W + x) + 2];
    }
    for (long p = 0; p < N; p++) assignment[p] = 0xFFFF;
    orc_spatial_patch_euclid(S, compactness, color_shift, patch); /* :147 */
    for (int k = 0; k < K; k++) clusters[k].is_updatable = 2;
    int all_active = 1;
    int* active_grid = NULL;
    float* old_yx = NULL;
    if (preemptive && S > 0) {
        active_grid = (int*)calloc((size_t)ceil_int(W, 2 * S) * ceil_int(H, 2 * S), sizeof(int));
        old_yx = (float*)malloc(sizeof(float) * 2 * (size_t)K);
    }
    int rem = 0;
    for (int it = 0; it < max_iter; it++) { /* :158-175 */
        assign_pass_euclid(-1, H, W, K, S, clusters, quad, 0.f, patch, assignment, min_dists, stride, rem);
        if (active_grid) {
            for (int k = 0; k < K; k++) {
                old_yx[2 * k] = clusters[k].y;
                old_yx[2 * k + 1] = clusters[k].x;
            }
            update_pass_masked(H, W, K, clusters, quad, assignment, stride, rem, all_active ? NULL : active_grid, 2 * S,
                               ceil_int(W, 2 * S));
            all_active = set_new_clusters(H, W, K, S, preemptive_thres, clusters, old_yx, active_grid);
        } else {
            update_pass(H, W, K, clusters, quad, assignment, stride, rem);
        }
        rem = (rem + 1) % stride;
    }
    free(active_grid);
    free(old_yx);
    for (int k = 0; k < K; k++) clusters[k].is_active = 1;
    assign_pass_euclid(-1, H, W, K, S, clusters, quad, 0.f, patch, assignment, min_dists, 1, 0); /* :178-181 */
    if (precca_out) memcpy(precca_out, assignment, sizeof(uint16_t) * (size_t)N);
    memcpy(out, assignment, sizeof(uint16_t) * (size_t)N);
    int thres = (int)round((double)(S * S) * (double)min_size_factor); /* :16 */
    orc_enforce_connectivity(out, H, W, K, thres);
    free(quad); free(assignment); free(min_dists); free(patch);
}

/* orc_iterate_real with the Euclidean term; ContextRealDistL2 (variant 1) and manhattan != 0 are the original */
void orc_iterate_real_metric(int variant, int H, int W, int K, const uint8_t* image, OrcCluster* clusters, uint16_t* out,
                             int max_iter, float compactness, float min_size_factor, int stride, int convert_to_lab,
                             int manhattan, uint16_t* precca_out) {
    if (manhattan || variant == 1) {
        orc_iterate_real(variant, H, W, K, image, clusters, out, max_iter, compactness, min_size_factor, stride,
                         convert_to_lab, precca_out);
        return;
    }
    if (H <= 0 || W <= 0 || K <= 0) return;
    int S = (int16_t)sqrt((double)(H * W / K));
    long N = (long)H * W;
    uint8_t* quad = (uint8_t*)malloc((size_t)N * 4);
    uint16_t* assignment = (uint16_t*)malloc(sizeof(uint16_t) * (size_t)N);
    float* min_dists = (float*)malloc(sizeof(float) * (size_t)N);
    int color_shift = convert_to_lab ? OUTPUT_SHIFT : 0;
    orc_rgb_to_quad(image, H, W, convert_to_lab, quad);
    for (int k = 0; k < K; k++) {
        int y = clampi((int)clusters[k].y, 0, H - 1), x = clampi((int)clusters[k].x, 0, W - 1);
        clusters[k].r = quad[4 * ((long)y * W + x)];
        clusters[k].g = quad[4 * ((long)y * W + x) + 1];
        clusters[k].b = quad[4 * ((long)y * W + x) + 2];
    }
    for (long p = 0; p < N; p++) assignment[p] = 0xFFFF;
    float coef = 1.0f / ((float)S / compactness);
    coef *= (float)(1 << color_shift);
    for (int k = 0; k < K; k++) clusters[k].is_updatable = 2;
    int rem = 0;
    for (int it = 0; it < max_iter; it++) {
        assign_pass_euclid(variant, H, W, K, S, clusters, quad, coef, NULL, assignment, min_dists, stride, rem);
        update_pass_real(variant, H, W, K, clusters, quad, assignment, stride, rem);
        rem = (rem + 1) % stride;
    }
    for (int k = 0; k < K; k++) clusters[k].is_active = 1;
    assign_pass_euclid(variant, H, W, K, S, clusters, quad, coef, NULL, assignment, min_dists, 1, 0);
    if (precca_out) memcpy(precca_out, assignment, sizeof(uint16_t) * (size_t)N);
    memcpy(out, assignment, sizeof(uint16_t) * (size_t)N);
    int thres = (int)round((double)(S * S) * (double)min_size_factor);
    orc_enforce_connectivity(out, H, W, K, thres);
    free(quad); free(assignment); free(min_dists);
}
