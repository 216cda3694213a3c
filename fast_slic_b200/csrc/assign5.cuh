// fast_slic_b200/csrc/assign5.cuh -- the assign + update hot loop, TMA-staged (round 2).
//
// Same contract as k_assign_warp (assign.cuh; /root/reference/src/context.cpp:200-298 assign / assign_clusters,
// :302-387 update; AVX2 form arch/x64/avx2.h:11-185): every pixel of the active rows takes the lexicographic
// minimum of (d, phase, k) over the clusters whose (2S+1)^2 window covers it, pixels no window covers keep
// their label, and the per-cluster sums of the update are accumulated exactly.  What changed is where the
// instructions go.  k_assign_warp spent 77 % of its issue slots outside the distance loop (ncu, round 1):
// per-tile candidate lists built by 8 lanes each, 64-bit address arithmetic and bounds predicates around
// every LDG/STG, a four-way one-hot compare per MMA.  Here:
//
//   * quad tiles arrive by TMA: one elected lane per warp issues cp.async.bulk.tensor.3d (3-D tensor map
//     (x, sub-row, image) whose row stride is `stride` image rows, so the sub-sampled rows land as a dense
//     [4][32*TPS] tile in the warp's shared block); completion on a per-warp mbarrier; the load of the
//     NEXT super tile is in flight while this one is processed.  Out-of-image parts of a box are zero-filled
//     by the hardware: no bounds predicates on the loads.
//   * labels leave by TMA: lanes put u16 labels into a [4][32*TPS] staging tile, one bulk tensor store per
//     super tile writes them (clipped by the hardware at the image edge).  Super tiles that contain a pixel
//     no window covers -- or that the image edge clips -- take a per-pixel store path instead, which also
//     implements "keep the previous label" (context.cpp:289-294 never fires for such pixels).
//   * ONE candidate list per super tile (32*TPS columns x 4 sub-rows): <= 32 candidates, one lane each,
//     ranked once by (phase, k) with vector loads of the keys; the per-tile lists are derived from it with a
//     REDUX.OR bit mask per tile (bit = rank), so a candidate's position in a tile list is a popcount and
//     the lists stay in visiting order without any per-tile sort.
//   * update: the one-hot operand needs 3 instead of 4 logic ops per word (rank bytes stay below 0x80),
//     and the second half of the MMA A operand (candidates 8..15) is skipped when a tile has <= 8.
//   * code generation: under the 64-register budget the compiler re-derived every shared-memory address from
//     threadIdx (and the loop constants from integer divisions) at each use -- a fifth of all instructions in
//     the first version of this kernel.  So: the warp-uniform walk constants come precomputed from the host
//     (constant bank), the warp's shared block is addressed through ONE opaque 32-bit base register, and every
//     access to it is an explicit ld.shared / st.shared with an immediate offset.
//
// HBM per processed pixel: 4 B quad read + 2 B label written, as before.
#pragma once
#include <cuda.h>  // CUtensorMap (types only; the encoder is fetched through cudaGetDriverEntryPoint, no libcuda link)

#include "assign.cuh"

#define A5_MAXWARPS 32
#define A5_WBLK 5504     // bytes of shared memory per warp (multiple of 128: TMA destinations need 128-byte alignment)
#define A5_OFF_QUAD 0    // [4][32*TPS] u32  quad tile                      (<= 2048 B)
#define A5_OFF_LAB 2048  // [4][32*TPS] u16  label staging tile             (<= 1024 B)
#define A5_OFF_ENT 3072  // [4][32] uint2    per tile {colour, patch offset} in visiting order (1024 B)
#define A5_OFF_TK 4096   // [4][40] u16      per tile cluster number in visiting order; [t][32] = 0xFFFE (320 B)
#define A5_TK_PITCH 80
#define A5_OFF_SCR 4416  // 1024 B scratch: CInfo[32] + keys[32] while the list is built; MMA staging [32][8] u32 afterwards
#define A5_OFF_KEY (A5_OFF_SCR + 512)
#define A5_OFF_BAR 5440  // the warp's mbarrier
#define A5_BIGKEY (FSLIC_BIGSP << 16)
#define A5_NOCAND 32u    // rank byte of a pixel that contributes to no candidate: matches none of 0..31, indexes the 0xFFFE slot

__device__ __forceinline__ uint32_t a5_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// explicit shared-window accesses: address register + immediate offset
template <int OFF> __device__ __forceinline__ uint32_t a5_lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(a), "n"(OFF));
    return v;
}
template <int OFF> __device__ __forceinline__ uint32_t a5_lds16(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1+%2];" : "=r"(v) : "r"(a), "n"(OFF));
    return v;
}
template <int OFF> __device__ __forceinline__ uint4 a5_lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4+%5];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a), "n"(OFF));
    return v;
}
template <int OFF> __device__ __forceinline__ void a5_sts16(uint32_t a, uint32_t v) {
    asm volatile("st.shared.u16 [%0+%1], %2;" ::"r"(a), "n"(OFF), "r"(v) : "memory");
}
template <int OFF> __device__ __forceinline__ void a5_sts32(uint32_t a, uint32_t v) {
    asm volatile("st.shared.u32 [%0+%1], %2;" ::"r"(a), "n"(OFF), "r"(v) : "memory");
}
template <int OFF> __device__ __forceinline__ void a5_sts64(uint32_t a, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.u32 [%0+%1], {%2,%3};" ::"r"(a), "n"(OFF), "r"(x), "r"(y) : "memory");
}
template <int OFF> __device__ __forceinline__ void a5_sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.shared.v4.u32 [%0+%1], {%2,%3,%4,%5};" ::"r"(a), "n"(OFF), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}

__device__ __forceinline__ void a5_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void a5_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void a5_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "A5_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra A5_DONE;\n"
        "bra A5_WAIT;\n"
        "A5_DONE:\n"
        "}" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void a5_tma_load_3d(uint32_t dst, const CUtensorMap* map, int x, int y, int z, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(z), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void a5_tma_store_3d(const CUtensorMap* map, uint32_t src, int x, int y, int z) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(map)),
                 "r"(src), "r"(x), "r"(y), "r"(z)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void a5_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void a5_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// prmt.b32, generic mode: result byte i = byte (sel nibble i & 7) of {a, b}, or that byte's sign replicated when the
// nibble's bit 3 is set
__device__ __forceinline__ uint32_t a5_prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}

// per-byte equality of two words whose bytes are all below 0x80 -> 0x80 in every equal byte (3 logic ops)
__device__ __forceinline__ uint32_t eq7(uint32_t w, uint32_t m) { return ~((w ^ m) + 0x7f7f7f7fu) & 0x80808080u; }

template <int TS, int STRIDE, bool UPDATE, int TPS, bool FUSE = false>
__global__ void __launch_bounds__(32 * A5_MAXWARPS, 1)
    k_assign5(const __grid_constant__ AssignParams ap, const __grid_constant__ CUtensorMap tm_quad,
              const __grid_constant__ CUtensorMap tm_lab, const uint32_t* __restrict__ quad, uint16_t* __restrict__ labels,
              const CInfo* __restrict__ cinfo, const int* __restrict__ cell_start, unsigned long long* __restrict__ acc,
              const uint16_t* __restrict__ g_tbl, fslic_cluster* clusters, CInfo* cinfo_next, int* cell_start_next,
              unsigned int* ticket) {
    constexpr int R = 4;                      // sub-rows per tile (one per register of a lane)
    constexpr int BW = 32 * TPS;              // columns of a super tile == TMA box width
    constexpr uint32_t QBYTES = BW * R * 4;   // bytes one quad box delivers (out-of-image parts included: zero fill)
    constexpr int ROWB = 2 * STRIDE * TS;     // patch bytes between two sub-rows
    static_assert(STRIDE >= 1, "the sub-row pitch is an immediate of the patch loads");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const uint32_t sbase = a5_smem(smem_raw);
    uint32_t lane = threadIdx.x & 31u;
    uint32_t wb = sbase + ap.tbl_bytes + (threadIdx.x >> 5) * A5_WBLK;  // this warp's shared block
    // opaque from here on: the compiler keeps the two registers instead of re-deriving them from threadIdx at each use
    asm volatile("" : "+r"(wb), "+r"(lane));
    const uint32_t bar = wb + A5_OFF_BAR;

    if (lane == 0) a5_mbar_init(bar, 1);
    if (lane < TPS) a5_sts16<A5_OFF_TK + 2 * A5_NOCAND>(wb + lane * A5_TK_PITCH, 0xFFFEu);  // "not covered" marker
    {   // the spatial patch, once per CTA (16-byte copies; the table is padded to a multiple of 8 elements)
        const uint4* src = reinterpret_cast<const uint4*>(g_tbl);
        uint4* dst = reinterpret_cast<uint4*>(smem_raw);
        for (int t = threadIdx.x; t < (ap.tbl_elems + 7) / 8; t += blockDim.x) dst[t] = src[t];
    }
    __syncthreads();

    const int S = ap.S, W = ap.W, H = ap.H;
    constexpr int stride = STRIDE;
    const uint32_t lt_mask = (1u << lane) - 1u;

    // super-tile walk without divisions: (b, ty, sx) advance by the host's (db, dty, dsx) with carries
    int st = (int)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5));
    int b = st / ap.per_img;
    int ty, sx;
    {
        const int tl0 = st - b * ap.per_img;
        ty = tl0 / ap.stx;
        sx = tl0 - ty * ap.stx;
    }
    uint32_t phase = 0;
    bool store_pending = false;  // warp uniform: a bulk store of this warp's staging tile may still be reading it
    if (st < ap.total && lane == 0) {
        a5_mbar_expect_tx(bar, QBYTES);
        a5_tma_load_3d(wb + A5_OFF_QUAD, &tm_quad, sx * BW, ty * R, b, bar);
    }

    for (; st < ap.total; st += ap.wstride) {
        // the super tile after this one (its quad box is requested while this one is processed)
        int nb = b + ap.db, nty = ty + ap.dty, nsx = sx + ap.dsx;
        if (nsx >= ap.stx) { nsx -= ap.stx; nty += 1; }
        if (nty >= ap.tiles_y) { nty -= ap.tiles_y; nb += 1; }
        const bool has_next = st + ap.wstride < ap.total;

        const int wsr0 = ty * R;
        const int nrow = min(R, ap.nsub - wsr0);  // valid sub-rows of this tile row (>= 1)
        const int wi0 = ap.rem + wsr0 * stride, wi1 = wi0 + (nrow - 1) * stride;
        const int sj0 = sx * BW, sj1 = min(sj0 + BW, W) - 1;
        const int ntile = min(TPS, ap.tiles_x - sx * TPS);  // tiles of this super tile that start inside the image
        const bool edge = (sj0 + BW > W) || (nrow < R);
        const CInfo* ci = reinterpret_cast<const CInfo*>(reinterpret_cast<const char*>(cinfo) + (size_t)((uint32_t)b * (uint64_t)ap.cinfo_img_bytes));
        const int* cs = reinterpret_cast<const int*>(reinterpret_cast<const char*>(cell_start) + (size_t)((uint32_t)b * (uint64_t)ap.cells_img_bytes));
        unsigned long long* ac = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(acc) + (size_t)((uint32_t)b * (uint64_t)ap.acc_img_bytes));

        // ---- L. the candidate list of the super tile: clusters with cy in [wi0-S, wi1+S], cx in [sj0-S, sj1+S] ----
        int n = 0;            // candidates found (warp uniform)
        uint32_t ncnt = 0;    // per-tile list lengths, one byte each
        {
            const int ylo = wi0 - S, yhi = wi1 + S, xlo = sj0 - S, xhi = sj1 + S;
            const int cr0 = div_g(max(ylo, 0), ap.Ginv), cr1 = div_g(min(yhi, H - 1), ap.Ginv);
            const int cc0 = div_g(max(xlo, 0), ap.Ginv), cc1 = div_g(min(xhi, W - 1), ap.Ginv);
            const int nr = cr1 - cr0 + 1;  // cell rows: one contiguous range of the cell-sorted records each
            int rs = 0, cnt = 0;
            if ((int)lane < nr) {
                const int* p = cs + (cr0 + (int)lane) * ap.cellW;
                rs = p[cc0];
                cnt = p[cc1 + 1] - rs;
            }
            int incl = cnt;  // inclusive scan over the nr ranges
            for (int o = 1; o < nr; o <<= 1) {
                const int y = __shfl_up_sync(FSLIC_FULL, incl, o);
                if ((int)lane >= o) incl += y;
            }
            const int T = __shfl_sync(FSLIC_FULL, incl, min(nr, 32) - 1);
            if (nr > 32) n = 33;  // cannot happen for G >= S (at most ~9 cell rows); treated like an overflow
            for (int t0 = 0; t0 < T && n <= 32; t0 += 32) {
                const int t = t0 + (int)lane;
                int row = 0;  // range of flat index t: the first one whose inclusive prefix exceeds t
                for (int r = 0; r < nr - 1; r++) row += (t >= __shfl_sync(FSLIC_FULL, incl, r));
                const int rincl = __shfl_sync(FSLIC_FULL, incl, row);
                const int rcnt = __shfl_sync(FSLIC_FULL, cnt, row);
                const int rstart = __shfl_sync(FSLIC_FULL, rs, row);
                bool hit = false;
                uint4 rec = make_uint4(0, 0, 0, 0);  // CInfo: x = cyx, y = colour, z = sort key
                if (t < T) {
                    rec = *reinterpret_cast<const uint4*>(ci + (rstart + (t - (rincl - rcnt))));
                    const int cy = (int16_t)(rec.x & 0xffff), cx = (int)rec.x >> 16;
                    hit = (cy >= ylo) && (cy <= yhi) && (cx >= xlo) && (cx <= xhi);
                }
                const unsigned m = __ballot_sync(FSLIC_FULL, hit);
                const int slot = n + __popc(m & lt_mask);
                if (hit && slot < 32) {
                    a5_sts128<A5_OFF_SCR>(wb + slot * 16, rec.x, rec.y, rec.z, rec.w);
                    a5_sts32<A5_OFF_KEY>(wb + slot * 4, rec.z);
                }
                n += __popc(m);
            }
            // pad the key vector to a multiple of 4 with +infinity (keys are phase << 16 | k < 2^18, all distinct)
            if (n <= 32 && (int)lane >= n && (int)lane < ((n + 3) & ~3)) a5_sts32<A5_OFF_KEY>(wb + lane * 4, 0xffffffffu);
            __syncwarp();
            if (n <= 32) {
                // lane a holds candidate a; rank = position in the reference's visiting order (context.cpp:214-242)
                const bool mine = (int)lane < n;
                uint4 rec = make_uint4(0, 0, 0xffffffffu, 0);
                if (mine) rec = a5_lds128<A5_OFF_SCR>(wb + lane * 16);
                const uint32_t key = rec.z;
                int rank = 0;
                uint32_t ka = wb;
                for (int u = 0; u < n; u += 4, ka += 16) {
                    const uint4 k4 = a5_lds128<A5_OFF_KEY>(ka);
                    rank += (k4.x < key) + (k4.y < key) + (k4.z < key) + (k4.w < key);
                }
                const int cy = (int16_t)(rec.x & 0xffff), cx = (int)rec.x >> 16;
                const uint32_t off = (uint32_t)(2 * ((ap.OY - cy) * TS + (ap.OX - cx)));
                const uint32_t rbit = mine ? (1u << rank) : 0u;
                const uint32_t below = rbit - 1u;
                const int cxr = cx - (sj0 - S);  // tile t lists the candidate iff 0 <= cxr - 32 t <= 2S + 31
                // tile t lists the candidates whose window can touch its 32 columns; bit r of the tile's mask <=>
                // the rank-r candidate is listed, so list position = number of listed candidates of smaller rank
#define A5_TILE_LIST(t)                                                                                  \
    if (t < TPS) {                                                                                       \
        const bool h = mine && ((unsigned)(cxr - 32 * t) <= (unsigned)(2 * S + 31));                     \
        const uint32_t mt = __reduce_or_sync(FSLIC_FULL, h ? rbit : 0u);                                 \
        if (h) {                                                                                         \
            const uint32_t pos = (uint32_t)__popc(mt & below);                                           \
            a5_sts64<A5_OFF_ENT + 256 * t>(wb + pos * 8, rec.y, off);                                    \
            a5_sts16<A5_OFF_TK + A5_TK_PITCH * t>(wb + pos * 2, rec.z & 0xffffu);                        \
        }                                                                                                \
        ncnt |= (uint32_t)__popc(mt) << (8 * t);                                                         \
    }
                A5_TILE_LIST(0) A5_TILE_LIST(1) A5_TILE_LIST(2) A5_TILE_LIST(3)
#undef A5_TILE_LIST
            }
            __syncwarp();
        }
        const bool ovf = n > 32;  // clusters piled on one spot: brute force for this super tile

        // ---- the quad tile of this super tile has landed; the staging tile is free again ----
        a5_mbar_wait(bar, phase);
        phase ^= 1u;
        if (store_pending) {
            if (lane == 0) a5_store_wait_read();
            __syncwarp();
            store_pending = false;
        }

        bool slow = false;  // warp uniform: the super tile needs the per-pixel store path
#pragma unroll 1
        for (int tq = 0; tq < ntile; tq++) {
            const int n_t = (int)((ncnt >> (8 * tq)) & 0xffu);
            const int tj0 = sj0 + 32 * tq;
            const int j = tj0 + (int)lane;
            const bool last = tq == ntile - 1;
            const uint32_t lq = wb + lane * 4 + tq * 128;            // this lane's pixel column in the quad tile
            const uint32_t ll = wb + lane * 2 + tq * 64;             // ... in the label staging tile
            const uint32_t et = wb + tq * 256;                       // this tile's entry list
            const uint32_t tk = wb + tq * A5_TK_PITCH;               // this tile's cluster numbers

            // ---- 1. pixels ----
            uint32_t q[R];
            q[0] = a5_lds32<A5_OFF_QUAD + 0 * BW * 4>(lq);
            q[1] = a5_lds32<A5_OFF_QUAD + 1 * BW * 4>(lq);
            q[2] = a5_lds32<A5_OFF_QUAD + 2 * BW * 4>(lq);
            q[3] = a5_lds32<A5_OFF_QUAD + 3 * BW * 4>(lq);

            if (ovf) {
                // ---- overflow: brute force straight from the cell grid, direct stores and atomics ----
                const size_t img_off = (size_t)b * H * W;
#pragma unroll
                for (int rr = 0; rr < R; rr++) {
                    if (j < W && rr < nrow) {
                        const int i = wi0 + rr * stride;
                        const uint32_t label = assign_pixel_generic(ap, i, j, q[rr], ci, cs, labels + img_off, [&](int di, int dj) {
                            return lds_u16(sbase + 2u * (uint32_t)((di + ap.OY) * TS + (dj + ap.OX)));
                        });
                        if (UPDATE && label != 0xFFFF) acc_add_pixel(ac, label, i, j, q[rr]);
                    }
                }
                if (last) {
                    __syncwarp();
                    if (has_next && lane == 0) {
                        a5_mbar_expect_tx(bar, QBYTES);
                        a5_tma_load_3d(wb + A5_OFF_QUAD, &tm_quad, nsx * BW, nty * R, nb, bar);
                    }
                }
                continue;
            }

            // ---- 2. distances ----
            // every (row, column) of the footprint is inside the patch for every listed candidate, valid or not.
            // patch entry of (row rr, candidate c) at shared byte address row0 + c.offset + rr * 2*stride*TS
            const uint32_t rowp = sbase + 2u * (uint32_t)(wi0 * TS + j);
            uint32_t best0 = 0xffffffffu, best1 = 0xffffffffu, best2 = 0xffffffffu, best3 = 0xffffffffu;
            {
                int c = 0;
                uint32_t ea = et;
#pragma unroll 2
                for (; c + 2 <= n_t; c += 2, ea += 16) {
                    const uint4 e = a5_lds128<A5_OFF_ENT>(ea);  // two entries: {colour, offset} x 2
                    const uint32_t p0 = rowp + e.y, p1 = rowp + e.w;
                    const uint32_t c1 = (uint32_t)c + 1u;
                    best0 = min(best0, min(sad4_acc(q[0], e.x, a5_lds16<0 * ROWB>(p0)) * 65536u + (uint32_t)c,
                                           sad4_acc(q[0], e.z, a5_lds16<0 * ROWB>(p1)) * 65536u + c1));
                    best1 = min(best1, min(sad4_acc(q[1], e.x, a5_lds16<1 * ROWB>(p0)) * 65536u + (uint32_t)c,
                                           sad4_acc(q[1], e.z, a5_lds16<1 * ROWB>(p1)) * 65536u + c1));
                    best2 = min(best2, min(sad4_acc(q[2], e.x, a5_lds16<2 * ROWB>(p0)) * 65536u + (uint32_t)c,
                                           sad4_acc(q[2], e.z, a5_lds16<2 * ROWB>(p1)) * 65536u + c1));
                    best3 = min(best3, min(sad4_acc(q[3], e.x, a5_lds16<3 * ROWB>(p0)) * 65536u + (uint32_t)c,
                                           sad4_acc(q[3], e.z, a5_lds16<3 * ROWB>(p1)) * 65536u + c1));
                }
                if (c < n_t) {
                    const uint32_t ex = a5_lds32<A5_OFF_ENT>(ea), p0 = rowp + a5_lds32<A5_OFF_ENT + 4>(ea);
                    best0 = min(best0, sad4_acc(q[0], ex, a5_lds16<0 * ROWB>(p0)) * 65536u + (uint32_t)c);
                    best1 = min(best1, sad4_acc(q[1], ex, a5_lds16<1 * ROWB>(p0)) * 65536u + (uint32_t)c);
                    best2 = min(best2, sad4_acc(q[2], ex, a5_lds16<2 * ROWB>(p0)) * 65536u + (uint32_t)c);
                    best3 = min(best3, sad4_acc(q[3], ex, a5_lds16<3 * ROWB>(p0)) * 65536u + (uint32_t)c);
                }
            }
            if (last) {
                // every lane has consumed its pixels of the last tile: the quad buffer may be overwritten
                __syncwarp();
                if (has_next && lane == 0) {
                    a5_mbar_expect_tx(bar, QBYTES);
                    a5_tma_load_3d(wb + A5_OFF_QUAD, &tm_quad, nsx * BW, nty * R, nb, bar);
                }
            }

            // ---- 3. labels into the staging tile ----
            if (edge) {  // pixels outside the image lose: the super tile takes the per-pixel store path anyway
                const uint32_t colbad = (j >= W) ? 0xffffffffu : 0u;
                best0 |= colbad;
                best1 |= colbad | ((1 < nrow) ? 0u : 0xffffffffu);
                best2 |= colbad | ((2 < nrow) ? 0u : 0xffffffffu);
                best3 |= colbad | ((3 < nrow) ? 0u : 0xffffffffu);
            }
            // rank byte per row: the winning candidate's position in the tile list, or A5_NOCAND
            const uint32_t rb0 = best0 < A5_BIGKEY ? (best0 & 0xffu) : A5_NOCAND;
            const uint32_t rb1 = best1 < A5_BIGKEY ? (best1 & 0xffu) : A5_NOCAND;
            const uint32_t rb2 = best2 < A5_BIGKEY ? (best2 & 0xffu) : A5_NOCAND;
            const uint32_t rb3 = best3 < A5_BIGKEY ? (best3 & 0xffu) : A5_NOCAND;
            a5_sts16<A5_OFF_LAB + 0 * BW * 2>(ll, a5_lds16<A5_OFF_TK>(tk + rb0 * 2));  // [32] holds 0xFFFE: "not covered"
            a5_sts16<A5_OFF_LAB + 1 * BW * 2>(ll, a5_lds16<A5_OFF_TK>(tk + rb1 * 2));
            a5_sts16<A5_OFF_LAB + 2 * BW * 2>(ll, a5_lds16<A5_OFF_TK>(tk + rb2 * 2));
            a5_sts16<A5_OFF_LAB + 3 * BW * 2>(ll, a5_lds16<A5_OFF_TK>(tk + rb3 * 2));
            const uint32_t rw = __byte_perm(__byte_perm(rb0, rb1, 0x3340), __byte_perm(rb2, rb3, 0x3340), 0x5410);
            const bool tile_cov = __all_sync(FSLIC_FULL, max(max(best0, best1), max(best2, best3)) < A5_BIGKEY);
            if (!tile_cov) slow = true;

            // ---- 4. update sums on the tensor cores (context.cpp:316-327) ----
            if (UPDATE) {
                // D[candidate][feature] += OneHot[candidate][pixel] * F[pixel][feature]   (m16n8k32, u8 x u8 -> s32)
                //   A = one-hot of the winning rank, built in registers (16 candidates per pass);
                //   B = [1, row, lane, L, a, b, 0, 0] per pixel, staged in shared memory.
                // Lane (g, tig) ends up with features (2 tig, 2 tig + 1) of candidates g and g + 8: exactly the two
                // halves of packed accumulator word tig.
                const uint32_t g = lane >> 2, tig = lane & 3u;  // MMA fragment coordinates
                const uint32_t lo01 = __byte_perm(q[0], q[1], 0x5140), lo23 = __byte_perm(q[2], q[3], 0x5140);
                const uint32_t hi01 = __byte_perm(q[0], q[1], 0x0062), hi23 = __byte_perm(q[2], q[3], 0x0062);
                const uint32_t fa = wb + lane * 32;
                a5_sts128<A5_OFF_SCR>(fa, 0x01010101u, 0x03020100u, lane * 0x01010101u, __byte_perm(lo01, lo23, 0x5410));
                a5_sts128<A5_OFF_SCR + 16>(fa, __byte_perm(lo01, lo23, 0x7632), __byte_perm(hi01, hi23, 0x5410), 0u, 0u);
                __syncwarp();
                const uint32_t fb = wb + tig * 32 + g * 4;  // feature g of pixel lanes tig, tig + 4 (+ 8 s4)
                const uint32_t flo = tig == 1 ? (uint32_t)tj0 : 0u, fhi = tig == 0 ? (uint32_t)wi0 : 0u;
                const uint32_t fmul = tig == 0 ? (uint32_t)stride : 1u;
                const int n16 = (n_t + 15) >> 4;
                // Common case (every pixel of the tile covered, at most 16 candidates): the ranks fit a nibble, and ONE
                // PRMT turns four of them into the one-hot bytes of candidate row g -- the selector nibble picks byte
                // (rank & 7) of an 8-byte pool that holds 0x80 at position g only, and its bit 3 (rank >= 8) replicates
                // that byte's sign: 0x80 <=> rank == g, 0xFF <=> rank == g + 8, 0 otherwise.
                const bool nib = tile_cov && n_t <= 16;
                uint32_t rw16 = 0, plo = 0, phi = 0;
                if (nib) {
                    rw16 = __byte_perm(rw | (rw >> 4), 0u, 0x4420);
                    plo = g < 4 ? (0x80u << (8 * g)) : 0u;
                    phi = g >= 4 ? (0x80u << (8 * (g - 4))) : 0u;
                }
                for (int nt = 0; nt < n16; nt++) {
                    int d[4] = {0, 0, 0, 0};
                    const uint32_t mg0 = (uint32_t)(nt * 16 + (int)g) * 0x01010101u, mg1 = mg0 + 0x08080808u;
                    const bool two = n_t > nt * 16 + 8;  // candidates g + 8 exist in this pass
                    if (nib) {
#define A5_MMAN(s4)                                                                                         \
    {                                                                                                       \
        const uint32_t w0 = __shfl_sync(FSLIC_FULL, rw16, 8 * s4 + tig), w1 = __shfl_sync(FSLIC_FULL, rw16, 8 * s4 + 4 + tig); \
        const uint32_t r0 = a5_prmt(plo, phi, w0), r1 = a5_prmt(plo, phi, w1);                              \
        const uint32_t t0 = r0 + r0, t1 = r1 + r1;                                                          \
        mma_u8_16x8x32(d, r0 & ~t0 & 0x80808080u, t0 & 0x80808080u, r1 & ~t1 & 0x80808080u, t1 & 0x80808080u, \
                       a5_lds32<A5_OFF_SCR + 256 * s4>(fb), a5_lds32<A5_OFF_SCR + 256 * s4 + 128>(fb));     \
    }
#define A5_MMAN1(s4)                                                                                        \
    {                                                                                                       \
        const uint32_t w0 = __shfl_sync(FSLIC_FULL, rw16, 8 * s4 + tig), w1 = __shfl_sync(FSLIC_FULL, rw16, 8 * s4 + 4 + tig); \
        mma_u8_16x8x32(d, a5_prmt(plo, phi, w0), 0u, a5_prmt(plo, phi, w1), 0u,                             \
                       a5_lds32<A5_OFF_SCR + 256 * s4>(fb), a5_lds32<A5_OFF_SCR + 256 * s4 + 128>(fb));     \
    }
                        if (two) {
                            A5_MMAN(0) A5_MMAN(1) A5_MMAN(2) A5_MMAN(3)
                        } else {  // all ranks below 8: the selected byte is the one-hot byte itself
                            A5_MMAN1(0) A5_MMAN1(1) A5_MMAN1(2) A5_MMAN1(3)
                        }
#undef A5_MMAN
#undef A5_MMAN1
                    } else if (two) {
#define A5_MMA2(s4)                                                                                         \
    {                                                                                                       \
        const uint32_t w0 = __shfl_sync(FSLIC_FULL, rw, 8 * s4 + tig), w1 = __shfl_sync(FSLIC_FULL, rw, 8 * s4 + 4 + tig); \
        mma_u8_16x8x32(d, eq7(w0, mg0), eq7(w0, mg1), eq7(w1, mg0), eq7(w1, mg1),                           \
                       a5_lds32<A5_OFF_SCR + 256 * s4>(fb), a5_lds32<A5_OFF_SCR + 256 * s4 + 128>(fb));     \
    }
                        A5_MMA2(0) A5_MMA2(1) A5_MMA2(2) A5_MMA2(3)
#undef A5_MMA2
                    } else {
#define A5_MMA1(s4)                                                                                         \
    {                                                                                                       \
        const uint32_t w0 = __shfl_sync(FSLIC_FULL, rw, 8 * s4 + tig), w1 = __shfl_sync(FSLIC_FULL, rw, 8 * s4 + 4 + tig); \
        mma_u8_16x8x32(d, eq7(w0, mg0), 0u, eq7(w1, mg0), 0u, a5_lds32<A5_OFF_SCR + 256 * s4>(fb),          \
                       a5_lds32<A5_OFF_SCR + 256 * s4 + 128>(fb));                                          \
    }
                        A5_MMA1(0) A5_MMA1(1) A5_MMA1(2) A5_MMA1(3)
#undef A5_MMA1
                    }
                    // sums are scaled by 128 (the one-hot byte is 0x80).  Packed accumulator word `tig` of a candidate:
                    //   tig 0: n | sum_y << 32   = v0            | (v1 * stride + n * wi0) << 32     (v0 = n, v1 = sum of row indices)
                    //   tig 1: sum_x | sum_L<<32 = v0 + n * tj0  | v1 << 32                          (v0 = sum of lane indices)
                    //   tig 2: sum_a | sum_b<<32 = v0            | v1 << 32
                    // i.e. lo = v0 + n * flo, hi = v1 * fmul + n * fhi with three per-lane constants: no branches.
#pragma unroll
                    for (int hh = 0; hh < 2; hh++) {
                        if (hh == 1 && !two) break;
                        const int c = nt * 16 + (int)g + 8 * hh;
                        const uint32_t v0 = (uint32_t)d[2 * hh] >> 7, v1 = (uint32_t)d[2 * hh + 1] >> 7;
                        const uint32_t cnt = __shfl_sync(FSLIC_FULL, v0, lane & ~3u);  // feature 0 lives in the tig = 0 lane
                        if (c < n_t && tig < 3 && cnt != 0) {
                            const uint32_t lo = v0 + cnt * flo, hi = v1 * fmul + cnt * fhi;
                            atomicAdd(&ac[a5_lds16<A5_OFF_TK>(tk + (uint32_t)c * 2) * 4 + tig],
                                      (unsigned long long)lo | ((unsigned long long)hi << 32));
                        }
                    }
                }
                __syncwarp();  // the MMA staging is rewritten by the next tile / the next list
            }
        }

        // ---- 5. labels out ----
        if (!ovf) {
            if (!slow) {
                a5_fence_async();  // the staging tile was written through the generic proxy
                __syncwarp();
                if (lane == 0) a5_tma_store_3d(&tm_lab, wb + A5_OFF_LAB, sj0, wsr0, b);
                store_pending = true;
            } else {
                // per-pixel path: the image edge clips this super tile, or some pixel is covered by no window
                __syncwarp();
                const size_t img_off = (size_t)b * H * W;
                for (int tq = 0; tq < ntile; tq++) {
                    const int j = sj0 + 32 * tq + (int)lane;
                    if (j >= W) continue;
                    for (int rr = 0; rr < nrow; rr++) {
                        const int i = wi0 + rr * stride;
                        const uint32_t v = a5_lds16<A5_OFF_LAB>(wb + (uint32_t)(rr * BW + 32 * tq + (int)lane) * 2);
                        uint16_t* lp = labels + img_off + (size_t)i * W + j;
                        if (v != 0xFFFEu) {
                            *lp = (uint16_t)v;
                        } else if ((i % ap.cfg_stride) >= ap.fresh_from) {
                            *lp = 0xFFFF;  // never assigned before: the reference's map still holds 0xFFFF here
                        } else if (UPDATE) {  // a stale label from an earlier pass still counts (context.cpp:318-319)
                            const uint16_t old = *lp;
                            if (old != 0xFFFF) acc_add_pixel(ac, old, i, j, quad[img_off + (size_t)i * W + j]);
                        }
                    }
                }
            }
        }
        __syncwarp();  // list staging, staging tile and MMA staging are rewritten by the next super tile
        b = nb; ty = nty; sx = nsx;
    }
    if (store_pending && lane == 0) a5_store_wait_read();  // the staging tile must outlive the last bulk store's read
    if (UPDATE && FUSE) {
        // Small batches: the bookkeeping between two passes (k_prepare3's work) runs right here, in the last CTA to
        // finish, instead of in a kernel of its own.  cinfo_next / cell_start_next alias cinfo / cell_start: they are
        // written only after every CTA of the grid has taken its ticket, i.e. has read them for the last time.
        __shared__ int s_last;
        __threadfence();  // this thread's RED.64 are performed before its CTA's ticket is
        __syncthreads();
        if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1u) ? 1 : 0;
        __syncthreads();
        if (s_last) {
            if (threadIdx.x == 0) *ticket = 0u;  // zero between launches
            __threadfence();
            PrepParams pp;
            pp.H = ap.H; pp.W = ap.W; pp.K = ap.K; pp.S = ap.S; pp.T = 2 * ap.S + 32;
            pp.G = ap.G; pp.cellW = ap.cellW; pp.cellH = ap.cellH; pp.ncell = ap.ncell;
            pp.first = 0; pp.finalize = 1; pp.last = 0; pp.noq = 0;
            pp.preempt = 0; pp.l1_thres = 0.f; pp.nactive = nullptr;
            for (int bi = 0; bi < ap.B; bi++)
                prepare_in_tail(pp, clusters + (size_t)bi * ap.K, acc + (size_t)bi * ap.K * 4, cinfo_next + (size_t)bi * ap.K,
                                cell_start_next + (size_t)bi * (ap.ncell + 1), smem_raw, (int)threadIdx.x, (int)blockDim.x);
        }
    }
}
