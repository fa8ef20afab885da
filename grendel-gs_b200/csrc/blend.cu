// Per-tile alpha blending: CUDA stages "70 render" (+81-83 statistics) and "b10 render"
// (/root/reference/analyze_statistic.py:1981-1987) -- the second half of
// GaussianRasterizer.render_gaussians and its autograd backward
// (/root/reference/gaussian_renderer/__init__.py:1271-1282, train_internal.py:195).
//
// One CTA = one 16x16 tile (BLOCK_X/Y are observable through _C.get_block_XY and baked into the
// reference's strip arithmetic, loss_distribution.py:2321-2330).  Both kernels are bound by instruction
// issue over (pixel, splat) pairs, not by HBM (ncu: issue slots ~85 % busy, DRAM ~2 %; algorithmic
// traffic is only 40 B / 76 B per instance, SURVEY.md 8d), so the design minimises issued instructions
// per USEFUL pair:
//   * the tile is cut into sixteen 4x4 pixel blocks; every HALF-warp owns one block and walks its own
//     candidate list, so one warp instruction advances two (block, splat) pairs and ~60 % of the lanes do
//     useful work in the blend path (an 8x4 block per full warp reached 37 %);
//   * candidates come from a 16-bit "which 4x4 blocks can this splat reach" mask computed at staging time
//     from the bounding box of the splat's {alpha >= 1/255} ellipse (conservative: per-pixel results are
//     unchanged); a warp ballots 32 masks at a time;
//   * the alpha < 1/255 test is done on the exponent (power < ln(1/(255 o)) - margin) so rejected pairs never
//     reach MUFU.EX2; finished / out-of-image pixels carry NaN coordinates so they fail it for free;
//   * sorted splat ids are turned into 48-byte packed records (3 x float4, built by k_count_tiles), gathered
//     once per (splat, tile) into shared memory;
//   * backward (one 8x4 block per full warp, see the note above k_blend_bwd): per-pixel weight m = dL/dG * G; its
//     six moments (sum m, m dx, m dy, m dx^2, m dx dy, m dy^2) and three colour sums are reduced over the warp by a
//     9-value transposing butterfly (14 shuffles instead of 45), stored in per-warp private shared-memory slots
//     (no shared atomics: sm_100 has no native fp32 ATOMS.ADD -- it compiles to a CAS loop), then ONE thread per
//     splat sums the warps, applies the splat's constants and issues ONE set of 9 global RED.ADD per
//     (splat, tile) -- instead of 9 atomics per (splat, pixel) in the classical design.  The per-pixel state is
//     just (T, behind-colour B): lanes that skip a splat run the same instructions with alpha = 0, which makes
//     every update a no-op, so the blend path has no per-lane branches or conditional moves.
//
// Round 2: SEGMENT-PARALLEL backward (k_blend_bwd_seg; round 3's default k_blend_bwd_seg3 walks the same way).  The
// forward stores, for every pixel of a tile, a
// checkpoint (T, colour summed over the LATER segments) every SEG_K entries of the tile list, so every (tile, SEG_K-entry
// segment) can be walked back to front on its own.  One WARP owns one such unit and ALL 256 pixels of the tile: lane l
// holds pixel l of each of the eight 8x4 blocks (state T and S = sum of the colour behind, weighted with dL/dpixel, in
// registers), loops over the blocks the splat can reach, accumulates the nine gradient sums in registers ACROSS the
// blocks, reduces them ONCE per (splat, tile) with the 9-value butterfly and issues one RED set straight away: no CTA
// barrier, no shared partial sums, no flush pass, 1 instead of ~1.9 reductions per (splat, tile).
#include "common.cuh"

#define BL_THREADS 256
#define BL_WARPS (BL_THREADS / 32)
#define BL_BLOCKS 16  // 4x4 pixel blocks per tile
#ifndef FW_CHUNK
#define FW_CHUNK 256
#endif

#define ALPHA_MIN (1.0f / 255.0f)
#define ALPHA_MAX 0.99f
#define T_EPS 0.0001f
#define FULL 0xffffffffu

// exp(x) for x <= 0 as one FMUL + MUFU.EX2 (results below 2^-126 flush to 0: far under the 1/255 alpha floor)
GS_D float gs_exp_neg(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
    return y;
}

// thread -> (4x4 block, pixel).  Warp w holds blocks 2w and 2w+1 (horizontal neighbours), one per half-warp.
struct Where { int blk, px, py, half, l16; };
GS_D Where where_am_i(int tile, int gx) {
    Where p;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    p.half = lane >> 4;
    p.l16 = lane & 15;
    const int by = w >> 1, bx = (w & 1) * 2 + p.half;
    p.blk = by * 4 + bx;
    p.px = (tile % gx) * GS_BLOCK_X + bx * 4 + (p.l16 & 3);
    p.py = (tile / gx) * GS_BLOCK_Y + by * 4 + (p.l16 >> 2);
    return p;
}

// Row-band extents of the splat's {power >= thr} ellipse.  The bounding box alone keeps every block of the box's
// corners, which a diagonal or elongated ellipse never reaches: on c2 a third of the (4x4 block, splat) candidates of the
// forward and a quarter of the backward's (8x4 block, splat) passes ended in the "no pixel passes the exponent test"
// exit.  For the four bands of four pixel rows of the tile, [xl, xh] is the exact x-range (tile coordinates) that
//   alpha' u^2 + beta' u v + gamma' v^2 <= tau     (u, v relative to the centre; alpha' = -a', beta' = -b', gamma' = -c', tau = -thr)
// covers over v in the band: the right boundary r(v) = kappa v + sqrt(tau/alpha') sqrt(1 - v^2/ey0^2), kappa = -beta'/(2 alpha'), is
// concave with its maximum at v_r = -beta' ex0 / (2 gamma') (the ellipse's rightmost point), so its maximum over the band is
// r(clamp(v_r, band)); the left boundary is the point mirror image.  ex0 / ey0 are the box's half extents as k_count_tiles
// computed them (compensated determinant), so needle-shaped conics do not cancel here either.  Widened by 2 % + 0.05 px
// in both directions (thr itself carries the 0.02 exponent margin): conservative, per-pixel results are unchanged
// (test_needle_splats_survive_block_culling, culled == unculled bit for bit).  Degenerate conics (ex = 3e38) and
// GS_DEBUG_NO_BLOCK_CULL keep every band of the box.
#define GS_BAND_ABS_MARGIN 0.05f
// approximate MUFU forms (relative error ~1e-7, three orders of magnitude inside the margins; the IEEE forms cost a
// fix-up branch each, eight times per staged splat)
GS_D float gs_rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
GS_D float gs_sqrt_approx(float x) { float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
GS_D void ellipse_bands(const float4 a, const float4 b, const float ex, const float ey, const float X0, const float Y0,
                        float (&xl)[4], float (&xh)[4]) {
    if (ex < 0.f) {
#pragma unroll
        for (int q = 0; q < 4; q++) { xl[q] = 1e30f; xh[q] = -1e30f; }
        return;
    }
    const bool exact = ex < 1e30f;
    const float ex0 = (ex - 0.5f) * (1.f / 1.02f), ey0 = (ey - 0.5f) * (1.f / 1.02f);
    const float mgx = 0.02f * ex0 + GS_BAND_ABS_MARGIN, mgy = 0.02f * ey0 + GS_BAND_ABS_MARGIN;
    const float inv_a = gs_rcp_approx(-a.z);         // 1 / alpha'
    const float kappa = 0.5f * a.w * inv_a;       // -beta' / (2 alpha')   (beta' = -a.w, alpha' = -a.z)
    const float hw2 = -b.z * inv_a;               // tau / alpha'
    const float v_r = -0.5f * a.w * ex0 * gs_rcp_approx(b.x);  // -beta' ex0 / (2 gamma') = -(-a.w) ex0 / (2 (-b.x))
    const float inv_ey0 = gs_rcp_approx(ey0);
    const float cx = a.x - X0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const float v0 = (Y0 + 4.f * q) - a.y, v1 = v0 + 3.f;
        float l = 1e30f, h = -1e30f;
        if (v1 >= -ey && v0 <= ey) {
            l = -1e30f; h = 1e30f;
            if (exact) {
                const float lo = v0 - mgy, hi = v1 + mgy;
                const float vh = fminf(fmaxf(v_r, lo), hi), vl = fminf(fmaxf(-v_r, lo), hi);
                const float qh = vh * inv_ey0, ql = vl * inv_ey0;
                const float sh = fmaxf(0.f, 1.f - qh * qh), sl = fmaxf(0.f, 1.f - ql * ql);
                h = cx + (kappa * vh + gs_sqrt_approx(hw2 * sh) + mgx);
                l = cx + (kappa * vl - gs_sqrt_approx(hw2 * sl) - mgx);
            }
        }
        xl[q] = l; xh[q] = h;
    }
}

// bit (by*4+bx) set <=> the splat's ellipse can reach 4x4 block (bx,by)
GS_D uint32_t block_mask16(const float4 a, const float4 b, float ex, float ey, float X0, float Y0) {
    float xl[4], xh[4];
    ellipse_bands(a, b, ex, ey, X0, Y0, xl, xh);
    uint32_t m = 0u;
#pragma unroll
    for (int q = 0; q < 4; q++) {
#pragma unroll
        for (int bx = 0; bx < 4; bx++)
            if (xh[q] >= 4.f * bx && xl[q] <= 4.f * bx + 3.f) m |= 1u << (4 * q + bx);
    }
    return m;
}

// staged splat: one 48-byte slot so a single address feeds all three shared-memory loads
struct __align__(16) SRec { float4 a; float4 b; float4 c; };

// ---- segment workspace shared by the forward (writer) and the segment-parallel backward (reader) -------------------
// SEG_K entries per segment.  Checkpoint slot of (tile t, boundary after segment s) = ranges[t].x / SEG_K + t + s:
// injective over all tiles without a scan (floor((x+l)/K) - floor(x/K) >= ceil(l/K) - 1), < R / SEG_K + T + 1.
// A slot holds one float4 per pixel, in the BACKWARD's order: index = (8x4 block) * 32 + lane.
#ifndef SEG_K
#define SEG_K 128
#endif
#define SEG_SLOT 256
struct SegWs {
    uint32_t *n_units;    // [1] number of (tile, segment) units appended by the forward
    uint32_t *tile_last;  // [T] deepest contributing entry of the tile (max n_contrib over its pixels)
    uint2 *units;         // [R / SEG_K + T] (tile, segment)
    float4 *ckpt;         // [(R / SEG_K + T + 1) * SEG_SLOT]
    uint16_t *cull;       // [R] the forward's 4x4-block mask of every entry it staged (the backward never walks further)
};
static size_t seg_align(size_t v) { return (v + 255) / 256 * 256; }
static size_t seg_bytes(int64_t R, int64_t T) {
    const size_t slots = (size_t)(R / SEG_K + T + 1);
    return 256 + seg_align((size_t)T * 4) + seg_align(slots * sizeof(uint2)) + slots * SEG_SLOT * sizeof(float4) +
           seg_align((size_t)R * sizeof(uint16_t));
}
static SegWs seg_carve(void *ws, int64_t R, int64_t T) {
    const size_t slots = (size_t)(R / SEG_K + T + 1);
    char *p = (char *)ws;
    SegWs w;
    w.n_units = (uint32_t *)p; p += 256;
    w.tile_last = (uint32_t *)p; p += seg_align((size_t)T * 4);
    w.units = (uint2 *)p; p += seg_align(slots * sizeof(uint2));
    w.ckpt = (float4 *)p; p += slots * SEG_SLOT * sizeof(float4);
    w.cull = (uint16_t *)p;
    return w;
}
extern "C" size_t gs_render_seg_bytes(int64_t R, int num_tiles) { return seg_bytes(R > 0 ? R : 0, num_tiles > 0 ? num_tiles : 0); }

#ifndef FW_MIN_CTAS
#define FW_MIN_CTAS 6
#endif
template <bool STATS, bool CKPT>
__global__ void __launch_bounds__(BL_THREADS, FW_MIN_CTAS)
k_blend_fwd(int W, int H, int tiles_per_view, const float4 *__restrict__ rec, const float *__restrict__ bg,
            const uint8_t *__restrict__ compute_locally, const uint2 *__restrict__ ranges,
            const uint32_t *__restrict__ ids, float *__restrict__ image, float *__restrict__ final_T,
            uint32_t *__restrict__ n_contrib, unsigned long long *__restrict__ stats, const SegWs seg) {
    __shared__ SRec s_rec[FW_CHUNK];
    __shared__ uint16_t s_cull[FW_CHUNK];
    __shared__ unsigned long long s_stats[3];
    __shared__ uint32_t s_red[BL_WARPS + 2];
    const int gx = (W + GS_BLOCK_X - 1) / GS_BLOCK_X;
    // blockIdx.x = view * tiles_per_view + tile: the views' tile arrays and images are concatenated (GsViews)
    const int view = blockIdx.x / tiles_per_view, tile = blockIdx.x - view * tiles_per_view;
    const int lane = threadIdx.x & 31;
    const Where me = where_am_i(tile, gx);
    const int px = me.px, py = me.py;
    const bool inside = px < W && py < H;
    const size_t HW = (size_t)H * W;
    const size_t pix = (size_t)py * W + px;
    image += (size_t)view * 3 * HW;
    final_T += (size_t)view * HW;
    n_contrib += (size_t)view * HW;
    if (!compute_locally[blockIdx.x]) {  // non-local tiles must read exactly 0 (loss_distribution.py:1875)
        if (inside) { image[pix] = 0.f; image[HW + pix] = 0.f; image[2 * HW + pix] = 0.f; }
        if (CKPT && threadIdx.x == 0) seg.tile_last[blockIdx.x] = 0u;
        return;
    }
    const uint2 range = ranges[blockIdx.x];
    const int total = (int)(range.y - range.x);
    const float X0 = (float)((tile % gx) * GS_BLOCK_X), Y0 = (float)((tile / gx) * GS_BLOCK_Y);
    const float qnan = __int_as_float(0x7fc00000);
    float pxf = inside ? (float)px : qnan, pyf = (float)py;  // NaN coordinates: the pixel never passes a test
    // colour is accumulated per SEG_K-entry segment (C) and folded front to back into Ctot at every segment boundary --
    // the same arithmetic with and without checkpoints, so both forward variants produce identical images
    float T = 1.f, C0 = 0.f, C1 = 0.f, C2 = 0.f, Ct0 = 0.f, Ct1 = 0.f, Ct2 = 0.f;
    uint32_t last = 0, blended = 0, considered = 0;
    bool done = !inside;
    const int blkA = me.blk - me.half;  // block of lanes 0-15; lanes 16-31 own blkA + 1
    // this pixel's entry in a checkpoint slot: (8x4 block = warp) * 32 + (row in block) * 8 + (column in block)
    float4 *ck = nullptr;
    int nck = 0;
    if (CKPT)
        ck = seg.ckpt + ((size_t)(range.x / SEG_K) + blockIdx.x) * SEG_SLOT + (threadIdx.x >> 5) * 32 + (me.l16 >> 2) * 8 +
             me.half * 4 + (me.l16 & 3);
    for (int base = 0; base < total; base += FW_CHUNK) {
        if (__syncthreads_count(done) == BL_THREADS) break;
        const int cnt = min(FW_CHUNK, total - base);
        for (int i = threadIdx.x; i < cnt; i += BL_THREADS) {
            const uint32_t g = ids[range.x + base + i];
            const float4 *r = rec + (size_t)3 * g;
            const float4 a = __ldg(r), b = __ldg(r + 1), c = __ldg(r + 2);
            s_rec[i].a = a; s_rec[i].b = b; s_rec[i].c = c;
            const uint16_t m16 = (uint16_t)block_mask16(a, b, c.z, c.w, X0, Y0);
            s_cull[i] = m16;
            if (CKPT) seg.cull[range.x + base + i] = m16;
        }
        __syncthreads();
        for (int g0 = 0; g0 < cnt; g0 += 32) {
            if (__all_sync(FULL, done)) break;  // checked once per 32 entries; finished pixels are NaN anyway
            {   // segment boundary: a pixel that is still alive here has its warp here, so its checkpoint gets written
                const int e0 = base + g0;
                if (e0 > 0 && (e0 & (SEG_K - 1)) == 0) {
                    if (CKPT) { ck[(size_t)nck * SEG_SLOT] = make_float4(T, C0, C1, C2); nck++; }
                    Ct0 += C0; Ct1 += C1; Ct2 += C2;
                    C0 = C1 = C2 = 0.f;
                }
            }
            const int jj = g0 + lane;
            const uint32_t m = jj < cnt ? (uint32_t)s_cull[jj] : 0u;
            const uint32_t cA = __ballot_sync(FULL, (m >> blkA) & 1u), cB = __ballot_sync(FULL, (m >> (blkA + 1)) & 1u);
            uint32_t mine = me.half ? cB : cA;  // this half-warp's candidates among the 32 entries
            while (__any_sync(FULL, mine != 0u)) {
                const bool has = mine != 0u;
                const int j = g0 + (has ? __ffs(mine) - 1 : 0);
                mine &= mine - 1u;
                const SRec *sr = &s_rec[j];
                const float4 a = sr->a, b = sr->b;
                const float dx = a.x - pxf, dy = a.y - pyf;
                const float power = dx * (a.z * dx + a.w * dy) + b.x * dy * dy;
                const bool ok = has && power >= b.z;  // false for NaN (finished / outside pixels)
                if (!__any_sync(FULL, ok)) continue;
                if (ok && power <= 0.f) {   // thr <= power <= 0  <=>  alpha >= 1/255 (thr = ln(1/(255 opacity)), no margin)
                    const float alpha = fminf(ALPHA_MAX, b.y * gs_exp_neg(power));
                    {
                        const float test_T = T * (1.f - alpha);
                        if (test_T < T_EPS) {
                            done = true;
                            pxf = qnan;
                            if (STATS) considered = (uint32_t)(base + j + 1);
                        } else {
                            const float2 gb = *reinterpret_cast<const float2 *>(&sr->c);
                            const float w = alpha * T;
                            C0 += b.w * w; C1 += gb.x * w; C2 += gb.y * w;
                            T = test_T;
                            last = (uint32_t)(base + j + 1);
                            if (STATS) blended++;
                        }
                    }
                }
            }
        }
    }
    if (inside) {
        image[pix] = (Ct0 + C0) + T * bg[0];
        image[HW + pix] = (Ct1 + C1) + T * bg[1];
        image[2 * HW + pix] = (Ct2 + C2) + T * bg[2];
        final_T[pix] = T;
        n_contrib[pix] = last;
        if (considered == 0) considered = (uint32_t)total;
    }
    if (CKPT) {
        // checkpoint s so far = (T, colour of segment s); the backward wants (T, colour of all LATER segments): suffix sums,
        // added back to front (small terms first, no cancellation)
        float r0 = C0, r1 = C1, r2 = C2;
        for (int s = nck - 1; s >= 0; s--) {
            const float4 c = ck[(size_t)s * SEG_SLOT];
            ck[(size_t)s * SEG_SLOT] = make_float4(c.x, r0, r1, r2);
            r0 += c.y; r1 += c.z; r2 += c.w;
        }
        // the tile's units for the backward: segments [0, ceil(deepest contributor / SEG_K))
        uint32_t m = inside ? last : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(FULL, m, o));
        if (lane == 0) s_red[threadIdx.x >> 5] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tl = 0;
#pragma unroll
            for (int w = 0; w < BL_WARPS; w++) tl = max(tl, s_red[w]);
            const uint32_t nseg = (tl + SEG_K - 1) / SEG_K;
            seg.tile_last[blockIdx.x] = tl;
            s_red[BL_WARPS] = nseg;
            s_red[BL_WARPS + 1] = nseg ? atomicAdd(seg.n_units, nseg) : 0u;
        }
        __syncthreads();
        const uint32_t nseg = s_red[BL_WARPS], ubase = s_red[BL_WARPS + 1];
        for (uint32_t i = threadIdx.x; i < nseg; i += BL_THREADS) seg.units[ubase + i] = make_uint2(blockIdx.x, nseg - 1 - i);
    }
    if (STATS) {  // stages 81-83: sums of tile-list length / entries walked / entries blended
        if (threadIdx.x < 3) s_stats[threadIdx.x] = 0ull;
        __syncthreads();
        unsigned long long v0 = inside ? (unsigned long long)total : 0ull, v1 = inside ? considered : 0u,
                           v2 = inside ? blended : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            v0 += __shfl_xor_sync(FULL, v0, o);
            v1 += __shfl_xor_sync(FULL, v1, o);
            v2 += __shfl_xor_sync(FULL, v2, o);
        }
        if (lane == 0) { atomicAdd(&s_stats[0], v0); atomicAdd(&s_stats[1], v1); atomicAdd(&s_stats[2], v2); }
        __syncthreads();
        if (threadIdx.x < 3) atomicAdd(&stats[3 * view + threadIdx.x], s_stats[threadIdx.x]);
    }
}

// ---- forward, packed variant: TWO pixels per lane, four 4x4 blocks per warp --------------------------------------------
// One CTA of 4 warps per tile.  Warp w owns the 16x4 pixel strip of rows 4w..4w+3, i.e. four 4x4 blocks; each QUARTER
// warp (8 lanes) owns one block and walks its own candidate list, each lane blending two horizontally adjacent pixels
// with packed fp32 arithmetic (fma.rn.f32x2 & co: one issue slot for both pixels).  One warp instruction therefore
// advances four (block, splat) pairs instead of two; the per-pixel arithmetic is the same operation sequence as
// k_blend_fwd (bit-identical images).
#define F2_THREADS 128
#define F2_WARPS 4
#ifndef F2_MIN_CTAS
#define F2_MIN_CTAS 8
#endif
// Two fp32 values in one 64-bit register, operated on by the packed instructions of sm_100 (FFMA2 / FMUL2 / FADD2).  Kept
// as opaque 64-bit values so that loop-carried state STAYS packed (float2 variables get scalarised and re-packed with
// register moves around every packed instruction).
typedef unsigned long long p2;
GS_D p2 p2_make(float lo, float hi) { p2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
GS_D p2 p2_bc(float v) { return p2_make(v, v); }
GS_D float p2_lo(p2 v) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); return lo; }
GS_D float p2_hi(p2 v) { float lo, hi; asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); return hi; }
GS_D p2 p2_fma(p2 a, p2 b, p2 c) { p2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
GS_D p2 p2_mul(p2 a, p2 b) { p2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
GS_D p2 p2_add(p2 a, p2 b) { p2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
// in-place forms for loop-carried accumulators: the tied operand keeps the value in ONE register pair across iterations
// (separate result registers made ptxas copy every packed state variable back at the end of each iteration)
GS_D void p2_fma_acc(p2 &c, p2 a, p2 b) { asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c) : "l"(a), "l"(b)); }
GS_D void p2_mul_acc(p2 &t, p2 f) { asm("mul.rn.f32x2 %0, %0, %1;" : "+l"(t) : "l"(f)); }
GS_D void p2_add_acc(p2 &c, p2 a) { asm("add.rn.f32x2 %0, %0, %1;" : "+l"(c) : "l"(a)); }

template <bool STATS, bool CKPT>
__global__ void __launch_bounds__(F2_THREADS, F2_MIN_CTAS)
k_blend_fwd2(int W, int H, int tiles_per_view, const float4 *__restrict__ rec, const float *__restrict__ bg,
             const uint8_t *__restrict__ compute_locally, const uint2 *__restrict__ ranges,
             const uint32_t *__restrict__ ids, float *__restrict__ image, float *__restrict__ final_T,
             uint32_t *__restrict__ n_contrib, unsigned long long *__restrict__ stats, const SegWs seg) {
    __shared__ SRec s_rec[FW_CHUNK + 1];   // + the slot an empty candidate list points at (entry g0 + 32 of the last group)
    __shared__ uint16_t s_cull[FW_CHUNK];
    __shared__ unsigned long long s_stats[3];
    __shared__ uint32_t s_red[F2_WARPS + 2];
    const int gx = (W + GS_BLOCK_X - 1) / GS_BLOCK_X;
    const int view = blockIdx.x / tiles_per_view, tile = blockIdx.x - view * tiles_per_view;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int quarter = lane >> 3, l8 = lane & 7;
    const int lx = quarter * 4 + (l8 & 1) * 2, ly = warp * 4 + (l8 >> 1);  // first pixel of the pair, inside the tile
    const int px = (tile % gx) * GS_BLOCK_X + lx, py = (tile / gx) * GS_BLOCK_Y + ly;
    const bool in0 = px < W && py < H, in1 = px + 1 < W && py < H;
    const size_t HW = (size_t)H * W;
    const size_t pix = (size_t)py * W + px;
    image += (size_t)view * 3 * HW;
    final_T += (size_t)view * HW;
    n_contrib += (size_t)view * HW;
    if (!compute_locally[blockIdx.x]) {  // non-local tiles must read exactly 0 (loss_distribution.py:1875)
        if (in0) { image[pix] = 0.f; image[HW + pix] = 0.f; image[2 * HW + pix] = 0.f; }
        if (in1) { image[pix + 1] = 0.f; image[HW + pix + 1] = 0.f; image[2 * HW + pix + 1] = 0.f; }
        if (CKPT && threadIdx.x == 0) seg.tile_last[blockIdx.x] = 0u;
        return;
    }
    const uint2 range = ranges[blockIdx.x];
    const int total = (int)(range.y - range.x);
    const float X0 = (float)((tile % gx) * GS_BLOCK_X), Y0 = (float)((tile / gx) * GS_BLOCK_Y);
    const float qnan = __int_as_float(0x7fc00000);
    // minus the pixel coordinates; NaN = finished / outside pixel, which then never passes a test
    float npx0 = in0 ? -(float)px : qnan, npx1 = in1 ? -(float)(px + 1) : qnan;
    const float pyf = (float)py;
    const p2 zero2 = p2_bc(0.f), one2 = p2_bc(1.f), mone2 = p2_bc(-1.f);
    p2 T = one2, C0 = zero2, C1 = zero2, C2 = zero2, Ct0 = zero2, Ct1 = zero2, Ct2 = zero2;
    uint32_t last0 = 0, last1 = 0, blended = 0, cons0 = 0, cons1 = 0;
    // a finished / outside pixel is one whose coordinate is NaN: no separate flags to maintain in the loop
#define F2_DONE (npx0 != npx0 && npx1 != npx1)
    // this pixel pair's entries in a checkpoint slot: (8x4 block) * 32 + (row in block) * 8 + (column in block)
    float4 *ck = nullptr;
    int nck = 0;
    if (CKPT)
        ck = seg.ckpt + ((size_t)(range.x / SEG_K) + blockIdx.x) * SEG_SLOT + (warp * 2 + (lx >> 3)) * 32 + (ly & 3) * 8 + (lx & 7);
    // a quarter warp without a candidate runs the iteration on entry g0 + clz(0) = g0 + 32 with an effective alpha of 0: whatever
    // record sits there must be finite (0 * inf would poison the colour sums), so slots the staging never wrote start as 0
    // (each thread clears exactly the slots it stages later: program order, no barrier)
    for (int i = threadIdx.x; i < FW_CHUNK + 1; i += F2_THREADS) {
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        s_rec[i].a = z; s_rec[i].b = z; s_rec[i].c = z;
    }
    for (int base = 0; base < total; base += FW_CHUNK) {
        if (__syncthreads_count(F2_DONE) == F2_THREADS) break;
        const int cnt = min(FW_CHUNK, total - base);
        for (int i = threadIdx.x; i < cnt; i += F2_THREADS) {
            const uint32_t g = ids[range.x + base + i];
            const float4 *r = rec + (size_t)3 * g;
            const float4 a = __ldg(r), b = __ldg(r + 1), c = __ldg(r + 2);
            // staged in the POSITIVE form q = -power = alpha' dx^2 + beta' dx dy + gamma' dy^2 with t = -thr >= 0: the pixel test
            // thr <= power <= 0 becomes 0 <= q <= t, ONE unsigned compare of the bit patterns (negative, NaN and inf
            // patterns are all above t's; q is never -0 because the non-negative gamma' dy^2 is added last)
            s_rec[i].a = make_float4(a.x, a.y, -a.z, -a.w);
            s_rec[i].b = make_float4(-b.x, b.y, fmaxf(-b.z, 0.f), b.w);
            s_rec[i].c = c;
            const uint16_t m16 = (uint16_t)block_mask16(a, b, c.z, c.w, X0, Y0);
            s_cull[i] = m16;
            if (CKPT) seg.cull[range.x + base + i] = m16;
        }
        __syncthreads();
        for (int g0 = 0; g0 < cnt; g0 += 32) {
            if (__all_sync(FULL, F2_DONE)) break;
            {   // segment boundary (see k_blend_fwd)
                const int e0 = base + g0;
                if (e0 > 0 && (e0 & (SEG_K - 1)) == 0) {
                    if (CKPT) {
                        ck[(size_t)nck * SEG_SLOT] = make_float4(p2_lo(T), p2_lo(C0), p2_lo(C1), p2_lo(C2));
                        ck[(size_t)nck * SEG_SLOT + 1] = make_float4(p2_hi(T), p2_hi(C0), p2_hi(C1), p2_hi(C2));
                        nck++;
                    }
                    Ct0 = p2_add(Ct0, C0); Ct1 = p2_add(Ct1, C1); Ct2 = p2_add(Ct2, C2);
                    C0 = C1 = C2 = zero2;
                }
            }
            // lane l inspects entry g0 + 31 - l: the HIGHEST set bit of a ballot is the EARLIEST candidate
            const int jj = g0 + 31 - lane;
            const uint32_t m = jj < cnt ? ((uint32_t)s_cull[jj] >> (warp * 4)) : 0u;
            const uint32_t c0 = __ballot_sync(FULL, m & 1u), c1 = __ballot_sync(FULL, m & 2u),
                           c2 = __ballot_sync(FULL, m & 4u), c3 = __ballot_sync(FULL, m & 8u);
            uint32_t mine = quarter == 0 ? c0 : quarter == 1 ? c1 : quarter == 2 ? c2 : c3;
            const p2 npx = p2_make(npx0, npx1);
            p2 npx_cur = npx;
            while (__any_sync(FULL, mine != 0u)) {
                const bool has = mine != 0u;
                const int lz = __clz((int)mine);       // 32 when empty: a finite slot (see the clearing loop above)
                const int j = g0 + lz;
                mine &= ~__funnelshift_rc(0x80000000u, 0u, lz);   // (0x80000000 >> lz), 0 for lz = 32 (clamped shift)
                const SRec *sr = &s_rec[j];
                const float4 a = sr->a, b = sr->b;
                const float dy = a.y - pyf;
                const p2 dx = p2_add(p2_bc(a.x), npx_cur);
                const float t = a.w * dy, u = b.x * dy * dy;
                const p2 pw = p2_fma(dx, p2_fma(p2_bc(a.z), dx, p2_bc(t)), p2_bc(u));   // q = -power (>= 0, or NaN)
                const uint32_t tb = __float_as_uint(b.z);
                const bool ok0 = has && __float_as_uint(p2_lo(pw)) <= tb, ok1 = has && __float_as_uint(p2_hi(pw)) <= tb;
#ifdef F2_EARLY_OUT   // with the row-band culling few iterations have no passing lane: the vote costs more than it skips
                if (!__any_sync(FULL, ok0 || ok1)) continue;   // (0.591 -> 0.581 ms on c2 without it)
#endif
                const p2 e = p2_mul(pw, p2_bc(-1.4426950408889634f));
                float G0, G1;
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(G0) : "f"(p2_lo(e)));
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(G1) : "f"(p2_hi(e)));
                const p2 araw = p2_mul(p2_bc(b.y), p2_make(G0, G1));
                const float al0 = fminf(ALPHA_MAX, p2_lo(araw)), al1 = fminf(ALPHA_MAX, p2_hi(araw));
                const bool v0 = ok0, v1 = ok1;   // 0 <= q <= t  <=>  alpha >= 1/255: no second test on alpha
                const p2 test_T = p2_mul(T, p2_fma(p2_make(al0, al1), mone2, one2));
                const bool end0 = v0 && p2_lo(test_T) < T_EPS, end1 = v1 && p2_hi(test_T) < T_EPS;
                const bool bl0 = v0 && !end0, bl1 = v1 && !end1;
                if (end0) { npx0 = qnan; if (STATS) cons0 = (uint32_t)(base + j + 1); }
                if (end1) { npx1 = qnan; if (STATS) cons1 = (uint32_t)(base + j + 1); }
                npx_cur = p2_make(npx0, npx1);
                // effective alpha: 0 for a pixel that does not blend this splat -- every update below is then a no-op, so
                // the packed state needs no per-component selects (T (1 - ae) is the same product as test_T when blending)
                const p2 ae = p2_make(bl0 ? al0 : 0.f, bl1 ? al1 : 0.f);
                const p2 w = p2_mul(ae, T);
                const float2 gb = *reinterpret_cast<const float2 *>(&sr->c);
                p2_fma_acc(C0, p2_bc(b.w), w); p2_fma_acc(C1, p2_bc(gb.x), w); p2_fma_acc(C2, p2_bc(gb.y), w);
                p2_mul_acc(T, p2_fma(ae, mone2, one2));
                last0 = bl0 ? (uint32_t)(base + j + 1) : last0; last1 = bl1 ? (uint32_t)(base + j + 1) : last1;
                if (STATS) blended += (bl0 ? 1u : 0u) + (bl1 ? 1u : 0u);
            }
        }
    }
    const float b0 = bg[0], b1 = bg[1], b2 = bg[2];
    const float T0 = p2_lo(T), T1 = p2_hi(T);
    if (in0) {
        image[pix] = (p2_lo(Ct0) + p2_lo(C0)) + T0 * b0; image[HW + pix] = (p2_lo(Ct1) + p2_lo(C1)) + T0 * b1;
        image[2 * HW + pix] = (p2_lo(Ct2) + p2_lo(C2)) + T0 * b2;
        final_T[pix] = T0; n_contrib[pix] = last0;
        if (cons0 == 0) cons0 = (uint32_t)total;
    }
    if (in1) {
        image[pix + 1] = (p2_hi(Ct0) + p2_hi(C0)) + T1 * b0; image[HW + pix + 1] = (p2_hi(Ct1) + p2_hi(C1)) + T1 * b1;
        image[2 * HW + pix + 1] = (p2_hi(Ct2) + p2_hi(C2)) + T1 * b2;
        final_T[pix + 1] = T1; n_contrib[pix + 1] = last1;
        if (cons1 == 0) cons1 = (uint32_t)total;
    }
    if (CKPT) {
        float r0x = p2_lo(C0), r1x = p2_lo(C1), r2x = p2_lo(C2), r0y = p2_hi(C0), r1y = p2_hi(C1), r2y = p2_hi(C2);
        for (int s = nck - 1; s >= 0; s--) {
            const float4 ca = ck[(size_t)s * SEG_SLOT], cb = ck[(size_t)s * SEG_SLOT + 1];
            ck[(size_t)s * SEG_SLOT] = make_float4(ca.x, r0x, r1x, r2x);
            ck[(size_t)s * SEG_SLOT + 1] = make_float4(cb.x, r0y, r1y, r2y);
            r0x += ca.y; r1x += ca.z; r2x += ca.w;
            r0y += cb.y; r1y += cb.z; r2y += cb.w;
        }
        uint32_t m = max(in0 ? last0 : 0u, in1 ? last1 : 0u);
        m = __reduce_max_sync(FULL, m);
        if (lane == 0) s_red[warp] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tl = 0;
#pragma unroll
            for (int w = 0; w < F2_WARPS; w++) tl = max(tl, s_red[w]);
            const uint32_t nseg = (tl + SEG_K - 1) / SEG_K;
            seg.tile_last[blockIdx.x] = tl;
            s_red[F2_WARPS] = nseg;
            s_red[F2_WARPS + 1] = nseg ? atomicAdd(seg.n_units, nseg) : 0u;
        }
        __syncthreads();
        const uint32_t nseg = s_red[F2_WARPS], ubase = s_red[F2_WARPS + 1];
        for (uint32_t i = threadIdx.x; i < nseg; i += F2_THREADS) seg.units[ubase + i] = make_uint2(blockIdx.x, nseg - 1 - i);
    }
    if (STATS) {  // stages 81-83: sums of tile-list length / entries walked / entries blended
        if (threadIdx.x < 3) s_stats[threadIdx.x] = 0ull;
        __syncthreads();
        unsigned long long v0 = (in0 ? (unsigned long long)total : 0ull) + (in1 ? (unsigned long long)total : 0ull),
                           v1 = (in0 ? cons0 : 0u) + (unsigned long long)(in1 ? cons1 : 0u), v2 = blended;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            v0 += __shfl_xor_sync(FULL, v0, o);
            v1 += __shfl_xor_sync(FULL, v1, o);
            v2 += __shfl_xor_sync(FULL, v2, o);
        }
        if (lane == 0) { atomicAdd(&s_stats[0], v0); atomicAdd(&s_stats[1], v1); atomicAdd(&s_stats[2], v2); }
        __syncthreads();
        if (threadIdx.x < 3) atomicAdd(&stats[3 * view + threadIdx.x], s_stats[threadIdx.x]);
    }
}

// ---- backward, tile-parallel (round 1; kept behind gs_debug_set(GS_DEBUG_BWD_TILE) and for callers without a segment
// workspace) ----------------------------------------------------------------------------------------------------------
// The backward keeps one 8x4 pixel block per FULL warp (8-bit cull mask, 128-entry chunks): the half-warp /
// 4x4 layout that helps the forward was measured slower here (2.18 vs 1.77 ms on c2) -- sixteen private
// partial-sum slots force 64-entry chunks, and the extra barriers + 64-thread flush cost more (barrier stalls
// 3.1 warps per issue) than the better lane utilisation returns.
#define BW8_CHUNK 128
#define BW8_STRIDE (BW8_CHUNK + 1)

GS_D void pixel_of_thread(int tile, int gx, int &px, int &py) {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    px = (tile % gx) * GS_BLOCK_X + (w & 1) * 8 + (lane & 7);
    py = (tile / gx) * GS_BLOCK_Y + (w >> 1) * 4 + (lane >> 3);
}

// bit w set <=> the splat's ellipse can reach warp w's 8x4 pixel block (w = 2 * band + column half)
GS_D uint32_t block_mask(const float4 a, const float4 b, float ex, float ey, float X0, float Y0) {
    float xl[4], xh[4];
    ellipse_bands(a, b, ex, ey, X0, Y0, xl, xh);
    uint32_t m = 0u;
#pragma unroll
    for (int wy = 0; wy < 4; wy++) {
        if (xh[wy] >= 0.f && xl[wy] <= 7.f) m |= 1u << (2 * wy);
        if (xh[wy] >= 8.f && xl[wy] <= 15.f) m |= 2u << (2 * wy);
    }
    return m;
}

// 9-value warp reduction.  After the call every lane holds in v[0] the warp total of value
// (lane >> 2) & 7, and in v[8] the warp total of value 8.
GS_D void warp_reduce9(float v[9], int lane) {
    {
        const bool h = lane & 16;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const float send = h ? v[i] : v[i + 4], keep = h ? v[i + 4] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
    }
    {
        const bool h = lane & 8;
#pragma unroll
        for (int i = 0; i < 2; i++) {
            const float send = h ? v[i] : v[i + 2], keep = h ? v[i + 2] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
    }
    {
        const bool h = lane & 4;
        const float send = h ? v[0] : v[1], keep = h ? v[1] : v[0];
        v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], 2);
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[8] += __shfl_xor_sync(0xffffffffu, v[8], o);
}

__global__ void __launch_bounds__(BL_THREADS)
k_blend_bwd(int W, int H, int tiles_per_view, const float4 *__restrict__ rec, const float *__restrict__ bg,
            const uint8_t *__restrict__ compute_locally, const uint2 *__restrict__ ranges,
            const uint32_t *__restrict__ ids, const float *__restrict__ final_T,
            const uint32_t *__restrict__ n_contrib, const float *__restrict__ dL_dimage,
            float *__restrict__ d_means2D, float *__restrict__ d_conic_opacity, float *__restrict__ d_rgb) {
    __shared__ SRec s_rec[BW8_CHUNK];
    __shared__ uint32_t s_id[BW8_CHUNK];
    __shared__ uint8_t s_cull[BW8_CHUNK];
    __shared__ float s_acc[BL_WARPS][9][BW8_STRIDE];
    __shared__ uint32_t s_mask[BL_WARPS][BW8_CHUNK / 32];
    __shared__ uint32_t s_max[BL_WARPS];
    const int gx = (W + GS_BLOCK_X - 1) / GS_BLOCK_X;
    if (!compute_locally[blockIdx.x]) return;
    const int view = blockIdx.x / tiles_per_view, tile = blockIdx.x - view * tiles_per_view;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int px, py;
    pixel_of_thread(tile, gx, px, py);
    const bool inside = px < W && py < H;
    const size_t HW = (size_t)H * W;
    const size_t pix = (size_t)py * W + px;
    final_T += (size_t)view * HW;
    n_contrib += (size_t)view * HW;
    dL_dimage += (size_t)view * 3 * HW;
    const uint2 range = ranges[blockIdx.x];
    const float X0 = (float)((tile % gx) * GS_BLOCK_X), Y0 = (float)((tile / gx) * GS_BLOCK_Y);
    const float pxf = (float)px, pyf = (float)py;
    const float T_final = inside ? final_T[pix] : 0.f;
    const uint32_t last = inside ? n_contrib[pix] : 0u;
    float dp0 = 0.f, dp1 = 0.f, dp2 = 0.f;
    if (inside) { dp0 = dL_dimage[pix]; dp1 = dL_dimage[HW + pix]; dp2 = dL_dimage[2 * HW + pix]; }
    const float bgdot = bg[0] * dp0 + bg[1] * dp1 + bg[2] * dp2;
    const float ddelx_dx = 0.5f * (float)W, ddely_dy = 0.5f * (float)H;
    // entries past the tile's deepest last-contributor cannot matter
    uint32_t m = last;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) s_max[warp] = m;
    __syncthreads();
    uint32_t n_total = 0;
#pragma unroll
    for (int w = 0; w < BL_WARPS; w++) n_total = max(n_total, s_max[w]);
    const uint32_t wlast = m;  // deepest entry this warp's pixels reach
    // B = colour of everything behind the current splat (back-to-front recurrence B += alpha (c - B)); with alpha
    // forced to 0 for lanes that do not blend this splat every state update below is a no-op for them, so the
    // blend path needs no per-lane branches or conditional moves.
    float T = T_final, B0 = 0.f, B1 = 0.f, B2 = 0.f;
    const int n_chunks = ((int)n_total + BW8_CHUNK - 1) / BW8_CHUNK;
    for (int c = n_chunks - 1; c >= 0; c--) {
        const int base = c * BW8_CHUNK;
        const int cnt = min(BW8_CHUNK, (int)n_total - base);
        __syncthreads();  // previous chunk's flush has finished reading shared memory
        if ((int)threadIdx.x < cnt) {
            const uint32_t g = ids[range.x + base + threadIdx.x];
            s_id[threadIdx.x] = g;
            const float4 *r = rec + (size_t)3 * g;
            const float4 a = __ldg(r), b = __ldg(r + 1), cc = __ldg(r + 2);
            s_rec[threadIdx.x].a = a; s_rec[threadIdx.x].b = b; s_rec[threadIdx.x].c = cc;
            s_cull[threadIdx.x] = (uint8_t)block_mask(a, b, cc.z, cc.w, X0, Y0);
        }
        uint32_t wmask = 0u;  // lane q holds bits [32q, 32q+32) of "this warp produced a partial for entry j"
        __syncthreads();
        if ((uint32_t)base < wlast) {
            for (int g0 = (cnt - 1) & ~31; g0 >= 0; g0 -= 32) {
                // lane l inspects entry g0 + 31 - l, so the LOWEST set bit of the ballot is the DEEPEST candidate and
                // the walk (back to front) pops bits with the cheap x & (x - 1)
                const int jj = g0 + 31 - lane;
                uint32_t cand = __ballot_sync(0xffffffffu, jj < cnt && ((s_cull[jj] >> warp) & 1));
                uint32_t mybits = 0u;
                const int last_rel = (int)last - base;  // entry j of this chunk is live for this pixel iff j < last_rel
                while (cand) {
                    const int b31 = 32 - __ffs(cand);   // = 31 - (index of the lowest set bit)
                    const int j = g0 + b31;
                    cand &= cand - 1u;
                    const SRec *sr = &s_rec[j];
                    const float4 a = sr->a, b = sr->b;
                    const float dx = a.x - pxf, dy = a.y - pyf;
                    const float power = dx * (a.z * dx + a.w * dy) + b.x * dy * dy;
                    bool ok = (j < last_rel) && power >= b.z;
                    if (!__any_sync(0xffffffffu, ok)) continue;
                    const float G = gs_exp_neg(power);
                    const float alpha = fminf(ALPHA_MAX, b.y * G);
                    ok = ok && power <= 0.f;   // thr <= power <= 0  <=>  alpha >= 1/255
                    if (!__any_sync(0xffffffffu, ok)) continue;
                    // Per-pixel weight m = dL/dG * G; the per-splat gradients are its moments over the pixels
                    // (S0, Sx, Sy, Sxx, Sxy, Syy) plus three colour sums; they are combined with the splat's
                    // constants once per (splat, tile) in the flush below.
                    float v[9];
                    {
                        const float2 gb = *reinterpret_cast<const float2 *>(&sr->c);
                        const float ae = ok ? alpha : 0.f;   // effective alpha: 0 = this lane skips the splat
                        float inv;                            // 1/(1-ae), 1-ae in [0.01, 1]: one MUFU.RCP
                        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(1.f - ae));
                        T = T * inv;                          // transmittance in front of this splat
                        const float d0 = b.w - B0, d1 = gb.x - B1, d2 = gb.y - B2;
                        const float dL_dalpha = (d0 * dp0 + d1 * dp1 + d2 * dp2) * T - (T_final * inv) * bgdot;
                        const float mw = ok ? b.y * dL_dalpha * G : 0.f;
                        const float dch = ae * T;
                        B0 += ae * d0; B1 += ae * d1; B2 += ae * d2;
                        const float mx_ = mw * dx, my_ = mw * dy;
                        v[0] = mx_; v[1] = my_; v[2] = mx_ * dx; v[3] = mx_ * dy; v[4] = my_ * dy; v[5] = mw;
                        v[6] = dch * dp0; v[7] = dch * dp1; v[8] = dch * dp2;
                    }
                    warp_reduce9(v, lane);
                    if ((lane & 3) == 0) s_acc[warp][lane >> 2][j] = v[0];
                    if (lane == 1) s_acc[warp][8][j] = v[8];
                    mybits |= 1u << b31;
                }
                if (lane == (g0 >> 5)) wmask = mybits;
            }
        }
        if (lane < BW8_CHUNK / 32) s_mask[warp][lane] = wmask;
        __syncthreads();
        if ((int)threadIdx.x < cnt) {
            const int j = threadIdx.x;
            float s[9];
#pragma unroll
            for (int q = 0; q < 9; q++) s[q] = 0.f;
            bool any = false;
#pragma unroll
            for (int w = 0; w < BL_WARPS; w++) {
                if ((s_mask[w][j >> 5] >> (j & 31)) & 1u) {
                    any = true;
#pragma unroll
                    for (int q = 0; q < 9; q++) s[q] += s_acc[w][q][j];
                }
            }
            if (any) {
                const uint32_t g = s_id[j];
                const float4 a = s_rec[j].a, b = s_rec[j].b;  // (mx,my,a',b') (c',opacity,thr,red); A=-2a' B=-b' C=-2c'
                // d power/d mean = (2a'dx + b'dy, 2c'dy + b'dx); dL/dmeans2D is per NDC unit: * (W/2, H/2)
                atomicAdd(d_means2D + 2 * (size_t)g, (2.f * a.z * s[0] + a.w * s[1]) * ddelx_dx);
                atomicAdd(d_means2D + 2 * (size_t)g + 1, (2.f * b.x * s[1] + a.w * s[0]) * ddely_dy);
                atomicAdd(d_conic_opacity + 4 * (size_t)g, -0.5f * s[2]);
                atomicAdd(d_conic_opacity + 4 * (size_t)g + 1, -s[3]);
                atomicAdd(d_conic_opacity + 4 * (size_t)g + 2, -0.5f * s[4]);
                atomicAdd(d_conic_opacity + 4 * (size_t)g + 3, __fdividef(s[5], b.y));
                atomicAdd(d_rgb + 3 * (size_t)g, s[6]);
                atomicAdd(d_rgb + 3 * (size_t)g + 1, s[7]);
                atomicAdd(d_rgb + 3 * (size_t)g + 2, s[8]);
            }
        }
    }
}


// ---- backward, segment-parallel (round 2; kept behind gs_debug_set(GS_DEBUG_BWD_SEG_R2)) ----------------------------
// One warp = one (tile, segment) unit, all 256 pixels of the tile: lane l owns pixel (l & 7, l >> 3) of each 8x4 block.
// Per-pixel state, walking back to front:  T = transmittance in front of the current splat,
//   S = sum over the entries BEHIND it of alpha_j T_j (c_j . dL/dpixel)  +  T_final (bg . dL/dpixel)
// so that dL/dalpha_k = T_k (c_k . dp) - S_k / (1 - alpha_k) -- the scalar form of the published recurrence
// (accum_rec / last_alpha, cuda_rasterizer/backward.cu) with the background term folded into the start value.
#define SG_WARPS 4
#define SG_THREADS (SG_WARPS * 32)
#define SG_STAGE 32  // records staged per pass: one per lane

#ifndef SG_MIN_CTAS
#define SG_MIN_CTAS 8
#endif
// values needed only when a pass is staged (every 32 entries) or in the per-splat tail live in shared memory, not in
// registers: the walk keeps 16 state + 9 sum + 12 record registers per lane and wants 8 CTAs per SM
struct SegCold { const uint32_t *ids; const uint16_t *cull; int cnt; uint32_t blive, blive_hi; };

__global__ void __launch_bounds__(SG_THREADS, SG_MIN_CTAS)
k_blend_bwd_seg(int W, int H, int tiles_per_view, const float4 *__restrict__ rec, const float *__restrict__ bg,
                const uint2 *__restrict__ ranges, const uint32_t *__restrict__ ids, const float *__restrict__ final_T,
                const uint32_t *__restrict__ n_contrib, const float *__restrict__ dL_dimage, const SegWs seg,
                float *__restrict__ d_means2D, float *__restrict__ d_conic_opacity, float *__restrict__ d_rgb) {
    __shared__ SRec s_rec_all[SG_WARPS][SG_STAGE];   // c = (green, blue, 1 / opacity, splat id bits)
    __shared__ float4 s_pix_all[SG_WARPS][8 * 32];   // per pixel: dL/dpixel (3) and the number of live entries (int bits)
    __shared__ uint32_t s_mask_all[SG_WARPS][SG_STAGE];
    __shared__ uint4 s_role_all[SG_WARPS][32];       // per lane: RED target pointer (lo, hi), row stride, scale bits
    __shared__ SegCold s_cold_all[SG_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t u = blockIdx.x * SG_WARPS + warp;
    if (u >= *seg.n_units) return;  // warps are independent: no CTA-level synchronisation anywhere below
    SRec *s_rec = s_rec_all[warp];
    float4 *s_pix = s_pix_all[warp] + lane;
    uint32_t *s_mask = s_mask_all[warp];
    const uint2 unit = seg.units[u];
    const int tile_g = (int)unit.x, sidx = (int)unit.y;
    const int view = tile_g / tiles_per_view, tile = tile_g - view * tiles_per_view;
    const int gx = (W + GS_BLOCK_X - 1) / GS_BLOCK_X;
    const uint2 range = ranges[tile_g];
    const int tl = (int)seg.tile_last[tile_g];
    const int seg_base = sidx * SEG_K;
    const int cnt = min(SEG_K, tl - seg_base);
    const size_t HW = (size_t)H * W;
    final_T += (size_t)view * HW;
    n_contrib += (size_t)view * HW;
    dL_dimage += (size_t)view * 3 * HW;
    const int X0 = (tile % gx) * GS_BLOCK_X, Y0 = (tile / gx) * GS_BLOCK_Y;
    const float bg0 = bg[0], bg1 = bg[1], bg2 = bg[2];
    const float4 *ck = seg.ckpt + ((size_t)(range.x / SEG_K) + tile_g + sidx) * SEG_SLOT + lane;
    float T[8], S[8];
    uint32_t blive = 0, blive_hi = 0;  // byte b: deepest live entry of block b over the warp
#pragma unroll
    for (int b = 0; b < 8; b++) {
        const int px = X0 + (b & 1) * 8 + (lane & 7), py = Y0 + (b >> 1) * 4 + (lane >> 3);
        const bool inside = px < W && py < H;
        const size_t pix = (size_t)py * W + px;
        float Tf = 0.f, d0 = 0.f, d1 = 0.f, d2 = 0.f;
        int last = 0;
        if (inside) {
            Tf = final_T[pix];
            last = (int)n_contrib[pix];
            d0 = dL_dimage[pix]; d1 = dL_dimage[HW + pix]; d2 = dL_dimage[2 * HW + pix];
        }
        const float sbg = Tf * (bg0 * d0 + bg1 * d1 + bg2 * d2);
        T[b] = Tf;
        S[b] = sbg;
        if (last > seg_base + SEG_K) {  // alive beyond this segment: the forward left its state at the boundary
            const float4 c = ck[b * 32];
            T[b] = c.x;
            S[b] = c.y * d0 + c.z * d1 + c.w * d2 + sbg;
        }
        const int live = max(0, min(SEG_K, last - seg_base));  // entries [0, live) of the segment are in front of the
        s_pix[b * 32] = make_float4(d0, d1, d2, __int_as_float(live));  // pixel's last contributor
        const uint32_t m = __reduce_max_sync(FULL, (uint32_t)live);
        if (b < 4) blive |= m << (8 * b); else blive_hi |= m << (8 * (b - 4));
    }
    {   // lane roles of the final RED: lanes 0,4,...,28 hold sums 0..7 after the butterfly, lane 1 sends sum 8
        const int role = (lane & 3) == 0 ? (lane >> 2) : (lane == 1 ? 8 : -1);
        float *rptr = nullptr;
        uint32_t rstride = 0;
        float rscale = 0.f;
        if (role >= 0) {
            if (role < 2) { rptr = d_means2D + role; rstride = 2; rscale = role == 0 ? -0.5f * (float)W : -0.5f * (float)H; }
            else if (role < 6) { rptr = d_conic_opacity + (role - 2); rstride = 4; rscale = role == 3 ? -1.f : (role == 5 ? 1.f : -0.5f); }
            else { rptr = d_rgb + (role - 6); rstride = 3; rscale = 1.f; }
        }
        const unsigned long long rp = (unsigned long long)rptr;
        s_role_all[warp][lane] = make_uint4((uint32_t)rp, (uint32_t)(rp >> 32), rstride, __float_as_uint(rscale));
        if (lane == 0) {
            SegCold c;
            c.ids = ids + range.x + seg_base; c.cull = seg.cull + range.x + seg_base; c.cnt = cnt; c.blive = blive; c.blive_hi = blive_hi;
            s_cold_all[warp] = c;
        }
    }
    const uint4 *s_role = &s_role_all[warp][lane];
    const SegCold *s_cold = &s_cold_all[warp];
    const float pxf0 = (float)(X0 + (lane & 7)), pyf0 = (float)(Y0 + (lane >> 3));
    for (int pass = (cnt - 1) / SG_STAGE; pass >= 0; pass--) {
        // stage 32 records, one per lane; entry i keeps only the blocks it can reach (bounding box of {alpha >= 1/255})
        // that still have a live pixel at depth i
        const int p0 = pass * SG_STAGE;
        __syncwarp();
        const SegCold cold = *s_cold;
        const int pn = min(SG_STAGE, cold.cnt - p0);
        if (lane < pn) {
            const int i = p0 + lane;
            const uint32_t g = cold.ids[i];
            const float4 *r = rec + (size_t)3 * g;
            const float4 a = __ldg(r), b = __ldg(r + 1), c = __ldg(r + 2);
            // the forward's 4x4-block mask of this entry (ellipse_bands, computed once per (splat, tile)); an 8x4 block is
            // two horizontally adjacent 4x4 blocks: OR the bit pairs, then pack the even bits
            uint32_t m = cold.cull[i];
            m = (m | (m >> 1)) & 0x5555u;
            m = (m | (m >> 1)) & 0x3333u;
            m = (m | (m >> 2)) & 0x0f0fu;
            m = (m | (m >> 4)) & 0x00ffu;
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const uint32_t bl = ((q < 4 ? cold.blive : cold.blive_hi) >> (8 * (q & 3))) & 0xffu;
                if ((uint32_t)i >= bl) m &= ~(1u << q);
            }
            // positive form q = -power, t = -thr (see k_blend_fwd2's staging): the pixel test is one unsigned compare
            s_rec[lane].a = make_float4(a.x, a.y, -a.z, -a.w);
            s_rec[lane].b = make_float4(-b.x, b.y, fmaxf(-b.z, 0.f), b.w);
            s_rec[lane].c = make_float4(c.x, c.y, gs_rcp_approx(b.y), __uint_as_float(g));
            s_mask[lane] = m;
        }
        __syncwarp();
        for (int jl = pn - 1; jl >= 0; jl--) {
            // warp-uniform by construction; the redux makes that visible to the compiler (uniform branches, no
            // reconvergence bookkeeping around the votes below)
            const uint32_t m8 = __reduce_or_sync(FULL, s_mask[jl]);
            if (m8 == 0u) continue;
            const int j = p0 + jl;
            const float4 a = s_rec[jl].a, b4 = s_rec[jl].b;
            const float2 c4 = *reinterpret_cast<const float2 *>(&s_rec[jl].c);  // (green, blue)
            const float mxl = a.x - pxf0, myl = a.y - pyf0;
            float v[9];
#pragma unroll
            for (int q = 0; q < 9; q++) v[q] = 0.f;
            bool any_full = false;
#pragma unroll
            for (int b = 0; b < 8; b++) {
                if (m8 & (1u << b)) {
                    const float4 pc = s_pix[b * 32];
                    const float dx = mxl - (float)((b & 1) * 8), dy = myl - (float)((b >> 1) * 4);
                    const float q = dx * (a.z * dx + a.w * dy) + b4.x * dy * dy;   // -power
                    const bool ok = (j < __float_as_int(pc.w)) && __float_as_uint(q) <= __float_as_uint(b4.z);
                    if (__any_sync(FULL, ok)) {
                        const float G = gs_exp_neg(-q);
                        const float alpha = fminf(ALPHA_MAX, b4.y * G);
                        const float ae = ok ? alpha : 0.f;   // effective alpha: 0 = this lane skips the splat
                        float inv;                            // 1/(1-ae), 1-ae in [0.01, 1]: one MUFU.RCP
                        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(1.f - ae));
                        const float Tk = T[b] * inv;          // transmittance in front of this splat
                        T[b] = Tk;
                        const float cd = b4.w * pc.x + c4.x * pc.y + c4.y * pc.z;
                        const float dL_dalpha = cd * Tk - S[b] * inv;
                        const float mw = ok ? b4.y * dL_dalpha * G : 0.f;
                        const float dch = ae * Tk;
                        S[b] += dch * cd;
                        const float mx_ = mw * dx, my_ = mw * dy;
                        v[0] += mx_; v[1] += my_; v[2] += mx_ * dx; v[3] += mx_ * dy; v[4] += my_ * dy; v[5] += mw;
                        v[6] += dch * pc.x; v[7] += dch * pc.y; v[8] += dch * pc.z;
                        any_full = true;
                    }
                }
            }
            if (!any_full) continue;
            {   // per-lane pre-mix (linear, commutes with the sums), so that every reduced value is ONE output element:
                // d power/d mean = (2a'dx + b'dy, 2c'dy + b'dx); dL/dopacity = sum(m) / opacity
                // (the staged a.z, a.w, b4.x are -a', -b', -c': the sign sits in the roles' scale factors)
                const float sx = v[0], sy = v[1];
                v[0] = 2.f * a.z * sx + a.w * sy;
                v[1] = 2.f * b4.x * sy + a.w * sx;
                v[5] *= s_rec[jl].c.z;
            }
            warp_reduce9(v, lane);
            const uint4 ro = *s_role;
            const float val = (lane == 1 ? v[8] : v[0]) * __uint_as_float(ro.w);
            float *rptr = reinterpret_cast<float *>((unsigned long long)ro.x | ((unsigned long long)ro.y << 32));
            // red.global: the pointer was rebuilt from integers, so a plain atomicAdd compiles to a GENERIC atomic with
            // an address-space check and a shared-memory CAS fallback behind it
            if (rptr) asm volatile("red.global.add.f32 [%0], %1;" ::"l"(rptr + (size_t)__float_as_uint(s_rec[jl].c.w) * ro.z), "f"(val) : "memory");
        }
    }
}

// ---- backward, segment-parallel, round 3 (default) ---------------------------------------------------------------------
// The unit, the per-pixel state and the per-pixel arithmetic of k_blend_bwd_seg (which stays behind GS_DEBUG_BWD_SEG_R2 for
// A/B runs); the nine sums of a splat hold the same values bit for bit, only their reduction over the warp is ordered
// differently.  Fewer issued instructions per (splat, tile):
//   * staging compacts a pass: only entries whose trimmed 8x4 mask is non-empty get a slot (and have their record
//     gathered), so the walk spends nothing on an entry no block of the warp can use;
//   * the sums accumulate as packed pairs (FMUL2 / FADD2 / FFMA2): (m dx, m dy), (m dx^2, m dx dy), colour 0 and 1;
//   * two consecutive splats share the end of the reduction.  Each runs butterfly levels 16 and 8 on its own (down to 3
//     values per lane: warp_reduce9_to3); the first one's 3 values wait in registers for the second, and levels 4, 2, 1
//     reduce the 6 values of both at once (warp_reduce_pair: 22 instead of 28 shuffles per two splats), ending in ONE RED
//     set of 18 lanes.  A splat left over at the end of the unit is reduced against zeros.

// levels 16 and 8 of warp_reduce9: afterwards v[0] / v[1] hold value (lane >> 2 & 6) / (lane >> 2 & 6) + 1 summed over the
// lanes that differ in bits 3 and 4, v[8] value 8 likewise
GS_D void warp_reduce9_to3(float v[9], int lane) {
    {
        const bool h = lane & 16;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const float send = h ? v[i] : v[i + 4], keep = h ? v[i + 4] : v[i];
            v[i] = keep + __shfl_xor_sync(FULL, send, 16);
        }
    }
    {
        const bool h = lane & 8;
#pragma unroll
        for (int i = 0; i < 2; i++) {
            const float send = h ? v[i] : v[i + 2], keep = h ? v[i + 2] : v[i];
            v[i] = keep + __shfl_xor_sync(FULL, send, 8);
        }
    }
    v[8] += __shfl_xor_sync(FULL, v[8], 16);
    v[8] += __shfl_xor_sync(FULL, v[8], 8);
}

// levels 4, 2, 1 for two splats A and B (their warp_reduce9_to3 results).  Returns, in lane 4i the warp total of A's value i,
// in lane 4i + 2 that of B's value i (i < 8), in lane 1 A's value 8 and in lane 5 B's value 8.
GS_D float warp_reduce_pair(float a0, float a1, float a8, float b0, float b1, float b8, int lane) {
    const bool h2 = lane & 4, h1 = lane & 2, h0 = lane & 1;
    const float x = (h2 ? a1 : a0) + __shfl_xor_sync(FULL, h2 ? a0 : a1, 4);
    const float y = (h2 ? b1 : b0) + __shfl_xor_sync(FULL, h2 ? b0 : b1, 4);
    float z = (h2 ? b8 : a8) + __shfl_xor_sync(FULL, h2 ? a8 : b8, 4);
    const float w = (h1 ? y : x) + __shfl_xor_sync(FULL, h1 ? x : y, 2);
    z += __shfl_xor_sync(FULL, z, 2);
    return (h0 ? z : w) + __shfl_xor_sync(FULL, h0 ? w : z, 1);
}

// the RED of warp_reduce_pair's result: role z = (row stride) | (splat B ? 256 : 0); only_a: the unit's last splat has no
// partner
GS_D void seg_red_pair(const uint4 ro, float val, uint32_t id_a, uint32_t id_b, bool only_a) {
    float *rptr = reinterpret_cast<float *>((unsigned long long)ro.x | ((unsigned long long)ro.y << 32));
    const bool second = ro.z & 256u;
    const uint32_t id = second ? id_b : id_a;
    // red.global: see k_blend_bwd_seg
    if (rptr && !(only_a && second))
        asm volatile("red.global.add.f32 [%0], %1;" ::"l"(rptr + (size_t)id * (ro.z & 255u)), "f"(val * __uint_as_float(ro.w))
                     : "memory");
}

struct SegWarp3 {
    SRec rec[SG_STAGE];      // compacted; c = (green, blue, 1 / opacity, splat id bits)
    float4 pix[8 * 32];      // per pixel: dL/dpixel (3) and the number of live entries (int bits)
    uint32_t mask[SG_STAGE]; // compacted: 8x4 block mask | (entry - pass start) << 8
    uint4 role[32];          // per lane: RED target pointer (lo, hi), row stride | splat B, scale bits
    float4 pend[32];         // per lane: the waiting splat's three partial sums and its id bits
    SegCold cold;
};

__global__ void __launch_bounds__(SG_THREADS, SG_MIN_CTAS)
k_blend_bwd_seg3(int W, int H, int tiles_per_view, const float4 *__restrict__ rec, const float *__restrict__ bg,
                 const uint2 *__restrict__ ranges, const uint32_t *__restrict__ ids, const float *__restrict__ final_T,
                 const uint32_t *__restrict__ n_contrib, const float *__restrict__ dL_dimage, const SegWs seg,
                 float *__restrict__ d_means2D, float *__restrict__ d_conic_opacity, float *__restrict__ d_rgb) {
    // one struct per warp, so that every per-lane slot is one base register plus a constant offset
    __shared__ SegWarp3 s_all[SG_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t u = blockIdx.x * SG_WARPS + warp;
    if (u >= *seg.n_units) return;  // warps are independent: no CTA-level synchronisation anywhere below
    SegWarp3 &sw = s_all[warp];
    SRec *s_rec = sw.rec;
    float4 *s_pix = sw.pix + lane;
    uint32_t *s_mask = sw.mask;
    const uint2 unit = seg.units[u];
    const int tile_g = (int)unit.x, sidx = (int)unit.y;
    const int view = tile_g / tiles_per_view, tile = tile_g - view * tiles_per_view;
    const int gx = (W + GS_BLOCK_X - 1) / GS_BLOCK_X;
    const uint2 range = ranges[tile_g];
    const int tl = (int)seg.tile_last[tile_g];
    const int seg_base = sidx * SEG_K;
    const int cnt = min(SEG_K, tl - seg_base);
    const size_t HW = (size_t)H * W;
    final_T += (size_t)view * HW;
    n_contrib += (size_t)view * HW;
    dL_dimage += (size_t)view * 3 * HW;
    const int X0 = (tile % gx) * GS_BLOCK_X, Y0 = (tile / gx) * GS_BLOCK_Y;
    const float bg0 = bg[0], bg1 = bg[1], bg2 = bg[2];
    const float4 *ck = seg.ckpt + ((size_t)(range.x / SEG_K) + tile_g + sidx) * SEG_SLOT + lane;
    float T[8], S[8];
    uint32_t blive = 0, blive_hi = 0;  // byte b: deepest live entry of block b over the warp
#pragma unroll
    for (int b = 0; b < 8; b++) {
        const int px = X0 + (b & 1) * 8 + (lane & 7), py = Y0 + (b >> 1) * 4 + (lane >> 3);
        const bool inside = px < W && py < H;
        const size_t pix = (size_t)py * W + px;
        float Tf = 0.f, d0 = 0.f, d1 = 0.f, d2 = 0.f;
        int last = 0;
        if (inside) {
            Tf = final_T[pix];
            last = (int)n_contrib[pix];
            d0 = dL_dimage[pix]; d1 = dL_dimage[HW + pix]; d2 = dL_dimage[2 * HW + pix];
        }
        const float sbg = Tf * (bg0 * d0 + bg1 * d1 + bg2 * d2);
        T[b] = Tf;
        S[b] = sbg;
        if (last > seg_base + SEG_K) {  // alive beyond this segment: the forward left its state at the boundary
            const float4 c = ck[b * 32];
            T[b] = c.x;
            S[b] = c.y * d0 + c.z * d1 + c.w * d2 + sbg;
        }
        const int live = max(0, min(SEG_K, last - seg_base));  // entries [0, live) of the segment are in front of the
        s_pix[b * 32] = make_float4(d0, d1, d2, __int_as_float(live));  // pixel's last contributor
        const uint32_t m = __reduce_max_sync(FULL, (uint32_t)live);
        if (b < 4) blive |= m << (8 * b); else blive_hi |= m << (8 * (b - 4));
    }
    {   // lane roles of the final RED (warp_reduce_pair): lane 4i / 4i + 2 add value i of splat A / B, lane 1 / 5 value 8
        const bool even = !(lane & 1);
        const int role = even ? (lane >> 2) : (lane == 1 || lane == 5 ? 8 : -1);
        const uint32_t second = even ? (lane >> 1) & 1 : (lane >> 2) & 1;
        float *rptr = nullptr;
        uint32_t rstride = 0;
        float rscale = 0.f;
        if (role >= 0) {
            if (role < 2) { rptr = d_means2D + role; rstride = 2; rscale = role == 0 ? -0.5f * (float)W : -0.5f * (float)H; }
            else if (role < 6) { rptr = d_conic_opacity + (role - 2); rstride = 4; rscale = role == 3 ? -1.f : (role == 5 ? 1.f : -0.5f); }
            else { rptr = d_rgb + (role - 6); rstride = 3; rscale = 1.f; }
        }
        const unsigned long long rp = (unsigned long long)rptr;
        sw.role[lane] = make_uint4((uint32_t)rp, (uint32_t)(rp >> 32), rstride | (second << 8), __float_as_uint(rscale));
        if (lane == 0) {
            SegCold c;
            c.ids = ids + range.x + seg_base; c.cull = seg.cull + range.x + seg_base; c.cnt = cnt; c.blive = blive; c.blive_hi = blive_hi;
            sw.cold = c;
        }
    }
    const uint4 *s_role = &sw.role[lane];
    const SegCold *s_cold = &sw.cold;
    const float pxf0 = (float)(X0 + (lane & 7)), pyf0 = (float)(Y0 + (lane >> 3));
    // a splat waiting for a partner in the shared reduction tail keeps its three partial sums and its id in shared memory
    // (in registers they pushed the walk's state into local memory)
    float4 *s_pend = &sw.pend[lane];
    bool pend = false;
    for (int p0 = (cnt - 1) & ~(SG_STAGE - 1); p0 >= 0; p0 -= SG_STAGE) {
        // stage up to 32 entries, one per lane; entry i keeps only the blocks it can reach that still have a live pixel at
        // depth i, and only entries with a block left get a (compacted) slot
        __syncwarp();
        const SegCold cold = *s_cold;
        const int pn = min(SG_STAGE, cold.cnt - p0);
        uint32_t m = 0u;
        if (lane < pn) {
            const int i = p0 + lane;
            // the forward's 4x4-block mask of this entry; an 8x4 block is two horizontally adjacent 4x4 blocks: OR the bit
            // pairs, then pack the even bits
            m = cold.cull[i];
            m = (m | (m >> 1)) & 0x5555u;
            m = (m | (m >> 1)) & 0x3333u;
            m = (m | (m >> 2)) & 0x0f0fu;
            m = (m | (m >> 4)) & 0x00ffu;
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const uint32_t bl = ((q < 4 ? cold.blive : cold.blive_hi) >> (8 * (q & 3))) & 0xffu;
                if ((uint32_t)i >= bl) m &= ~(1u << q);
            }
        }
        const uint32_t act = __ballot_sync(FULL, m != 0u);
        if (m != 0u) {
            const int slot = __popc(act & ((1u << lane) - 1u));
            const uint32_t g = cold.ids[p0 + lane];
            const float4 *r = rec + (size_t)3 * g;
            const float4 a = __ldg(r), b = __ldg(r + 1), c = __ldg(r + 2);
            // positive form q = -power, t = -thr (see k_blend_fwd2's staging): the pixel test is one unsigned compare
            s_rec[slot].a = make_float4(a.x, a.y, -a.z, -a.w);
            s_rec[slot].b = make_float4(-b.x, b.y, fmaxf(-b.z, 0.f), b.w);
            s_rec[slot].c = make_float4(c.x, c.y, gs_rcp_approx(b.y), __uint_as_float(g));
            s_mask[slot] = m | ((uint32_t)lane << 8);
        }
        __syncwarp();
        for (int k = __popc(act) - 1; k >= 0; k--) {
            // warp-uniform by construction; the redux makes that visible to the compiler (see k_blend_bwd_seg)
            const uint32_t mw8 = __reduce_or_sync(FULL, s_mask[k]);
            const uint32_t m8 = mw8 & 0xffu;
            const int j = p0 + (int)(mw8 >> 8);
            const float4 a = s_rec[k].a, b4 = s_rec[k].b;
            const float2 c4 = *reinterpret_cast<const float2 *>(&s_rec[k].c);  // (green, blue)
            const float mxl = a.x - pxf0, myl = a.y - pyf0;
            // the nine sums: (m dx, m dy), (m dx^2, m dx dy), m dy^2, m, (colour 0, colour 1), colour 2
            const p2 zero2 = p2_bc(0.f);
            p2 s01 = zero2, s23 = zero2, s67 = zero2;
            float s4 = 0.f, s5 = 0.f, s8 = 0.f;
            bool any_full = false;
#pragma unroll
            for (int b = 0; b < 8; b++) {
                if (m8 & (1u << b)) {
                    const float4 pc = s_pix[b * 32];
                    const float dx = mxl - (float)((b & 1) * 8), dy = myl - (float)((b >> 1) * 4);
                    const float q = dx * (a.z * dx + a.w * dy) + b4.x * dy * dy;   // -power
                    const bool ok = (j < __float_as_int(pc.w)) && __float_as_uint(q) <= __float_as_uint(b4.z);
                    if (__any_sync(FULL, ok)) {
                        const float G = gs_exp_neg(-q);
                        const float alpha = fminf(ALPHA_MAX, b4.y * G);
                        const float ae = ok ? alpha : 0.f;   // effective alpha: 0 = this lane skips the splat
                        float inv;                            // 1/(1-ae), 1-ae in [0.01, 1]: one MUFU.RCP
                        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(1.f - ae));
                        const float Tk = T[b] * inv;          // transmittance in front of this splat
                        T[b] = Tk;
                        const float cd = b4.w * pc.x + c4.x * pc.y + c4.y * pc.z;
                        const float dL_dalpha = cd * Tk - S[b] * inv;
                        const float mw = ok ? b4.y * dL_dalpha * G : 0.f;
                        const float dch = ae * Tk;
                        S[b] += dch * cd;
                        const p2 d = p2_make(dx, dy);
                        const p2 mxy = p2_mul(p2_bc(mw), d);                 // (m dx, m dy)
                        p2_add_acc(s01, mxy);
                        p2_fma_acc(s23, p2_bc(p2_lo(mxy)), d);               // (m dx dx, m dx dy)
                        s4 += p2_hi(mxy) * dy;
                        s5 += mw;
                        p2_fma_acc(s67, p2_bc(dch), p2_make(pc.x, pc.y));
                        s8 += dch * pc.z;
                        any_full = true;
                    }
                }
            }
            if (!any_full) continue;
            float v[9];
            {   // per-lane pre-mix as in k_blend_bwd_seg: every reduced value is ONE output element
                const float sx = p2_lo(s01), sy = p2_hi(s01);
                v[0] = 2.f * a.z * sx + a.w * sy;
                v[1] = 2.f * b4.x * sy + a.w * sx;
                v[2] = p2_lo(s23); v[3] = p2_hi(s23); v[4] = s4;
                v[5] = s5 * s_rec[k].c.z;
                v[6] = p2_lo(s67); v[7] = p2_hi(s67); v[8] = s8;
            }
            warp_reduce9_to3(v, lane);
            const uint32_t id = __float_as_uint(s_rec[k].c.w);
            if (!pend) {
                *s_pend = make_float4(v[0], v[1], v[8], __uint_as_float(id));
                pend = true;
                continue;
            }
            const float4 pa = *s_pend;
            seg_red_pair(*s_role, warp_reduce_pair(pa.x, pa.y, pa.z, v[0], v[1], v[8], lane), __float_as_uint(pa.w), id, false);
            pend = false;
        }
    }
    if (pend) {
        const float4 pa = *s_pend;
        seg_red_pair(*s_role, warp_reduce_pair(pa.x, pa.y, pa.z, 0.f, 0.f, 0.f, lane), __float_as_uint(pa.w), 0u, true);
    }
}

template <bool STATS, bool CKPT>
static void launch_fwd(int grid, cudaStream_t stream, int W, int H, int T1, const float *rec, const float *bg,
                       const uint8_t *cl, const uint32_t *ranges, const uint32_t *ids, float *image, float *final_T,
                       uint32_t *n_contrib, int64_t *stats, const SegWs &seg) {
    if (g_gs_debug_flags & GS_DEBUG_FWD_HALFWARP)
        k_blend_fwd<STATS, CKPT><<<grid, BL_THREADS, 0, stream>>>(
            W, H, T1, reinterpret_cast<const float4 *>(rec), bg, cl, reinterpret_cast<const uint2 *>(ranges), ids, image,
            final_T, n_contrib, reinterpret_cast<unsigned long long *>(stats), seg);
    else
        k_blend_fwd2<STATS, CKPT><<<grid, F2_THREADS, 0, stream>>>(
            W, H, T1, reinterpret_cast<const float4 *>(rec), bg, cl, reinterpret_cast<const uint2 *>(ranges), ids, image,
            final_T, n_contrib, reinterpret_cast<unsigned long long *>(stats), seg);
}

int gs_launch_blend_forward(int num_views, int64_t R, int H, int W, const float *rec, const float *bg,
                            const uint8_t *compute_locally, const uint32_t *ranges, const uint32_t *ids_sorted,
                            float *image, float *final_T, uint32_t *n_contrib, int64_t *stats, void *seg_ws,
                            size_t seg_ws_bytes, cudaStream_t stream) {
    const int gx = (W + GS_BLOCK_X - 1) / GS_BLOCK_X, gy = (H + GS_BLOCK_Y - 1) / GS_BLOCK_Y;
    const int T1 = gx * gy;
    SegWs seg = {nullptr, nullptr, nullptr, nullptr};
    if (seg_ws) {
        if (seg_ws_bytes < seg_bytes(R, (int64_t)T1 * num_views)) {
            gs_set_error("gs_render_forward: segment workspace too small (%zu < %zu)", seg_ws_bytes,
                         seg_bytes(R, (int64_t)T1 * num_views));
            return GS_ENOMEM;
        }
        GS_REQUIRE(((uintptr_t)seg_ws & 255) == 0, "segment workspace must be 256-byte aligned");
        seg = seg_carve(seg_ws, R, (int64_t)T1 * num_views);
        GS_CUDA_TRY(cudaMemsetAsync(seg.n_units, 0, 256, stream));
    }
    if (stats) GS_CUDA_TRY(cudaMemsetAsync(stats, 0, 3 * sizeof(int64_t) * (size_t)num_views, stream));
    GsStageTimer timer(GS_STAGE_BLEND_FWD, stream);
    const int grid = T1 * num_views;
    if (stats && seg_ws)
        launch_fwd<true, true>(grid, stream, W, H, T1, rec, bg, compute_locally, ranges, ids_sorted, image, final_T, n_contrib, stats, seg);
    else if (stats)
        launch_fwd<true, false>(grid, stream, W, H, T1, rec, bg, compute_locally, ranges, ids_sorted, image, final_T, n_contrib, stats, seg);
    else if (seg_ws)
        launch_fwd<false, true>(grid, stream, W, H, T1, rec, bg, compute_locally, ranges, ids_sorted, image, final_T, n_contrib, stats, seg);
    else
        launch_fwd<false, false>(grid, stream, W, H, T1, rec, bg, compute_locally, ranges, ids_sorted, image, final_T, n_contrib, stats, seg);
    GS_LAUNCH_CHECK();
    return GS_OK;
}

extern "C" int gs_render_backward(int P, int64_t R, int image_height, int image_width, const float *rec,
                                  const float *bg, const uint8_t *compute_locally, const uint32_t *ranges,
                                  const uint32_t *ids_sorted, const float *final_T, const uint32_t *n_contrib,
                                  const float *dL_dimage, const void *seg_ws, size_t seg_ws_bytes, float *dL_dmeans2D,
                                  float *dL_dconic_opacity, float *dL_drgb, void *stream) {
    return gs_render_backward_batched(1, P, R, image_height, image_width, rec, bg, compute_locally, ranges, ids_sorted,
                                      final_T, n_contrib, dL_dimage, seg_ws, seg_ws_bytes, dL_dmeans2D, dL_dconic_opacity,
                                      dL_drgb, stream);
}

extern "C" int gs_render_backward_batched(int num_views, int P, int64_t R, int image_height, int image_width,
                                          const float *rec, const float *bg, const uint8_t *compute_locally,
                                          const uint32_t *ranges, const uint32_t *ids_sorted, const float *final_T,
                                          const uint32_t *n_contrib, const float *dL_dimage, const void *seg_ws,
                                          size_t seg_ws_bytes, float *dL_dmeans2D, float *dL_dconic_opacity,
                                          float *dL_drgb, void *stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GS_REQUIRE(num_views >= 1 && num_views <= GS_MAX_VIEWS, "num_views must be in [1, GS_MAX_VIEWS]");
    GS_REQUIRE(P >= 0 && R >= 0 && image_height > 0 && image_width > 0, "sizes");
    if (P == 0) return GS_OK;
    GS_REQUIRE(dL_dmeans2D && dL_dconic_opacity && dL_drgb, "null output");
    if (dL_dmeans2D == dL_dconic_opacity + 4 * (size_t)P && dL_drgb == dL_dmeans2D + 2 * (size_t)P) {
        GS_CUDA_TRY(cudaMemsetAsync(dL_dconic_opacity, 0, sizeof(float) * 9 * (size_t)P, stream));   // one block (ops._grad_block)
    } else {
        GS_CUDA_TRY(cudaMemsetAsync(dL_dmeans2D, 0, sizeof(float) * 2 * (size_t)P, stream));
        GS_CUDA_TRY(cudaMemsetAsync(dL_dconic_opacity, 0, sizeof(float) * 4 * (size_t)P, stream));
        GS_CUDA_TRY(cudaMemsetAsync(dL_drgb, 0, sizeof(float) * 3 * (size_t)P, stream));
    }
    if (R == 0) return GS_OK;
    GS_REQUIRE(rec && bg && compute_locally && ranges && ids_sorted && final_T && n_contrib && dL_dimage, "null input");
    const int gx = (image_width + GS_BLOCK_X - 1) / GS_BLOCK_X, gy = (image_height + GS_BLOCK_Y - 1) / GS_BLOCK_Y;
    GsStageTimer timer(GS_STAGE_BLEND_BWD, stream);
    if (seg_ws && !(g_gs_debug_flags & GS_DEBUG_BWD_TILE)) {
        const int64_t T = (int64_t)gx * gy * num_views;
        if (seg_ws_bytes < seg_bytes(R, T)) {
            gs_set_error("gs_render_backward: segment workspace too small");
            return GS_ENOMEM;
        }
        const SegWs seg = seg_carve(const_cast<void *>(seg_ws), R, T);
        const int64_t max_units = R / SEG_K + T;   // >= sum over tiles of ceil(walked entries / SEG_K)
        const unsigned grid = (unsigned)((max_units + SG_WARPS - 1) / SG_WARPS);
        if (g_gs_debug_flags & GS_DEBUG_BWD_SEG_R2)
            k_blend_bwd_seg<<<grid, SG_THREADS, 0, stream>>>(
                image_width, image_height, gx * gy, reinterpret_cast<const float4 *>(rec), bg,
                reinterpret_cast<const uint2 *>(ranges), ids_sorted, final_T, n_contrib, dL_dimage, seg, dL_dmeans2D,
                dL_dconic_opacity, dL_drgb);
        else
            k_blend_bwd_seg3<<<grid, SG_THREADS, 0, stream>>>(
                image_width, image_height, gx * gy, reinterpret_cast<const float4 *>(rec), bg,
                reinterpret_cast<const uint2 *>(ranges), ids_sorted, final_T, n_contrib, dL_dimage, seg, dL_dmeans2D,
                dL_dconic_opacity, dL_drgb);
        GS_LAUNCH_CHECK();
        return GS_OK;
    }
    k_blend_bwd<<<gx * gy * num_views, BL_THREADS, 0, stream>>>(
        image_width, image_height, gx * gy, reinterpret_cast<const float4 *>(rec), bg, compute_locally,
        reinterpret_cast<const uint2 *>(ranges), ids_sorted, final_T, n_contrib, dL_dimage, dL_dmeans2D, dL_dconic_opacity,
        dL_drgb);
    GS_LAUNCH_CHECK();
    return GS_OK;
}
