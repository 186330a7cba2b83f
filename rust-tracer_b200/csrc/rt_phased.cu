// rt_phased.cu -- PHASED variant: the TILE algorithm as four homogeneous launches.
//
// The fused TILE kernel mixes two very different kinds of work in one CTA: the
// hierarchy cull (one warp, a long dependent chain per step) and the per-sample
// tests (every lane busy).  Warps waiting for a cull hold registers and hide no
// latency.  Here each phase is its own launch on one stream, so every SM runs one
// kind of work at full occupancy; intermediates are a few MB and stay in L2:
//
//   K1 cull_primary   one warp per CULL tile (CW x CH pixel tiles): walks the
//                     skip-pointer hierarchy against the tile's cone, dropping what
//                     lies wholly behind a leaf that every ray of the tile hits
//                     (primary_occlusion); appends candidate chunks {v = c - eye,
//                     v.v, r*r, index, image-space box}, sorted front to back.
//   K2 test_primary   one warp per PIXEL tile: box pre-filter (warp rectangle, then
//                     the lane's own pixel block) + the reference's exact f32
//                     ray-sphere test (primitive.rs:55-72) over the survivors, until
//                     the next candidate cannot start before what the lane holds;
//                     writes the winner index per sample and the tile's
//                     hit-distance range (atomicMin/Max).
//   K3 cull_shadow    one warp per cull tile: shadow beam from that range, walk,
//                     append shadow candidate chunks {c, r*r, disc in the plane
//                     perpendicular to the light}; a leaf that occludes every shadow
//                     ray of the tile ends the walk (shadow_cover).
//   K4 shade_store    one warp per pixel tile: winner distance, normal, g, shadow
//                     origin (render.rs:194-199), disc pre-filter (warp rectangle,
//                     then per slot) + exact any-hit tests (render.rs:202-208),
//                     accumulation in reference sample order, RGBA8 quantisation,
//                     one framebuffer store per pixel (pair).
//
// Every pre-filter keeps a superset of what the exact test can accept (the worst-case
// f32 error of the discriminant is folded into the radii); the exact tests are the
// reference's operations one by one, so the bytes are the oracle's.  A cull tile whose
// candidates do not fit the pool (or whose shadow list passes RT_SHADOW_CAP) is flagged
// and its pixel tiles fall back to the per-lane walk (lane_traverse): the output never
// depends on the pool size.  Exactness argument: see rt_tile.cu and DESIGN.md section 4.
#include <type_traits>

#include "rt_pack.cuh"
#include "rt_kernels.h"

namespace rt {

static constexpr uint32_t NO_CHUNK = 0xffffffffu;
static constexpr uint32_t OVERFLOWED = 0xfffffffeu;
// Shadow chain of a cull tile whose shadow rays are ALL occluded by one leaf (shadow_cover, rt_cull.cuh: the exact
// any-hit test cannot miss it for any origin the tile can produce): no list, no tests -- K4 marks every shadow ray
// of the tile occluded (render.rs:208 reads only has_missed()).
static constexpr uint32_t COVERED = 0xfffffffdu;
// Shadow candidates per tile beyond which the per-lane any-hit walk is cheaper than the list (measured:
// level 10 tiles with 1,000-2,800 candidates; 384 sends too many supersampled tiles to the walk, 1536 too few).
#ifndef RT_SHADOW_CAP
#define RT_SHADOW_CAP 768
#endif
#ifndef RT_P_WARPS
#define RT_P_WARPS 4
#endif
static constexpr int P_WARPS = RT_P_WARPS;  // warps per block of the cull launches (independent warps)
// K2 / K4 are latency-bound: more resident warps win until the register cap spills.  Measured on C3 (4K, 4x4):
// 24 / 28 / 32 / 36 / 40 warps per SM = 80 / 72 / 64 / 56 / 48 registers: 1.57 / 1.44 / 1.38 / 1.35 / 1.37 ms with the
// round-1 kernels; with K4 no longer recomputing the hit distance 36 warps are 2.9 % (C3) / 3.9 % (C4) ahead of 32
// and neutral on the 1-spp frame.
#ifndef RT_PHASED_WARPS_PER_SM
#define RT_PHASED_WARPS_PER_SM 36
#endif
constexpr int phased_min_blocks(int warps_per_block) {
    return RT_PHASED_WARPS_PER_SM / warps_per_block > 0 ? RT_PHASED_WARPS_PER_SM / warps_per_block : 1;
}

struct CullShared {
    float4 cand4[T_CAND];
    float2 cand2[T_CAND];
    uint32_t stack[T_STACK];
    float key[T_CAND];  // primary flush: lower bound of a candidate's hit distance (front-to-back order)
};

// Geometry shared by the four phases.
template <int SPP, int PXW, int PXH, int CW, int CH>
struct Geo {
    static constexpr int NPX = PXW * PXH, NS = SPP * SPP, S = NPX * NS;
    static constexpr float FRAC = (float)(SPP - 1) / (float)SPP;  // largest sub-sample offset
    static constexpr int TW = 8 * PXW, TH = 4 * PXH;  // pixel tile (one warp)
    static constexpr int BW = TW * CW, BH = TH * CH;  // cull tile
    uint32_t ptiles_x, ptiles_y, ctiles_x, ctiles_y;
    __host__ __device__ Geo(uint32_t width, uint32_t rows) {
        ptiles_x = (width + TW - 1) / TW;
        ptiles_y = (rows + TH - 1) / TH;
        ctiles_x = (ptiles_x + CW - 1) / CW;
        ctiles_y = (ptiles_y + CH - 1) / CH;
    }
    __host__ __device__ uint32_t n_ptiles() const { return ptiles_x * ptiles_y; }
    __host__ __device__ uint32_t n_ctiles() const { return ctiles_x * ctiles_y; }
};

// Cone of a cull tile.
template <class G>
RT_DEV PrimaryBeam cull_tile_beam(const RenderParams &p, uint32_t ct_x, uint32_t ct_y) {
    const float frac = G::FRAC;
    const uint32_t x0 = ct_x * G::BW, j0 = ct_y * G::BH;
    const uint32_t xh = min(x0 + G::BW, p.width) - 1u, jh = min(j0 + G::BH, p.row_count) - 1u;
    const float ya = (float)(image_row(p, j0)), yb = (float)(image_row(p, jh));
    return make_primary_beam(p, (float)x0, (float)xh + frac, fminf(ya, yb), fmaxf(ya, yb) + frac);
}

// Conservative image-space bounds {x_lo, x_hi, y_lo, y_hi} (sample coordinates: pixel + sub-sample
// offset, image rows) of the primary rays whose EXACT f32 test against a candidate can pass.
// a = {v = c - eye, v.v}, rr = r*r.  A ray of raw direction (X, Y, Z) (render.rs:240-242) reaches the
// sphere only if its projection on the camera's xz-plane passes within R of (qx, qz):
// (qx Z - qz X)^2 <= R^2 (X^2 + Z^2), a quadratic in X/Z whose roots bound X; likewise Y.  R is the
// radius inflated by the worst-case rounding of the discriminant (cull_radius) plus the f32 error of the
// ray direction (< 5e-7 rad, at most 4e-6 at these distances).  Acceleration only: not parity arithmetic.
RT_DEV float4 screen_box(const RenderParams &p, float4 a, float rr) {
    float qx = a.x, qy = a.y, qz = a.z;
    if (p.has_basis) {  // camera coordinates (orthonormal basis: checked by the host before this variant runs)
        qx = fmaf(a.x, p.basis[0], fmaf(a.y, p.basis[1], a.z * p.basis[2]));
        qy = fmaf(a.x, p.basis[3], fmaf(a.y, p.basis[4], a.z * p.basis[5]));
        qz = fmaf(a.x, p.basis[6], fmaf(a.y, p.basis[7], a.z * p.basis[8]));
    }
    const float R = fmaf(asqrt(fmaf(EPS_DISC, a.w + rr, rr)), 1.001f, 1e-5f);
    if (!(qz > 1.01f * R)) return make_float4(-RT_INF, RT_INF, -RT_INF, RT_INF);  // not strictly in front: no bound
    const float A = fmaf(qz, qz, -R * R);
    const float k = adiv((float)p.width, A);
    const float cx = qx * qz * k, cy = qy * qz * k;
    const float hx = R * asqrt(fmaf(qx, qx, A)) * k, hy = R * asqrt(fmaf(qy, qy, A)) * k;
    const float sx = fmaf(hx, 1.0005f, fmaf(fabsf(cx), 1e-5f, 0.05f));
    const float sy = fmaf(hy, 1.0005f, fmaf(fabsf(cy), 1e-5f, 0.05f));
    const float hw = 0.5f * (float)p.width, hh = 0.5f * (float)p.height;
    // x_res = X + W/2 ; y_res = H/2 - Y (render.rs:240-241)
    return make_float4((cx - sx) + hw, (cx + sx) + hw, hh - (cy + sy), hh - (cy - sy));
}
RT_DEV bool box_overlaps(float4 box, float x0, float x1, float y0, float y1) {
    return box.y >= x0 && box.x <= x1 && box.w >= y0 && box.z <= y1;
}

// Warp-wide float min / max through the integer REDUX instruction: the map below is monotonic
// from float order (NaN-free inputs, +-inf included) to signed-int order and is its own inverse.
RT_DEV int f2ord(float f) {
    const int b = __float_as_int(f);
    return b ^ ((b >> 31) & 0x7fffffff);
}
RT_DEV float ord2f(int k) { return __int_as_float(k ^ ((k >> 31) & 0x7fffffff)); }
RT_DEV float warp_min_f(float f) { return ord2f(__reduce_min_sync(FULLMASK, f2ord(f))); }
RT_DEV float warp_max_f(float f) { return ord2f(__reduce_max_sync(FULLMASK, f2ord(f))); }

// Asynchronous staging of a chunk into shared memory (LDGSTS): the copy is in flight while the warp
// generates its rays; stage_wait() + __syncthreads() right before the first use.
RT_DEV void stage_async(uint4 *dst, const uint4 *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
RT_DEV void stage_wait() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }

static constexpr uint32_t PU = 4;  // 16-byte units per primary candidate record
static constexpr uint32_t SU = 3;  // 16-byte units per shadow candidate record

// Append the warp's candidate list to the pool as a chunk {count, next} + records, chained in
// front of `head`.  The exact-test operands are stored as broadcast PAIRS so that the packed f32x2
// tests of K2 / K4 (two rays per instruction) load them straight into register pairs:
//   primary (PU units): {vx,vx,vy,vy} {vz,vz,-v.v,-v.v} {r*r,r*r,index,0} {x_lo,x_hi,y_lo,y_hi}
//   shadow  (SU units): {cx,cx,cy,cy} {cz,cz,r*r,r*r} {c.e1, c.e2, R^2, 0}
// The last unit of each record is what the per-lane pre-filters read: the image-space box of the
// rays that can hit (screen_box), and the candidate's disc in the plane perpendicular to the light.
RT_DEV uint32_t flush_reserve(const RenderParams &p, int lane, uint32_t n, uint32_t rec_units, uint32_t head, bool &ok) {
    const uint32_t units = 1u + rec_units * n;
    // A reservation that starts past the capacity is handed back, so once the pool is exhausted the counter hovers
    // at pool_cap + (reservations in flight) and can never wrap past 2^32 and hand out units that alias live
    // chunks (pool_cap <= 2^26; the API allows 65535 x 65535 frames).  The comparison is 64-bit.  (Reading the
    // counter before adding would also stop the growth, but a load of the address every warp's atomics hit costs
    // a contended L2 round trip per flush: measured +24 % on a whole C2 frame.)
    uint32_t base = 0;
    if (lane == 0) {
        base = atomicAdd(p.pool_count, units);
        if (base > p.pool_cap) atomicSub(p.pool_count, units);
    }
    base = __shfl_sync(FULLMASK, base, 0);
    ok = (uint64_t)base + units <= (uint64_t)p.pool_cap;
    if (ok && lane == 0) p.pool[base] = make_uint4(n, head, 0u, 0u);
    return base;
}
RT_DEV uint32_t flush_primary(const RenderParams &p, CullShared &sm, int lane, uint32_t n, uint32_t head) {
    if (n == 0 || head == OVERFLOWED) return head;
    bool ok;
    const uint32_t base = flush_reserve(p, lane, n, PU, head, ok);
    if (!ok) return OVERFLOWED;
    // Records are written front to back by a lower bound of the distance the exact test can return.  With
    // disc_f32 <= disc + eps (eps = EPS_DISC (v.v + r*r), rt_cull.cuh) the f32 root b - sqrt(disc_f32) is smallest
    // head-on, where it is |v| - sqrt(r*r + eps): the inflated radius of the cull, not r (for the smallest leaves
    // the two differ by ~1e-3).  K2 stops a lane's candidate loop as soon as that bound exceeds the distances
    // the lane already holds.
    for (uint32_t c = lane; c < n; c += 32) {
        const float vv = sm.cand4[c].w, rr = sm.cand2[c].x;
        sm.key[c] = fmaf(asqrt(vv) - asqrt(fmaf(EPS_DISC, vv + rr, rr)), 0.99999f, -1e-5f);
    }
    __syncwarp();
    for (uint32_t c = lane; c < n; c += 32) {
        const float kc = sm.key[c];
        uint32_t rank = 0;
        for (uint32_t j = 0; j < n; j++) {
            const float kj = sm.key[j];
            rank += (kj < kc || (kj == kc && j < c)) ? 1u : 0u;
        }
        const float4 a = sm.cand4[c];
        const float2 e = sm.cand2[c];
        const uint32_t ax = __float_as_uint(a.x), ay = __float_as_uint(a.y), az = __float_as_uint(a.z);
        const uint32_t nvv = __float_as_uint(-a.w), rr = __float_as_uint(e.x);
        const float4 box = screen_box(p, a, e.x);
        uint4 *rec = p.pool + base + 1u + PU * rank;
        rec[0] = make_uint4(ax, ax, ay, ay);
        rec[1] = make_uint4(az, az, nvv, nvv);
        rec[2] = make_uint4(rr, rr, __float_as_uint(e.y), __float_as_uint(kc));
        rec[3] = make_uint4(__float_as_uint(box.x), __float_as_uint(box.y), __float_as_uint(box.z), __float_as_uint(box.w));
    }
    return base;
}
RT_DEV uint32_t flush_shadow(const RenderParams &p, const CullShared &sm, const ShadowBeam &B, int lane, uint32_t n, uint32_t head) {
    if (n == 0 || head == OVERFLOWED) return head;
    bool ok;
    const uint32_t base = flush_reserve(p, lane, n, SU, head, ok);
    if (!ok) return OVERFLOWED;
    for (uint32_t c = lane; c < n; c += 32) {
        const float4 a = sm.cand4[c];  // {c, r*r}
        const uint32_t ax = __float_as_uint(a.x), ay = __float_as_uint(a.y), az = __float_as_uint(a.z), rr = __float_as_uint(a.w);
        // |c - origin| <= |c - P0| + len + rho for every shadow origin of the tile (beam_test(ShadowBeam))
        const float qx = a.x - B.px, qy = a.y - B.py, qz = a.z - B.pz;
        const float vmax = asqrt(fmaf(qx, qx, fmaf(qy, qy, qz * qz))) + B.len + B.rho;
        // exact test passes => distance(c, shadow line) <= sqrt(rr + eps (vv + rr)); + 1e-5 for the f32
        // projections onto (e1, e2) here and in K4 (|o|, |c| < 16: < 3e-6 each)
        const float R = fmaf(asqrt(fmaf(EPS_DISC, fmaf(vmax, vmax, a.w), a.w)), 1.001f, 1e-5f);
        const float cu = fmaf(a.x, p.lframe[0], fmaf(a.y, p.lframe[1], a.z * p.lframe[2]));
        const float cv = fmaf(a.x, p.lframe[3], fmaf(a.y, p.lframe[4], a.z * p.lframe[5]));
        uint4 *rec = p.pool + base + 1u + SU * c;
        rec[0] = make_uint4(ax, ax, ay, ay);
        rec[1] = make_uint4(az, az, rr, rr);
        rec[2] = make_uint4(__float_as_uint(cu), __float_as_uint(cv), __float_as_uint(R * R), 0u);
    }
    return base;
}

// ---------------------------------------------------------------------------
// K1: primary cull, one warp per cull tile
// ---------------------------------------------------------------------------
// The primary cull can run on tiles K1C x K1C cull tiles large: the K1C x K1C cull tiles under one walk
// share its chain (each of their headers gets the same head).  Measured on B200: with 2 x 2 the 8K / 4x4
// frame (259,200 cull tiles) gains 3.5 % -- a quarter of the walks, each only a little longer -- while 4K
// frames lose 4-10 % (longer lists for K2 to filter, weaker occlusion pruning), so launch_phased picks
// K1C = 2 only above 150,000 cull tiles.  The shadow cull always keeps the small tiles: its beams need the
// tight depth range.
template <int SPP, int PXW, int PXH, int CW, int CH, int K1C>
__global__ void __launch_bounds__(32 * P_WARPS) phase_cull_primary(const RenderParams p) {
    using G = Geo<SPP, PXW, PXH, CW, CH>;                   // the cull tiles K2-K4 work on
    using GC = Geo<SPP, PXW, PXH, CW * K1C, CH * K1C>;      // the tiles this launch walks for
    __shared__ CullShared shared[P_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const G geo(p.width, p.row_count);
    const GC geoc(p.width, p.row_count);
    const uint32_t cc = blockIdx.x * P_WARPS + warp;
    if (cc >= geoc.n_ctiles()) return;
    CullShared &sm = shared[warp];
    const uint32_t ccx = cc % geoc.ctiles_x, ccy = cc / geoc.ctiles_x;
    const PrimaryBeam pb = cull_tile_beam<GC>(p, ccx, ccy);
    CullState cs;
    cull_begin<true>(p, sm, pb, lane, cs);
    uint32_t head = NO_CHUNK;
    bool done;
    do {
        done = cull_run<true>(p, sm, pb, lane, cs);
        head = flush_primary(p, sm, lane, cs.ncand, head);
        __syncwarp();
    } while (!done && head != OVERFLOWED);
    if (lane < K1C * K1C) {
        const uint32_t fx = ccx * K1C + (uint32_t)(lane % K1C), fy = ccy * K1C + (uint32_t)(lane / K1C);
        if (fx < geo.ctiles_x && fy < geo.ctiles_y) p.tile_hdr[fy * geo.ctiles_x + fx] = make_uint4(head, NO_CHUNK, 0x7f800000u, 0u);
    }
}

// ---------------------------------------------------------------------------
// K2: exact closest-hit tests, one warp per pixel tile
// ---------------------------------------------------------------------------
template <int SPP, int PXW, int PXH, int CW, int CH>
__global__ void __launch_bounds__(32 * CW * CH, phased_min_blocks(CW * CH)) phase_test_primary(const RenderParams p) {
    using G = Geo<SPP, PXW, PXH, CW, CH>;
    constexpr int S = G::S, NS = G::NS;
    __shared__ uint4 stage[1 + PU * T_CAND];  // the cull tile's first candidate chunk, shared by its pixel tiles
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const G geo(p.width, p.row_count);
    // one block per cull tile, one warp per pixel tile of it
    const uint32_t ct = blockIdx.y * geo.ctiles_x + blockIdx.x;  // 2-D grid of cull tiles: no division
    const uint32_t pt_x = blockIdx.x * CW + (uint32_t)(warp % CW), pt_y = blockIdx.y * CH + (uint32_t)(warp / CW);
    const uint32_t pt = pt_y * geo.ptiles_x + pt_x;
    const uint32_t tile_x0 = pt_x * G::TW, tile_j0 = pt_y * G::TH;
    const V3 eye = v3(p.eye[0], p.eye[1], p.eye[2]);
    const ONE2 one = f2s(p.one);  // 1.0f the compiler cannot see (rt_pack.cuh)
    // The winner's distance travels with its index: 8 bytes per sample.  At one sample per pixel they stay in L2; on
    // supersampled frames they stream through HBM (C3: 1.06 GB written here, read once by K4 -- 25 % of the HBM rate
    // over the two launches), which costs less than K4 recomputing the distance: measured -5.3 % on C3, -6.7 % on C4
    // against 4-byte winners.  The path is instruction-bound, not HBM-bound.
    uint2 *winner = reinterpret_cast<uint2 *>(p.winner) + (size_t)pt * S * 32;
    // streaming stores (and streaming loads in K4): the winners pass through L2 once and must not evict the scene and
    // the candidate chunks, which every tile re-reads (measured: -1.2 % on C3)
    auto put_winner = [&](int s, uint32_t idx, float dist) { __stcs(&winner[s * 32 + lane], make_uint2(idx, __float_as_uint(dist))); };

    uint32_t bx, bj;  // first pixel of this lane's block
    slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, 0, bx, bj);
    const bool lane_in = bx < p.width && bj < p.row_count;
    const uint32_t head = p.tile_hdr[ct].x;
    if (head == NO_CHUNK) return;  // no candidate at all: K4 sees an empty hit range and never reads the winners
    const bool staged = head != OVERFLOWED;
    if (staged) {  // stage the first chunk (almost always the only one) in shared memory, asynchronously
        const uint32_t units = 1u + PU * __ldg(&p.pool[head]).x;
        for (uint32_t u = threadIdx.x; u < units; u += blockDim.x) stage_async(&stage[u], &p.pool[head + u]);
    }
    if (pt_x >= geo.ptiles_x || pt_y >= geo.ptiles_y) {  // cull tile on the frame edge: only the block's barrier is left to do
        if (staged) {
            stage_wait();
            __syncthreads();
        }
        return;
    }
    auto fetch = [&](uint32_t base, uint32_t off) { return base == head ? stage[off] : __ldg(&p.pool[base + off]); };
    float tmin = RT_INF, tmax = 0.0f;

    if (head == OVERFLOWED) {  // pool exhausted for this cull tile: the per-lane walk (group.rs:72-83)
        for (int s = 0; s < S; s++) {
            uint32_t x, j;
            slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, s / NS, x, j);
            uint32_t bi = NO_HIT;
            float hitd = RT_INF;
            if (x < p.width && j < p.row_count) {
                const V3 d = slot_dir<SPP>(p, x, image_row(p, j), s % NS);
                lane_traverse<false>(p.sph, p.skip, p.n_nodes, eye, d, hitd, bi);
                if (hitd == RT_INF) bi = NO_HIT;
                else tmin = fminf(tmin, fabsf(hitd)), tmax = fmaxf(tmax, fabsf(hitd));
            }
            put_winner(s, bi, hitd);
        }
    } else {
        // Sample-coordinate rectangles of this lane's own block and of the warp's pixel tile: a
        // candidate whose screen_box misses the rectangle cannot be hit by any of its rays.
        constexpr float frac = G::FRAC;
        float lx0, lx1, ly0, ly1, wx0, wx1, wy0, wy1;
        {
            const uint32_t xh = min(bx + PXW, p.width) - 1u, jh = min(bj + PXH, p.row_count) - 1u;
            const float ya = (float)(image_row(p, bj)), yb = (float)(image_row(p, jh));
            lx0 = (float)bx, lx1 = (float)xh + frac, ly0 = fminf(ya, yb), ly1 = fmaxf(ya, yb) + frac;
        }
        {
            const uint32_t xh = min(tile_x0 + G::TW, p.width) - 1u, jh = min(tile_j0 + G::TH, p.row_count) - 1u;
            const float ya = (float)(image_row(p, tile_j0)), yb = (float)(image_row(p, jh));
            wx0 = (float)tile_x0, wx1 = (float)xh + frac, wy0 = fminf(ya, yb), wy1 = fmaxf(ya, yb) + frac;
        }
        // candidates c0..c1 (at most 32) of a chunk -> bit mask of those this LANE's block can see.
        // First every lane tests ONE candidate against the warp tile's rectangle (ballot), then each
        // lane tests the survivors against its own.
        auto cand_box = [&](uint32_t base, uint32_t c) {
            const uint4 u = fetch(base, 4u + PU * c);
            return make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w));
        };
        auto chunk_mask = [&](uint32_t base, uint32_t c0, uint32_t c1) {
            const bool w_ok = (c0 + lane < c1) && box_overlaps(cand_box(base, c0 + lane), wx0, wx1, wy0, wy1);
            uint32_t mask = 0;
            for (uint32_t wm = __ballot_sync(FULLMASK, w_ok); wm; wm &= wm - 1u) {
                const uint32_t c = c0 + (uint32_t)__ffs((int)wm) - 1u;
                if (box_overlaps(cand_box(base, c), lx0, lx1, ly0, ly1)) mask |= 1u << (c - c0);
            }
            return lane_in ? mask : 0u;
        };
        // One pass covers all of the lane's slots (S <= 4): the staged chunk is awaited after ray generation, so
        // the copy overlaps it.  With more passes the deferred barrier costs registers (spills under the 64-register
        // cap), so it is taken up front.
        constexpr bool LAZY = S <= 4;
        uint32_t mask0 = 0;  // mask of the first 32 candidates of the first chunk: reused by every slot pair
        if (!LAZY) {
            stage_wait();
            __syncthreads();
            mask0 = chunk_mask(head, 0u, min(stage[0].x, 32u));
        }
        // GP packed pairs (two slots each) per pass: every candidate record is loaded once for all of them and
        // the pairs' dependency chains interleave.
        constexpr int GP = (S >= 4) ? 2 : 1;
#pragma unroll 1
        for (int g0 = 0; g0 < S; g0 += 2 * GP) {
            V3x2 d[GP];
            F2 bd[GP];
            uint32_t bi[GP][2];
#pragma unroll
            for (int k = 0; k < GP; k++) {
                const int s0 = min(g0 + 2 * k, S - 1), s1 = min(s0 + 1, S - 1);  // a pair past the end repeats the last slot
                uint32_t x0, j0, x1, j1;
                slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, s0 / NS, x0, j0);
                slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, s1 / NS, x1, j1);
                d[k] = slot_dir2<SPP>(one, p, x0, image_row(p, j0), s0 % NS, x1, image_row(p, j1), s1 % NS);
                bd[k] = f2s(RT_INF);
                bi[k][0] = bi[k][1] = 0u;  // meaningful only once bd is finite (see `test`)
            }
            if (LAZY) {  // the only pass: every warp of the block arrives here exactly once
                stage_wait();
                __syncthreads();
                mask0 = chunk_mask(head, 0u, min(stage[0].x, 32u));
            }
            auto test = [&](const uint4 u0, const uint4 u1, const uint4 u2) {
                V3x2 v;
                v.x = f2(__uint_as_float(u0.x), __uint_as_float(u0.y));
                v.y = f2(__uint_as_float(u0.z), __uint_as_float(u0.w));
                v.z = f2(__uint_as_float(u1.x), __uint_as_float(u1.y));
                const F2 nvv = f2(__uint_as_float(u1.z), __uint_as_float(u1.w));
                const F2 rr = f2(__uint_as_float(u2.x), __uint_as_float(u2.y));
                const uint32_t idx = u2.z;
#pragma unroll
                for (int k = 0; k < GP; k++) {
                    const F2 dist = primary_distance2(one, v, nvv, rr, d[k]);
                    // primitive.rs:79 + pre-order visiting: strictly closer wins, ties -> lowest index.  Distances are
                    // never negative (a root below zero is a miss, and -0 cannot arise: r*r > 0 keeps the discriminant
                    // off -0), so their bit patterns order like the values and {distance, index} compares as ONE
                    // unsigned 64-bit key.  A miss is +inf: it never beats the initial {+inf, 0}.
                    const unsigned long long k0 = ((unsigned long long)__float_as_uint(dist.x) << 32) | idx;
                    const unsigned long long k1 = ((unsigned long long)__float_as_uint(dist.y) << 32) | idx;
                    if (k0 < (((unsigned long long)__float_as_uint(bd[k].x) << 32) | bi[k][0])) bd[k].x = dist.x, bi[k][0] = idx;
                    if (k1 < (((unsigned long long)__float_as_uint(bd[k].y) << 32) | bi[k][1])) bd[k].y = dist.y, bi[k][1] = idx;
                }
            };
            // farthest distance the lane still has to beat (+inf while one of its slots has no hit)
            auto held = [&]() {
                float h = fmaxf(bd[0].x, bd[0].y);
#pragma unroll
                for (int k = 1; k < GP; k++) h = fmaxf(h, fmaxf(bd[k].x, bd[k].y));
                return h;
            };
            // hot path: the first 32 candidates of the staged chunk, straight from shared memory; they come
            // front to back, so the lane is done once a candidate cannot start before what it holds
            for (uint32_t m = mask0; m; m &= m - 1u) {
                const uint32_t c = (uint32_t)__ffs((int)m) - 1u;
                const uint4 u2 = stage[3u + PU * c];
                if (__uint_as_float(u2.w) > held()) break;
                test(stage[1u + PU * c], stage[2u + PU * c], u2);
            }
            // cold path: the rest of the staged chunk and any further chunks of the chain
            for (uint32_t base = head; base != NO_CHUNK;) {
                const uint4 hdr = fetch(base, 0u);
                const uint32_t n = hdr.x;
                for (uint32_t c0 = (base == head) ? 32u : 0u; c0 < n; c0 += 32) {
                    for (uint32_t m = chunk_mask(base, c0, min(n, c0 + 32u)); m; m &= m - 1u) {
                        const uint32_t c = c0 + (uint32_t)__ffs((int)m) - 1u;
                        const uint4 u2 = fetch(base, 3u + PU * c);
                        if (__uint_as_float(u2.w) > held()) break;  // each chunk is sorted front to back
                        test(fetch(base, 1u + PU * c), fetch(base, 2u + PU * c), u2);
                    }
                }
                base = hdr.y;
            }
#pragma unroll
            for (int k = 0; k < GP; k++) {
                const int s0 = g0 + 2 * k, s1 = s0 + 1;
                if (s0 < S) {
                    const bool hit = bd[k].x != RT_INF;
                    put_winner(s0, hit ? bi[k][0] : NO_HIT, bd[k].x);
                    if (hit) tmin = fminf(tmin, bd[k].x), tmax = fmaxf(tmax, bd[k].x);
                }
                if (s1 < S) {
                    const bool hit = bd[k].y != RT_INF;
                    put_winner(s1, hit ? bi[k][1] : NO_HIT, bd[k].y);
                    if (hit) tmin = fminf(tmin, bd[k].y), tmax = fmaxf(tmax, bd[k].y);
                }
            }
        }
    }
    // hit-distance range of the cull tile (positive floats order as uints)
    const uint32_t lo = __reduce_min_sync(FULLMASK, __float_as_uint(tmin));
    const uint32_t hi = __reduce_max_sync(FULLMASK, __float_as_uint(tmax));
    if (lane == 0 && lo != 0x7f800000u) {
        uint32_t *h = reinterpret_cast<uint32_t *>(&p.tile_hdr[ct]);
        atomicMin(h + 2, lo);
        atomicMax(h + 3, hi);
    }
}

// ---------------------------------------------------------------------------
// K3: shadow cull, one warp per cull tile
// ---------------------------------------------------------------------------
template <int SPP, int PXW, int PXH, int CW, int CH>
__global__ void __launch_bounds__(32 * P_WARPS) phase_cull_shadow(const RenderParams p) {
    using G = Geo<SPP, PXW, PXH, CW, CH>;
    __shared__ CullShared shared[P_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const G geo(p.width, p.row_count);
    const uint32_t ct = blockIdx.x * P_WARPS + warp;
    if (ct >= geo.n_ctiles()) return;
    CullShared &sm = shared[warp];
    const uint4 hdr = p.tile_hdr[ct];
    if (hdr.z == 0x7f800000u || hdr.x == OVERFLOWED) {  // no hit in this tile / tile handled by the per-lane walk
        if (lane == 0) reinterpret_cast<uint32_t *>(&p.tile_hdr[ct])[1] = hdr.x == OVERFLOWED ? OVERFLOWED : NO_CHUNK;
        return;
    }
    const PrimaryBeam pb = cull_tile_beam<G>(p, ct % geo.ctiles_x, ct / geo.ctiles_x);
    const V3 eye = v3(p.eye[0], p.eye[1], p.eye[2]);
    ShadowBeam sb;
    {
        const float tlo = __uint_as_float(hdr.z), thi = __uint_as_float(hdr.w);
        const float off = thi * 3.6e-4f + 1e-6f;  // |normal * distance * sqrt(eps)| <= distance * 3.4527e-4
        float a0 = adiv(tlo, pb.secp) * 0.99999f - off;
        float a1 = thi + off;
        if (pb.wide) {  // no usable cone: origins anywhere within thi of the eye
            a0 = 0.0f;
            a1 = 0.0f;
            sb.rho = thi * 1.001f + off;
        } else {
            sb.rho = thi * (pb.tanp + 3.6e-4f) * 1.001f + 1e-6f;
        }
        sb.none = false;
        sb.px = fmaf(a0, pb.ax, eye.x), sb.py = fmaf(a0, pb.ay, eye.y), sb.pz = fmaf(a0, pb.az, eye.z);
        sb.ax = pb.ax, sb.ay = pb.ay, sb.az = pb.az;
        sb.lx = -p.light[0], sb.ly = -p.light[1], sb.lz = -p.light[2];  // render.rs:206
        sb.len = a1 - a0;
        float nx = sb.ay * sb.lz - sb.az * sb.ly, ny = sb.az * sb.lx - sb.ax * sb.lz, nz = sb.ax * sb.ly - sb.ay * sb.lx;
        float sn = asqrt(nx * nx + ny * ny + nz * nz);
        sb.degenerate = pb.wide || !(sn > 0.05f);
        float isn = adiv(1.0f, fmaxf(sn, 1e-20f));
        sb.nx = nx * isn, sb.ny = ny * isn, sb.nz = nz * isn;
        sb.cosq = sb.ax * sb.lx + sb.ay * sb.ly + sb.az * sb.lz;
        sb.inv_sin = isn * 1.00001f;
        sb.inv_sin2 = isn * isn * 1.00001f;
        sb.rmin = p.leaf_rmin;
    }
    CullState cs;
    cull_begin<false>(p, sm, sb, lane, cs);
    uint32_t head = NO_CHUNK;
    bool done;
    uint32_t total = 0;
    do {
        done = cull_run<false>(p, sm, sb, lane, cs);
        total += cs.ncand;
        if (cs.covered) {  // one leaf settles every shadow ray of the tile: whatever was listed before is moot
            head = COVERED;
            break;
        }
        // Past a few hundred candidates the list costs more than the per-lane any-hit walk (measured at level 10:
        // tiles with 1,000-2,800 candidates); such a tile is handed to that walk, as on pool exhaustion.
        if (total > (uint32_t)RT_SHADOW_CAP) head = OVERFLOWED;
        head = flush_shadow(p, sm, sb, lane, cs.ncand, head);
        __syncwarp();
    } while (!done && head != OVERFLOWED);
    if (lane == 0) reinterpret_cast<uint32_t *>(&p.tile_hdr[ct])[1] = head;
}

// ---------------------------------------------------------------------------
// K4: shading, shadow tests, accumulation, store; one warp per pixel tile
// ---------------------------------------------------------------------------
// F32: each pixel is stored as the float4 {r, g, b, alpha} that RGBA8 output quantises (16 bytes at x * 16 of its
// row) instead of those four bytes.  Everything before the store is the same code.  `tid` is threadIdx.x read in the
// __global__ function, where the compiler knows its range from the launch bounds (render_body, rt_kernels.cu).
template <int SPP, int PXW, int PXH, int CW, int CH, bool DIAG, bool F32>
__device__ __forceinline__ void shade_store_body(const RenderParams &p, const uint32_t tid) {
    using G = Geo<SPP, PXW, PXH, CW, CH>;
    constexpr int S = G::S, NS = G::NS;
    __shared__ uint4 stage[1 + SU * T_CAND];  // the cull tile's first shadow-candidate chunk
    const int lane = tid & 31, warp = tid >> 5;
    const G geo(p.width, p.row_count);
    // one block per cull tile, one warp per pixel tile of it
    const uint32_t ct = blockIdx.y * geo.ctiles_x + blockIdx.x;  // 2-D grid of cull tiles: no division
    const uint32_t pt_x = blockIdx.x * CW + (uint32_t)(warp % CW), pt_y = blockIdx.y * CH + (uint32_t)(warp / CW);
    const uint32_t pt = pt_y * geo.ptiles_x + pt_x;
    const uint32_t tile_x0 = pt_x * G::TW, tile_j0 = pt_y * G::TH;
    const uint2 *winner = reinterpret_cast<const uint2 *>(p.winner) + (size_t)pt * S * 32;  // {leaf index, hit distance} per slot (K2)
    const ONE2 one = f2s(p.one);  // 1.0f the compiler cannot see (rt_pack.cuh)

    const V3 eye = v3(p.eye[0], p.eye[1], p.eye[2]);
    const V3 light = v3(p.light[0], p.light[1], p.light[2]);
    const V3 to_light = vmulf(light, -1.0f);  // render.rs:206
    // render.rs:172-186, :199 -- constants folded at compile time in IEEE f32
    constexpr float OBJ_R = 174.0f / 255.0f, OBJ_G = 49.0f / 255.0f, BG_R = 34.0f / 255.0f, BG_G = 10.0f / 255.0f;
    const float AMB_R = fmul(BG_R, 0.8f), AMB_G = fmul(BG_G, 0.8f);  // render.rs:181-186
    const bool pair_aligned = ((reinterpret_cast<uintptr_t>(p.out) | p.pitch) & 7u) == 0;
    const float sqrt_eps = __uint_as_float(0x39b504f3u);       // sqrt(f32::EPSILON) = 3.4526698e-4
    const float recip = frecip(fmul((float)SPP, (float)SPP));  // render.rs:219-220

    uint32_t bx, bj;
    slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, 0, bx, bj);
    const bool lane_in = bx < p.width && bj < p.row_count;
    const uint4 tile_hdr = p.tile_hdr[ct];
    const uint32_t head = tile_hdr.y;
    constexpr bool LAZY = S <= 4;  // one group per lane: await the staged chunk after phase A (see K2)
    const bool staged = head < COVERED;
    if (staged) {  // stage the first chunk (almost always the only one) in shared memory, asynchronously
        const uint32_t units = 1u + SU * __ldg(&p.pool[head]).x;
        for (uint32_t u = tid; u < units; u += blockDim.x) {
            if (LAZY) stage_async(&stage[u], &p.pool[head + u]);
            else stage[u] = __ldg(&p.pool[head + u]);
        }
    }
    if (!LAZY) __syncthreads();
    if (pt_x >= geo.ptiles_x || pt_y >= geo.ptiles_y) {  // cull tile on the frame edge: only the block's barrier is left to do
        if (LAZY && staged) {
            stage_wait();
            __syncthreads();
        }
        return;
    }
    unsigned n_hits = 0, n_shadow = 0;
    float cr = 0.0f, cg = 0.0f, alpha = 0.0f;  // red, green (= blue), alpha of the pixel being accumulated (render.rs:233-234)
    if (tile_hdr.z == 0x7f800000u) {
        // no ray of this cull tile hit anything: every sample adds BACKGROUND (render.rs:190-193)
        if (lane_in) {
            for (int smp = 0; smp < NS; smp++) cr = fadd(cr, BG_R), cg = fadd(cg, BG_G);
            if constexpr (F32) {
                const float4 v = make_float4(fmul(cr, recip), fmul(cg, recip), fmul(cg, recip), fmul(0.0f, recip));
                for (int pi = 0; pi < G::NPX; pi++) {
                    uint32_t x, j;
                    slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, pi, x, j);
                    if (x < p.width && j < p.row_count)
                        *reinterpret_cast<float4 *>(p.out + (size_t)out_row(p, j) * p.pitch + (size_t)x * 16) = v;
                }
                return;
            }
            const uint32_t g8 = scale_u8_fast(fmul(cg, recip));
            const uint32_t px = scale_u8_fast(fmul(cr, recip)) | (g8 << 8) | (g8 << 16) | (scale_u8_fast(fmul(0.0f, recip)) << 24);
            for (int pi = 0; pi < G::NPX; pi++) {
                uint32_t x, j;
                slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, pi, x, j);
                if (x < p.width && j < p.row_count) {
                    *reinterpret_cast<uint32_t *>(p.out + (size_t)out_row(p, j) * p.pitch + (size_t)x * 4) = px;
                    if (DIAG && p.kinds)
                        for (int smp = 0; smp < NS; smp++) p.kinds[((size_t)j * p.width + x) * NS + smp] = K_BACKGROUND;
                }
            }
        }
    } else {
        // Every lane takes part (warp-wide ballots below); lanes outside the frame have no hits and store nothing.
        const V3x2 eye2 = v3x2s(eye), light2 = v3x2s(light), to_light2 = v3x2s(to_light);
        constexpr int GS = 4;  // slots per group: two packed pairs share one candidate pre-filter pass
#pragma unroll 1
        for (int g0 = 0; g0 < S; g0 += GS) {
#ifndef RT_K4_NO_PREFETCH
            // the next group's winners: in L1 by the time phase A of that group loads them (measured: -1 % on 4x4 frames)
            if (S > GS && g0 + GS < S) {
#pragma unroll
                for (int i = 0; i < GS; i++)
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(winner + (size_t)(g0 + GS + i) * 32 + lane));
            }
#endif
            // ---- A: hit point, normal, g and shadow origin of the group's slots (render.rs:188-199) ----
            V3x2 no[2];           // minus the shadow origins, per pair
            // Minus the shadow origins' coordinates (u, v) in the plane perpendicular to the light.  Supersampled frames keep them
            // per pair, packed over the pair's two slots (nu, nv: 6 packed instructions per pair instead of 12 scalar ones,
            // and the pre-filter measures both slots of a pair at once: C3 -3.2 %); the one-sample-per-pixel kernels keep one
            // (u, v) pair per slot (nuv) -- there the packed form measured 1 % slower.
            constexpr bool UV_PER_SLOT = NS == 1;
            F2 nuv[2][2], nu[2], nv[2];
            float g[GS];          // g = normal . light; +inf = no hit
            uint32_t pend = 0, occluded = 0;  // bit 2k+i: slot i of pair k still needs / has found an occluder
            uint32_t xs[GS], js[GS];
#pragma unroll
            for (int k = 0; k < 2; k++) {
                const int s0 = g0 + 2 * k, s1 = (s0 + 1 < S) ? s0 + 1 : s0;
                if (s0 < S) {
                    slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, s0 / NS, xs[2 * k], js[2 * k]);
                    slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, s1 / NS, xs[2 * k + 1], js[2 * k + 1]);
                    const V3x2 d = slot_dir2<SPP>(one, p, xs[2 * k], image_row(p, js[2 * k]), s0 % NS, xs[2 * k + 1],
                                                  image_row(p, js[2 * k + 1]), s1 % NS);
                    const uint2 a = __ldcs(&winner[s0 * 32 + lane]), b = __ldcs(&winner[s1 * 32 + lane]);  // read once: streaming
                    const uint32_t wi0 = a.x, wi1 = b.x;
                    F2 dist = f2(__uint_as_float(a.y), __uint_as_float(b.y));  // primitive.rs:55-72, as K2 computed it
                    const bool hit0 = wi0 != NO_HIT, hit1 = wi1 != NO_HIT;
                    const float4 w0 = __ldg(&p.sph[hit0 ? wi0 : 0u]), w1 = __ldg(&p.sph[hit1 ? wi1 : 0u]);
                    const V3x2 cen = V3x2{f2(w0.x, w1.x), f2(w0.y, w1.y), f2(w0.z, w1.z)};
                    if (!hit0) dist.x = 1.0f;
                    if (!hit1) dist.y = 1.0f;
                    // primitive.rs:83 normal; render.rs:194 g; render.rs:199 shadow origin
                    const V3x2 nrm = vnormalized2<(NS > 1)>(one, vadd2(one, eye2, vsub2(one, vmulf2(d, dist), cen)));
                    const F2 gg = vdot2(one, nrm, light2);
                    const V3x2 o = vadd2(one, vadd2(one, eye2, vmulf2(d, dist)), vmulf2(nrm, f2mul(dist, f2s(sqrt_eps))));
                    no[k] = V3x2{f2neg(o.x), f2neg(o.y), f2neg(o.z)};
                    if constexpr (UV_PER_SLOT) {
                        // -(o . e1, o . e2) per slot, computed straight into the pair the pre-filter adds to a candidate
                        nuv[k][0] = f2(fmaf(no[k].x.x, p.lframe[0], fmaf(no[k].y.x, p.lframe[1], no[k].z.x * p.lframe[2])),
                                       fmaf(no[k].x.x, p.lframe[3], fmaf(no[k].y.x, p.lframe[4], no[k].z.x * p.lframe[5])));
                        nuv[k][1] = f2(fmaf(no[k].x.y, p.lframe[0], fmaf(no[k].y.y, p.lframe[1], no[k].z.y * p.lframe[2])),
                                       fmaf(no[k].x.y, p.lframe[3], fmaf(no[k].y.y, p.lframe[4], no[k].z.y * p.lframe[5])));
                    } else {
                        // -(o . e1) and -(o . e2) of the pair's two slots at once (pre-filter only, not parity arithmetic: FMA is fine)
                        nu[k] = f2fma(no[k].x, f2s(p.lframe[0]), f2fma(no[k].y, f2s(p.lframe[1]), f2mul(no[k].z, f2s(p.lframe[2]))));
                        nv[k] = f2fma(no[k].x, f2s(p.lframe[3]), f2fma(no[k].y, f2s(p.lframe[4]), f2mul(no[k].z, f2s(p.lframe[5]))));
                    }
                    g[2 * k] = hit0 ? gg.x : RT_INF;
                    g[2 * k + 1] = hit1 ? gg.y : RT_INF;
                    if (hit0 && !(gg.x >= 0.0f)) pend |= 1u << (2 * k);
                    if (hit1 && !(gg.y >= 0.0f) && s1 != s0) pend |= 2u << (2 * k);
                } else {
                    no[k] = V3x2{f2s(0.0f), f2s(0.0f), f2s(0.0f)};
                    nuv[k][0] = nuv[k][1] = nu[k] = nv[k] = f2s(0.0f);
                    g[2 * k] = g[2 * k + 1] = RT_INF;
                    xs[2 * k] = xs[2 * k + 1] = js[2 * k] = js[2 * k + 1] = 0xffffffffu;
                }
            }
            if (LAZY && staged) {  // the only group: every warp of the block arrives here exactly once
                stage_wait();
                __syncthreads();
            }
            // ---- B: shadow rays {pos: o, dir: -light} against the tile's candidates (render.rs:202-208) ----
            if (head == COVERED) {  // every shadow ray of this cull tile is occluded (shadow_cover): nothing to test
                occluded = pend;
                pend = 0;
            }
            if (head == OVERFLOWED) {  // per-lane walk, any-hit
#pragma unroll
                for (int i = 0; i < GS; i++) {
                    if ((pend >> i) & 1u) {
                        float sh = RT_INF;
                        uint32_t dummy = 0;
                        const V3x2 o = V3x2{f2neg(no[i >> 1].x), f2neg(no[i >> 1].y), f2neg(no[i >> 1].z)};
                        lane_traverse<true>(p.sph, p.skip, p.n_nodes, (i & 1) ? hi(o) : lo(o), to_light, sh, dummy);
                        if (sh != RT_INF) occluded |= 1u << i;
                    }
                }
                pend = 0;
            }
            // exact any-hit test of pair k against one candidate (primitive.rs:56-68)
            auto shadow_test = [&](const int k, const uint4 u0, const uint4 u1) {
                V3x2 cc;
                cc.x = f2(__uint_as_float(u0.x), __uint_as_float(u0.y));
                cc.y = f2(__uint_as_float(u0.z), __uint_as_float(u0.w));
                cc.z = f2(__uint_as_float(u1.x), __uint_as_float(u1.y));
                const F2 rr = f2(__uint_as_float(u1.z), __uint_as_float(u1.w));
                const V3x2 sv = vadd2(one, cc, no[k]);  // center - ray.pos
                const F2 b = vdot2(one, sv, to_light2);
                const F2 disc = f2add(one, f2sub(one, f2mul(b, b), vdot2(one, sv, sv)), rr);
                // finite iff disc >= 0 and !(b + sqrt(disc) < 0) (primitive.rs:60-68); b >= 0 settles the latter
                bool f0 = !(disc.x < 0.0f), f1 = !(disc.y < 0.0f);
                if ((f0 && b.x < 0.0f) || (f1 && b.y < 0.0f)) {
                    const F2 t2 = f2add(one, b, fsqrt_nr2(disc));
                    f0 = f0 && !(t2.x < 0.0f);
                    f1 = f1 && !(t2.y < 0.0f);
                }
                const uint32_t f = (((f0 ? 1u : 0u) | (f1 ? 2u : 0u)) << (2 * k)) & pend;
                pend &= ~f;
                occluded |= f;
            };
            if (__ballot_sync(FULLMASK, pend != 0u) != 0u && head < COVERED) {
                // Rectangle of the warp's pending shadow origins in the plane perpendicular to the light.
                float ulo = RT_INF, uhi = -RT_INF, vlo = RT_INF, vhi = -RT_INF;
#pragma unroll
                for (int i = 0; i < GS; i++) {
                    if ((pend >> i) & 1u) {
                        const F2 q = UV_PER_SLOT ? nuv[i >> 1][i & 1] : (i & 1) ? f2(nu[i >> 1].y, nv[i >> 1].y) : f2(nu[i >> 1].x, nv[i >> 1].x);
                        ulo = fminf(ulo, -q.x), uhi = fmaxf(uhi, -q.x), vlo = fminf(vlo, -q.y), vhi = fmaxf(vhi, -q.y);
                    }
                }
                ulo = warp_min_f(ulo), uhi = warp_max_f(uhi), vlo = warp_min_f(vlo), vhi = warp_max_f(vhi);
                // one chunk of the tile's chain: STAGED = the first one, read from shared memory
                auto run_chunk = [&](auto staged_tag, uint32_t base) -> uint32_t {
                    constexpr bool STAGED = decltype(staged_tag)::value;
                    auto unit = [&](uint32_t off) { return STAGED ? stage[off] : __ldg(&p.pool[base + off]); };
                    const uint4 hdr = unit(0u);
                    for (uint32_t c0 = 0; c0 < hdr.x; c0 += 32) {
                        // warp level: lane tests candidate c0 + lane (disc vs rectangle)
                        bool w_ok = false;
                        if (c0 + lane < hdr.x) {
                            const uint4 u = unit(3u + SU * (c0 + lane));
                            const float cu = __uint_as_float(u.x), cv = __uint_as_float(u.y);
                            const float du = fmaxf(fmaxf(ulo - cu, cu - uhi), 0.0f), dv = fmaxf(fmaxf(vlo - cv, cv - vhi), 0.0f);
                            w_ok = du * du + dv * dv <= __uint_as_float(u.z);
                        }
                        // lane level: the survivors against each pending slot (packed over the two plane coordinates)
                        uint32_t m0 = 0, m1 = 0;
                        for (uint32_t wm = __ballot_sync(FULLMASK, w_ok); wm; wm &= wm - 1u) {
                            const uint32_t b = (uint32_t)__ffs((int)wm) - 1u;
                            const uint4 u = unit(3u + SU * (c0 + b));
                            const float r2 = __uint_as_float(u.z);
                            bool h0, h1;
                            if constexpr (UV_PER_SLOT) {
                                const F2 cuv = f2(__uint_as_float(u.x), __uint_as_float(u.y));
                                const F2 d00 = __fadd2_rn(cuv, nuv[0][0]), d01 = __fadd2_rn(cuv, nuv[0][1]);
                                const F2 d10 = __fadd2_rn(cuv, nuv[1][0]), d11 = __fadd2_rn(cuv, nuv[1][1]);
                                const F2 q00 = f2mul(d00, d00), q01 = f2mul(d01, d01), q10 = f2mul(d10, d10), q11 = f2mul(d11, d11);
                                h0 = ((pend & 1u) && q00.x + q00.y <= r2) || ((pend & 2u) && q01.x + q01.y <= r2);
                                h1 = ((pend & 4u) && q10.x + q10.y <= r2) || ((pend & 8u) && q11.x + q11.y <= r2);
                            } else {
                                // squared distance from the candidate's centre to both slots of a pair at once
                                const F2 cu = f2s(__uint_as_float(u.x)), cv = f2s(__uint_as_float(u.y));
                                const F2 du0 = __fadd2_rn(cu, nu[0]), dv0 = __fadd2_rn(cv, nv[0]);
                                const F2 du1 = __fadd2_rn(cu, nu[1]), dv1 = __fadd2_rn(cv, nv[1]);
                                const F2 q0 = f2fma(dv0, dv0, f2mul(du0, du0)), q1 = f2fma(dv1, dv1, f2mul(du1, du1));
                                h0 = ((pend & 1u) && q0.x <= r2) || ((pend & 2u) && q0.y <= r2);
                                h1 = ((pend & 4u) && q1.x <= r2) || ((pend & 8u) && q1.y <= r2);
                            }
                            if (h0) m0 |= 1u << b;
                            if (h1) m1 |= 1u << b;
                        }
                        // exact tests of the survivors (both pairs per candidate: one record load, two
                        // independent dependency chains)
                        if (!(pend & 3u)) m0 = 0;
                        if (!(pend & 12u)) m1 = 0;
                        for (uint32_t m = m0 | m1; m && pend; m &= m - 1u) {
                            const uint32_t c = c0 + (uint32_t)__ffs((int)m) - 1u;
                            const uint4 u0 = unit(1u + SU * c), u1 = unit(2u + SU * c);
                            shadow_test(0, u0, u1);
                            shadow_test(1, u0, u1);
                        }
                    }
                    return hdr.y;
                };
                uint32_t next = run_chunk(std::true_type{}, head);
                while (next != NO_CHUNK && __ballot_sync(FULLMASK, pend != 0u) != 0u) next = run_chunk(std::false_type{}, next);
            }
            // ---- C: accumulate in reference sample order (render.rs:236-250), quantise, store (render.rs:92-109) ----
            // Only red and green are carried: OBJECT, BACKGROUND and AMBIENT_OFFSET have g == b (render.rs:172-186)
            // and both channels go through the same operations, so blue equals green bit for bit.
            uint32_t px[GS];
            bool px_ok[GS];
#pragma unroll
            for (int i = 0; i < GS; i++) {
                const int s = g0 + i;
                px[i] = 0u, px_ok[i] = false;
                if (s < S) {
                    const int smp = s % NS;
                    const uint32_t x = xs[i], j = js[i];
                    const bool inside = x < p.width && j < p.row_count;
                    if (smp == 0) cr = 0.0f, cg = 0.0f, alpha = 0.0f;
                    uint8_t kind;
                    if (g[i] == RT_INF) {  // render.rs:190-193
                        cr = fadd(cr, BG_R), cg = fadd(cg, BG_G);
                        kind = K_BACKGROUND;
                    } else if (g[i] >= 0.0f) {  // render.rs:195-198
                        cr = fadd(cr, AMB_R), cg = fadd(cg, AMB_G);
                        kind = K_AWAY;
                        if (DIAG && inside) n_hits++;
                    } else {
                        if (DIAG && inside) n_hits++, n_shadow++;
                        const float ng = -g[i];
                        if (!((occluded >> i) & 1u)) {  // render.rs:208-210
                            cr = fadd(fadd(cr, fmul(OBJ_R, ng)), AMB_R), cg = fadd(fadd(cg, fmul(OBJ_G, ng)), AMB_G);
                            alpha = fadd(alpha, 1.0f);
                            kind = K_LIT;
                        } else {  // render.rs:211-214
                            cr = fadd(fadd(cr, BG_R), fmul(AMB_R, ng)), cg = fadd(fadd(cg, BG_G), fmul(AMB_G, ng));
                            kind = K_SHADOWED;
                        }
                    }
                    if (DIAG && p.kinds && inside) p.kinds[((size_t)j * p.width + x) * NS + smp] = kind;
                    if (smp == NS - 1) {
                        // render.rs:249-250: * 1/(spp*spp); for one sample that factor is exactly 1.0f and x * 1 == x
                        const float qr = NS == 1 ? cr : fmul(cr, recip), qg = NS == 1 ? cg : fmul(cg, recip);
                        const float al = NS == 1 ? alpha : fmul(alpha, recip);
                        // Floats are stored as the pixel completes (a pair of them would be two 16-byte stores anyway);
                        // px_ok stays false, so the RGBA8 stores below store nothing.
                        if constexpr (F32) {
                            if (inside)
                                *reinterpret_cast<float4 *>(p.out + (size_t)out_row(p, j) * p.pitch + (size_t)x * 16) =
                                    make_float4(qr, qg, qg, al);
                            continue;
                        }
                        const uint32_t g8 = scale_u8_fast(qg);
                        // one sample: alpha is exactly 0 or 1, and trunc(0.5 + 255 * 1) = 255
                        const uint32_t a8 = NS == 1 ? (al != 0.0f ? 255u : 0u) : scale_u8_fast(al);
                        px[i] = scale_u8_fast(qr) | (g8 << 8) | (g8 << 16) | (a8 << 24);
                        px_ok[i] = inside;
                    }
                }
            }
            if (NS == 1 && PXW == 2) {
                // slots 2k, 2k+1 are horizontal neighbours (slot_pixel): one 8-byte store per pair
#pragma unroll
                for (int i = 0; i < GS; i += 2) {
                    uint8_t *at = p.out + (size_t)out_row(p, js[i]) * p.pitch + (size_t)xs[i] * 4;
                    if (px_ok[i] && px_ok[i + 1] && pair_aligned) {
                        *reinterpret_cast<uint2 *>(at) = make_uint2(px[i], px[i + 1]);
                    } else {
                        if (px_ok[i]) *reinterpret_cast<uint32_t *>(at) = px[i];
                        if (px_ok[i + 1]) *reinterpret_cast<uint32_t *>(at + 4) = px[i + 1];
                    }
                }
            } else {
#pragma unroll
                for (int i = 0; i < GS; i++)
                    if (px_ok[i]) *reinterpret_cast<uint32_t *>(p.out + (size_t)out_row(p, js[i]) * p.pitch + (size_t)xs[i] * 4) = px[i];
            }
        }
    }
    if (DIAG && p.ray_counters) {
        n_hits = __reduce_add_sync(FULLMASK, n_hits);
        n_shadow = __reduce_add_sync(FULLMASK, n_shadow);
        if (lane == 0) {
            atomicAdd(&p.ray_counters[0], (unsigned long long)n_hits);
            atomicAdd(&p.ray_counters[1], (unsigned long long)n_shadow);
        }
    }
}

template <int SPP, int PXW, int PXH, int CW, int CH, bool DIAG>
__global__ void __launch_bounds__(32 * CW * CH, phased_min_blocks(CW * CH)) phase_shade_store(const RenderParams p) {
    shade_store_body<SPP, PXW, PXH, CW, CH, DIAG, false>(p, threadIdx.x);
}

template <int SPP, int PXW, int PXH, int CW, int CH>
__global__ void __launch_bounds__(32 * CW * CH, phased_min_blocks(CW * CH)) phase_shade_store_f32(const RenderParams p) {
    shade_store_body<SPP, PXW, PXH, CW, CH, false, true>(p, threadIdx.x);
}

// ---------------------------------------------------------------------------
// AOV store: the geometry of K2's winners, in place of K3 + K4; one warp per pixel tile
// ---------------------------------------------------------------------------
// Per pixel, over the samples that hit (reference sample order): the sum of the unit normals and the hit count,
// both times 1/(spp*spp), and the nearest hit's distance and point (the first sample wins a tie).  Stored as two
// float4 {nx, ny, nz, coverage} {distance, px, py, pz} at x * 32 of the pixel's row.  The normal and the hit point
// are phase A of K4 (render.rs:194, :199 first term), so the normal is the one K4 shades with.
template <int SPP, int PXW, int PXH, int CW, int CH>
__global__ void __launch_bounds__(32 * CW * CH, phased_min_blocks(CW * CH)) phase_aov_store(const RenderParams p) {
    using G = Geo<SPP, PXW, PXH, CW, CH>;
    constexpr int S = G::S, NS = G::NS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const G geo(p.width, p.row_count);
    const uint32_t ct = blockIdx.y * geo.ctiles_x + blockIdx.x;
    const uint32_t pt_x = blockIdx.x * CW + (uint32_t)(warp % CW), pt_y = blockIdx.y * CH + (uint32_t)(warp / CW);
    if (pt_x >= geo.ptiles_x || pt_y >= geo.ptiles_y) return;
    const uint32_t pt = pt_y * geo.ptiles_x + pt_x;
    const uint32_t tile_x0 = pt_x * G::TW, tile_j0 = pt_y * G::TH;
    const uint2 *winner = reinterpret_cast<const uint2 *>(p.winner) + (size_t)pt * S * 32;  // {leaf index, hit distance} per slot (K2)
    const ONE2 one = f2s(p.one);
    const V3x2 eye2 = v3x2s(v3(p.eye[0], p.eye[1], p.eye[2]));
    const float recip = frecip(fmul((float)SPP, (float)SPP));  // render.rs:219-220
    auto store = [&](uint32_t x, uint32_t j, float4 a, float4 b) {
        float4 *at = reinterpret_cast<float4 *>(p.out + (size_t)out_row(p, j) * p.pitch + (size_t)x * 32);
        at[0] = a;
        at[1] = b;
    };

    if (p.tile_hdr[ct].z == 0x7f800000u) {
        // no ray of this cull tile hit anything, and K2 wrote no winners: every sample is a miss
        const float4 a = make_float4(0.0f, 0.0f, 0.0f, 0.0f), b = make_float4(RT_INF, 0.0f, 0.0f, 0.0f);  // 0 * recip = +0
        for (int pi = 0; pi < G::NPX; pi++) {
            uint32_t x, j;
            slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, pi, x, j);
            if (x < p.width && j < p.row_count) store(x, j, a, b);
        }
        return;
    }
    float nx = 0.0f, ny = 0.0f, nz = 0.0f, cnt = 0.0f, dmin = RT_INF, px = 0.0f, py = 0.0f, pz = 0.0f;
#pragma unroll 1
    for (int s0 = 0; s0 < S; s0 += 2) {
        const int s1 = (s0 + 1 < S) ? s0 + 1 : s0;  // a pair past the end repeats the last slot
        uint32_t x0, j0, x1, j1;
        slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, s0 / NS, x0, j0);
        slot_pixel<PXW, PXH>(tile_x0, tile_j0, lane, s1 / NS, x1, j1);
        const V3x2 d = slot_dir2<SPP>(one, p, x0, image_row(p, j0), s0 % NS, x1, image_row(p, j1), s1 % NS);
        const uint2 a = __ldcs(&winner[s0 * 32 + lane]), b = __ldcs(&winner[s1 * 32 + lane]);
        const bool hit0 = a.x != NO_HIT, hit1 = b.x != NO_HIT;
        F2 dist = f2(__uint_as_float(a.y), __uint_as_float(b.y));  // primitive.rs:55-72, as K2 computed it
        const float4 w0 = __ldg(&p.sph[hit0 ? a.x : 0u]), w1 = __ldg(&p.sph[hit1 ? b.x : 0u]);
        const V3x2 cen = V3x2{f2(w0.x, w1.x), f2(w0.y, w1.y), f2(w0.z, w1.z)};
        if (!hit0) dist.x = 1.0f;
        if (!hit1) dist.y = 1.0f;
        // primitive.rs:83 normal; render.rs:199 hit point (pos + dir * distance)
        const V3x2 nrm = vnormalized2<(NS > 1)>(one, vadd2(one, eye2, vsub2(one, vmulf2(d, dist), cen)));
        const V3x2 hp = vadd2(one, eye2, vmulf2(d, dist));
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const int s = s0 + k;
            if (k == 1 && s1 == s0) break;
            const bool hit = k ? hit1 : hit0;
            if (s % NS == 0) nx = ny = nz = cnt = 0.0f, dmin = RT_INF, px = py = pz = 0.0f;
            if (hit) {
                const float t = k ? dist.y : dist.x;
                nx = fadd(nx, k ? nrm.x.y : nrm.x.x), ny = fadd(ny, k ? nrm.y.y : nrm.y.x), nz = fadd(nz, k ? nrm.z.y : nrm.z.x);
                cnt = fadd(cnt, 1.0f);
                if (t < dmin) dmin = t, px = k ? hp.x.y : hp.x.x, py = k ? hp.y.y : hp.y.x, pz = k ? hp.z.y : hp.z.x;
            }
            if (s % NS == NS - 1) {
                const uint32_t x = k ? x1 : x0, j = k ? j1 : j0;
                if (x < p.width && j < p.row_count)
                    store(x, j, make_float4(fmul(nx, recip), fmul(ny, recip), fmul(nz, recip), fmul(cnt, recip)),
                          make_float4(dmin, px, py, pz));
            }
        }
    }
}

}  // namespace rt

using namespace rt;

template <int SPP, int PXW, int PXH, int CW, int CH>
static cudaError_t launch_phased(bool diag, RtPixels fmt, const RenderParams &p, cudaStream_t stream) {
    using G = Geo<SPP, PXW, PXH, CW, CH>;
    const G geo(p.width, p.row_count);
    const uint32_t nc = geo.n_ctiles(), np = geo.n_ptiles();
    if (nc == 0 || np == 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(p.pool_count, 0, sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    const unsigned cb = (nc + P_WARPS - 1) / P_WARPS;
    const dim3 tiles2d(geo.ctiles_x, geo.ctiles_y);  // K2 / K4: one block per cull tile
    if (nc > 150000u) {
        const Geo<SPP, PXW, PXH, CW * 2, CH * 2> geoc(p.width, p.row_count);
        phase_cull_primary<SPP, PXW, PXH, CW, CH, 2><<<(geoc.n_ctiles() + P_WARPS - 1) / P_WARPS, 32 * P_WARPS, 0, stream>>>(p);
    } else {
        phase_cull_primary<SPP, PXW, PXH, CW, CH, 1><<<cb, 32 * P_WARPS, 0, stream>>>(p);
    }
    phase_test_primary<SPP, PXW, PXH, CW, CH><<<tiles2d, 32 * CW * CH, 0, stream>>>(p);
    if (fmt == RT_PIXELS_AOV) {  // geometry only: no shadow cull, no shading
        phase_aov_store<SPP, PXW, PXH, CW, CH><<<tiles2d, 32 * CW * CH, 0, stream>>>(p);
        return cudaGetLastError();
    }
    phase_cull_shadow<SPP, PXW, PXH, CW, CH><<<cb, 32 * P_WARPS, 0, stream>>>(p);
    if (fmt == RT_PIXELS_F32)
        phase_shade_store_f32<SPP, PXW, PXH, CW, CH><<<tiles2d, 32 * CW * CH, 0, stream>>>(p);
    else if (diag)
        phase_shade_store<SPP, PXW, PXH, CW, CH, true><<<tiles2d, 32 * CW * CH, 0, stream>>>(p);
    else
        phase_shade_store<SPP, PXW, PXH, CW, CH, false><<<tiles2d, 32 * CW * CH, 0, stream>>>(p);
    return cudaGetLastError();
}

// Scratch the phased pipeline needs for a frame of `rows` x `width`, `spp`: winner
// indices (4 B per padded sample), tile headers (16 B per cull tile) and the
// candidate pool (16 B units).
void rt_phased_scratch(uint32_t width, uint32_t rows, uint32_t spp, int shape, size_t *winner_bytes, size_t *hdr_bytes,
                       uint32_t *pool_units) {
    uint32_t nc = 0, np = 0, S = 0;
#define RT_GEO(SPP, PXW, PXH, CW, CH)                     \
    {                                                     \
        Geo<SPP, PXW, PXH, CW, CH> g(width, rows);        \
        nc = g.n_ctiles(), np = g.n_ptiles(), S = g.S;    \
    }
    switch (spp) {
        case 1:
            if (shape == 1) RT_GEO(1, 2, 2, 4, 4) else if (shape == 5) RT_GEO(1, 2, 2, 4, 2) else if (shape == 6) RT_GEO(1, 2, 2, 2, 4) else if (shape == 2) RT_GEO(1, 4, 2, 1, 2) else if (shape == 3) RT_GEO(1, 2, 1, 2, 4) else if (shape == 4) RT_GEO(1, 2, 1, 1, 2) else RT_GEO(1, 2, 2, 2, 2)
            break;
        case 2:
            if (shape == 1) RT_GEO(2, 1, 1, 4, 4) else RT_GEO(2, 1, 1, 2, 2)
            break;
        case 3:
            RT_GEO(3, 1, 1, 2, 2)
            break;
        case 4:
            if (shape == 1) RT_GEO(4, 1, 1, 4, 4) else RT_GEO(4, 1, 1, 2, 2)
            break;
        case 5:
            RT_GEO(5, 1, 1, 2, 2)
            break;
        case 6:
            RT_GEO(6, 1, 1, 2, 2)
            break;
        case 7:
            RT_GEO(7, 1, 1, 2, 2)
            break;
        default:
            RT_GEO(8, 1, 1, 2, 2)
            break;
    }
#undef RT_GEO
    *winner_bytes = (size_t)np * S * 32 * sizeof(uint2);  // {leaf index, hit distance} per (padded) sample
    *hdr_bytes = (size_t)nc * sizeof(uint4);
    uint64_t units = (uint64_t)nc * 384u;
    if (units < (1u << 20)) units = 1u << 20;
    if (units > (1u << 26)) units = 1u << 26;  // 1 GiB of 16-byte units
    *pool_units = (uint32_t)units;
}

cudaError_t rt_launch_render_phased(bool diag, RtPixels fmt, const RenderParams &p, cudaStream_t stream, int shape) {
    // shape 0: cull tile = 2x2 pixel tiles; shape 1: 4x4 pixel tiles
    switch (p.spp) {
        case 1:
            if (shape == 5) return launch_phased<1, 2, 2, 4, 2>(diag, fmt, p, stream);  // 64x16 cull tile
            if (shape == 6) return launch_phased<1, 2, 2, 2, 4>(diag, fmt, p, stream);  // 32x32 cull tile
            if (shape == 2) return launch_phased<1, 4, 2, 1, 2>(diag, fmt, p, stream);  // 8 pixels per lane
            if (shape == 3) return launch_phased<1, 2, 1, 2, 4>(diag, fmt, p, stream);  // 2 pixels per lane, 32x16 cull tile
            if (shape == 4) return launch_phased<1, 2, 1, 1, 2>(diag, fmt, p, stream);  // 2 pixels per lane, 16x8 cull tile
            return shape == 1 ? launch_phased<1, 2, 2, 4, 4>(diag, fmt, p, stream) : launch_phased<1, 2, 2, 2, 2>(diag, fmt, p, stream);
        case 2:
            return shape == 1 ? launch_phased<2, 1, 1, 4, 4>(diag, fmt, p, stream) : launch_phased<2, 1, 1, 2, 2>(diag, fmt, p, stream);
        case 3:
            return launch_phased<3, 1, 1, 2, 2>(diag, fmt, p, stream);
        case 4:
            return shape == 1 ? launch_phased<4, 1, 1, 4, 4>(diag, fmt, p, stream) : launch_phased<4, 1, 1, 2, 2>(diag, fmt, p, stream);
        // 25 .. 64 samples per pixel: one pixel per lane, its samples in groups of four slots like the 4x4 case
        case 5:
            return launch_phased<5, 1, 1, 2, 2>(diag, fmt, p, stream);
        case 6:
            return launch_phased<6, 1, 1, 2, 2>(diag, fmt, p, stream);
        case 7:
            return launch_phased<7, 1, 1, 2, 2>(diag, fmt, p, stream);
        case 8:
            return launch_phased<8, 1, 1, 2, 2>(diag, fmt, p, stream);
        default:
            return cudaErrorInvalidValue;
    }
}
