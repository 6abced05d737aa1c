// The wavefront path tracer.  Replaces `__global__ Kernel` and everything it calls
// (raygpu/kernel.cu:244-333, 432-512, 640-691, 703-994, 998-1093) plus CudaStarter's launch
// (kernel.cu:2562-2669) and the host accumulate loop (kernel.cu:2211-2218).
//
// The reference runs one thread per pixel through spp x depth x BVH nodes in a single megakernel.
// Here a frame is cut into batches of (pixel, sample) paths and each batch runs as a wavefront:
//
//   k_generate   camera rays for every path slot of the batch                (kernel.cu:1016-1076)
//   repeat max_depth times:
//     k_trace    persistent warps, every lane refills itself from the ray queue; closest hit through the 64 B
//                four-wide nodes (16-bit quantised child boxes, two 256-bit loads) with a shared-memory stack,
//                Moeller-Trumbore in the reference's operation order        (kernel.cu:468-512, 277-313)
//     k_shade    normal / texture / material scatter or termination; the unit-sphere rejection sampling of a
//                warp's rays is pooled and drained with per-lane refill; survivors are appended to the next
//                ray queue in ray order, one atomic per warp iteration      (kernel.cu:787-982)
//   k_resolve    per pixel, sum the batch's samples in sample order into the accumulator
//
// Terminated paths write their radiance to contrib[slot] exactly once, so the image is a
// deterministic function of (scene, settings, seed) whatever order the queues end up in.
//
// This TU is compiled with -fmad=false: arithmetic rounds operation by operation like the
// host-compiled reference; the box test asks for its FMAs explicitly.
#include "drb_internal.h"
#include "device_scene.cuh"
#include "philox.cuh"
#include "vec.cuh"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

namespace {

constexpr int kTraceThreads = 128;
#ifndef DRB_TRACE_STEPS
#define DRB_TRACE_STEPS 2
#endif
// Children that are hit besides the nearest one are pushed unsorted for scenes up to this many primitives, far-to-near
// (five compare-exchanges) above it: the sort costs 2 % on the million-triangle frame and returns 4 % on the
// 10 M-triangle city, whose rays cross many more boxes before they hit something.
#ifndef DRB_SORTED_PUSH_FROM
#define DRB_SORTED_PUSH_FROM (4 << 20)
#endif
constexpr int kSteps = DRB_TRACE_STEPS;   // descent steps per lane between two rounds of warp votes
constexpr uint32_t kInvalidPid = 0xFFFFFFFFu;
constexpr float kTMax = 10000.0f;       // singlehit's mindist / aabb2's t_max, kernel.cu:246, 435
constexpr float kEps = 0.0001f;         // hit_tri's EPSILON, kernel.cu:283

struct Camera {
    f3 from, llc, horizontal, vertical, uu, vu;
    float lens_radius;
    float wdiv, hdiv;                   // float(W / div), float(H / div), kernel.cu:1067-1068
};

struct FrameParams {
    int W, H;                           // pixel grid traced
    int tiles_x, tiles_y;               // 8x4 pixel tiles
    uint32_t tile_rank, tile_count;     // this call traces the tiles t with t % tile_count == tile_rank (1 GPU: 0, 1)
    uint32_t samples;                   // samples per pixel in this batch
    uint32_t sample_base;               // global index of the batch's first sample
    uint64_t seed;
    int backtex;
    float bg_intensity;
    float scene_scale;                  // max |coordinate| of the scene bounds
    Camera cam;
};

struct DevScene {
    float qlo[3], qscale[3];            // quantisation grid of the node boxes (drb_quant_grid)
    float pad_cap;                      // 0.49 x the largest grid extent: upper limit of the per-ray slab padding
    const WideNode* wnodes;
    const Prim* prims;
    const ShadeRec* recs;
    const DevTexture* textures;
    int nprims, ntextures;
};

// counters[]: 0,1 = ray queue sizes (ping-pong), 2 = trace ticket, 4..5 = 64-bit ray total
enum { CNT_Q0 = 0, CNT_Q1 = 1, CNT_TICKET = 2, CNT_SHADE_TICKET = 3, CNT_RAYS = 4, CNT_WORDS = 8 };

struct Queues {
    float4* ray_o[2];                   // (origin, pid bits)
    float4* ray_d[2];                   // (direction, rng draw count bits)
    float4* thr[2];                     // (attenuation rgb, 0)
    uint2* hit;                         // (t bits, prim slot or -1)
    float4* contrib;                    // radiance per path slot
    uint32_t* counters;
};

// ---- path slot <-> pixel / sample ---------------------------------------------------------------
// slot = ((tile * samples) + s) * 32 + lane, lane = (y & 3) * 8 + (x & 7): a warp is one 8x4 pixel
// tile at one sample index (coherent camera rays), consecutive warps are consecutive samples of it.
DRB_D bool slot_to_pixel(const FrameParams& fp, uint32_t slot, int& x, int& y, uint32_t& s)
{
    const uint32_t lane = slot & 31u, unit = slot >> 5;
    s = unit % fp.samples;
    const uint32_t tile = (unit / fp.samples) * fp.tile_count + fp.tile_rank;      // local tile -> image tile
    x = (int)(tile % (uint32_t)fp.tiles_x) * 8 + (int)(lane & 7u);
    y = (int)(tile / (uint32_t)fp.tiles_x) * 4 + (int)(lane >> 3);
    return x < fp.W && y < fp.H && tile < (uint32_t)(fp.tiles_x * fp.tiles_y);
}

// ---- sampling helpers (kernel.cu:640-662, 988-994) ----------------------------------------------
// The reference draws the components inside one make_float3(...) argument list, whose evaluation
// order C++ leaves unspecified.  The oracle build (g++) evaluates it right to left, so the FIRST
// draw of an attempt lands in the LAST component; the stream is consumed the same way here so that
// paths stay aligned with the oracle draw for draw.  (Any order is the same distribution.)
// The rejection test.  The reference rejects when pow(getLength(p), 2) >= 1 with getLength = sqrtf(dot(p, p))
// (kernel.cu:200-203, 641); that is decided by d = dot(p, p) alone, without the square root: for d >= 1 the correctly
// rounded root is >= 1 and so is its square; for d < 1 the root rounds to at most 1 - 2^-24 (sqrt(1 - 2^-24) lies below
// the midpoint 1 - 2^-25), whose square, under powf's sub-ulp error as under a float multiply, stays below 1.
// (random_in_unit_sphere itself, kernel.cu:640-647, lives in k_shade's pooled sampling stage: one lane per request with
// refill, then teams of lanes for the last requests; both consume words draws, draws + 1, draws + 2 per attempt.)
DRB_D f3 random_in_unit_disk(PathRng& rng)
{
    for (;;) {
        const float b = rng.uniform(), a = rng.uniform();
        const f3 p = mk3(a * 2.0f - 1.0f, b * 2.0f - 1.0f, 0.0f);
        if (dot(p, p) >= 1.0f) continue;
        return p;
    }
}

// ---- k_generate ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_generate(FrameParams fp, uint32_t nslots, Queues q)
{
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= nslots) return;
    int x, y; uint32_t s;
    if (!slot_to_pixel(fp, slot, x, y, s)) {
        q.ray_o[0][slot] = make_float4(0.f, 0.f, 0.f, __uint_as_float(kInvalidPid));
        q.ray_d[0][slot] = make_float4(0.f, 0.f, 0.f, 0.f);
        q.thr[0][slot] = make_float4(0.f, 0.f, 0.f, 0.f);
        return;
    }
    PathRng rng;
    rng.init(fp.seed, (uint32_t)x, (uint32_t)y, fp.sample_base + s, 0u);
    const Camera& c = fp.cam;
    // kernel.cu:1067-1068: float(x) + double uniform, divided by float(W/div), rounded to float
    const double u1 = (double)rng.uniform();
    const float nu = (float)(((double)(float)x + u1) / (double)c.wdiv);
    const double u2 = (double)rng.uniform();
    const float nv = (float)(((double)(float)y + u2) / (double)c.hdiv);
    const f3 rd = mk3(c.lens_radius) * random_in_unit_disk(rng);
    const f3 offset = c.uu * mk3(rd.x) + c.vu * mk3(rd.y);
    const f3 dir = c.llc + mk3(nu) * c.horizontal + mk3(nv) * c.vertical - c.from - offset;
    const f3 org = c.from + offset;
    q.ray_o[0][slot] = make_float4(org.x, org.y, org.z, __uint_as_float(slot));
    q.ray_d[0][slot] = make_float4(dir.x, dir.y, dir.z, __uint_as_float(rng.draws));
    q.thr[0][slot] = make_float4(1.f, 1.f, 1.f, __uint_as_float((uint32_t)x | ((uint32_t)y << 16)));   // pixel rides along: no divisions in k_shade
}

// ---- closest hit ----------------------------------------------------------------------------------
DRB_D float safe_inv(float d)
{
    // aabb2 divides by the direction component (kernel.cu:252); a zero component behaves like a
    // vanishing one here, which keeps the slab arithmetic free of inf - inf.  The inverse only feeds the
    // box test, whose planes are padded by 2^-19 of the coordinates involved: the one-ulp error of the
    // approximate reciprocal (a relative 6e-8 on every plane distance) is 30 times below that, so the
    // test stays conservative -- and the three IEEE divisions per ray (~35 instructions, run by the few
    // lanes that are refilling while the rest of the warp waits) become three MUFU.RCP.
    const float lim = 1.0e-20f;
    if (fabsf(d) < lim) d = copysignf(lim, d);
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
    return r;
}

// hit_tri (kernel.cu:277-313) on precomputed edges; updates (best, bestp) under the acceptance rules
// of singlehit / hit (kernel.cu:449, 488): EPS < t < 10000 and t < best
DRB_D void intersect_prim(const Prim* __restrict__ prims, int slot, const f3& o, const f3& d, float& best, int& bestp)
{
    const f8 pab = ldg256(&prims[slot].a);
    const float4 pa = pab.lo, pb = pab.hi;
    if (__float_as_int(pa.w) == DRB_KIND_TRI) {
        const float4 pc = ldg256(&prims[slot].c).lo;
        const f3 v0 = xyz(pa), e1 = xyz(pb), e2 = xyz(pc);
        const f3 h = cross(d, e2);
        const float a = dot(e1, h);
        if (a > -kEps && a < kEps) return;
        const float f = __frcp_rn(a);               // correctly rounded 1/a == (float)(1.0 / a) of kernel.cu:293
        const f3 sv = o - v0;
        const float u = f * dot(sv, h);
        if (u < 0.0f || u > 1.0f) return;
        const f3 qv = cross(sv, e1);
        const float v = f * dot(d, qv);
        if (v < 0.0f || u + v > 1.0f) return;
        const float t = f * dot(e2, qv);
        if (t > kEps && t < best) { best = t; bestp = slot; }
    } else {
        // hit_sphere (kernel.cu:316-333): near root only
        const f3 oc = o - xyz(pa);
        const float radius = pb.x;
        const float ld = length(d), lo = length(oc);
        const float a = ld * ld;
        const float half_b = dot(oc, d);
        const float c = lo * lo - radius * radius;
        const float disc = half_b * half_b - a * c;
        if (disc < 0.0f) return;
        const float t = (-half_b - sqrtf(disc)) / a;
        if (t > 0.0f && t < best) { best = t; bestp = slot; }
    }
}

// the float 2^23 + q for the 16-bit half of `w` that `sel` names: bytes (q.lo, q.hi, 0x00, 0x4B)
DRB_D float prmt_exp23(uint32_t w, uint32_t sel)
{
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(0x4B000000u), "r"(sel));
    return __uint_as_float(r);
}

constexpr int kSentinel = (int)0x80000000;     // bottom of every traversal stack: "this lane has no ray in flight"

// What one traversal answers.  kClosest and kClosestSorted: the closest hit, hit()'s query (kernel.cu:468-512), with the hit
// children besides the nearest one pushed unsorted or far-to-near (see DRB_SORTED_PUSH_FROM); a ray's result is (t, primitive
// slot).  kAnyHit: does hit()'s test accept some primitive at t < tmax?  The ray's tmax (already clamped to 10000) rides in
// the w component of the direction stream, starts `best`, and so is the slab test's far bound; the first accepted primitive
// ends the ray, and the result is one byte.  The primitive test is intersect_prim started from best = tmax, so both modes
// accept the same primitives below that bound and occluded == (closest id >= 0 && closest t < tmax) exactly: the padded
// boxes never cull an accepted hit (§4 of DESIGN.md), and a box holding a hit at t < tmax still passes with its far bound
// lowered to tmax.  (Once a ray accepts, best < tmax, but the ray has ended and tests no further box.)
enum TraceMode { kClosest, kClosestSorted, kAnyHit };

// Persistent traversal with per-lane dynamic ray fetch (after Aila & Laine, "Understanding the Efficiency of
// Ray Traversal on GPUs", HPG 2009).  The reference walks its threaded tree one thread per pixel (hit(),
// kernel.cu:468-512); incoherent bounces then leave most lanes of a warp idle while the longest ray
// finishes.  Here a lane keeps (ray, node, stack) state.  Every iteration each lane does ONE step -- an
// internal node (both child boxes of the 64 B node, near child next, far child pushed) or the leaf it
// popped (one primitive) -- and the warp re-converges.  When fewer than `refill` lanes still have a ray,
// the idle lanes claim fresh rays from the queue with ONE atomic per warp (ballot + popc + shfl), so warps
// stay populated until the queue runs dry.  (A while-while variant measured slower on B200: with
// one-primitive leaves, lanes that reach a leaf wait for the slowest descent.)
// Traces the first `count` rays of ro / rdv, taken in queue order; the result of a ray goes to hit (closest) or occluded
// (any hit) at its queue position.
template <TraceMode kMode>
DRB_D void traverse(const DevScene& sc, float scene_scale, const float4* __restrict__ ro, const float4* __restrict__ rdv,
                    uint2* __restrict__ hit, uint8_t* __restrict__ occluded, uint32_t* counters, uint32_t count,
                    int refill, int leaf_batch, int step_min)
{
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;

    int node = kSentinel;
    int leaf = 0;                                   // stashed leaf (~primitive slot, always < 0), 0 = none
    uint32_t ray = 0xFFFFFFFFu;
    bool exhausted = false;                         // warp-uniform: the queue has been handed out completely
    f3 o = mk3(0.f), d = mk3(0.f);
    // per-ray plane constants, per axis as (near, far) pairs: (t_near, t_far) = (2^23 + q_near, 2^23 + q_far) * (s, s) + (c_near, c_far),
    // near / far plane picked by the PRMT selectors
    float2 sxx = {}, syy = {}, szz = {}, cxx = {}, cyy = {}, czz = {};
    uint32_t snx = 0x7410u, sny = 0x7410u, snz = 0x7410u, sfx = 0x7432u, sfy = 0x7432u, sfz = 0x7432u;   // PRMT selectors of the near / far plane
    float best = kTMax; int bestp = -1;
    // traversal stack in dynamic shared memory, [level][thread], sized by the host to the tree height + 2: every
    // lane owns a bank, so pushes and pops at different depths are still one conflict-free wavefront per warp
    // (a local-memory stack costs one L1 wavefront per distinct depth), and there is no spill path.
    extern __shared__ int s_stack[];
    int* sp = s_stack + threadIdx.x;                // points at the next free slot of this lane's column
#define DRB_PUSH(v) do { *sp = (v); sp += 128; } while (0)
#define DRB_POP() (sp -= 128, *sp)

    for (;;) {
        // ---- refill idle lanes ----------------------------------------------------------------------
        const bool idle = (node == kSentinel && leaf == 0);
        const unsigned midle = __ballot_sync(0xffffffffu, idle);
        if (midle == 0xffffffffu && exhausted) break;
        if (!exhausted && (midle == 0xffffffffu || 32 - __popc(midle) < refill)) {
            const int leader = __ffs(midle) - 1;
            uint32_t base = 0;
            if ((int)lane == leader) base = atomicAdd(&counters[CNT_TICKET], (uint32_t)__popc(midle));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (base + (uint32_t)__popc(midle) >= count) exhausted = true;
            if (idle) {
                const uint32_t i = base + (uint32_t)__popc(midle & lt_mask);
                if (i < count) {
                    const float4 o4 = ro[i], d4 = rdv[i];
                    bool skip;                                      // the ray has no result to search for
                    if constexpr (kMode == kAnyHit) skip = !(d4.w > 0.0f);    // nothing is accepted at t < tmax <= 0 (t > 1e-4 / t > 0)
                    else skip = __float_as_uint(o4.w) == kInvalidPid;
                    if (skip || sc.nprims == 0) {
                        if constexpr (kMode == kAnyHit) occluded[i] = 0;
                        else hit[i] = make_uint2(__float_as_uint(-1.0f), 0xFFFFFFFFu);
                    } else {
                        ray = i;
                        o = xyz(o4); d = xyz(d4);
                        const float ix = safe_inv(d.x), iy = safe_inv(d.y), iz = safe_inv(d.z);
                        // per-ray slab padding: on top of the quantisation margin the ray sees every box grown by a few
                        // ulps of the distances involved, so a hit the triangle test accepts by rounding is never culled
                        // An empty child slot (min 65535 > max 0) fails the test as long as twice the padding stays below the
                        // grid's extent on ONE axis, so the padding is capped just under half the largest extent.  The cap only
                        // binds for origins ~10^5 scene sizes away, where it still leaves tens of ulps of margin; without it such
                        // a ray would follow empty links (they carry the stack sentinel's bits) and overrun the stack bound.
                        const float pad = fminf((fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fabsf(o.z)) + scene_scale) * 1.9073486e-6f, sc.pad_cap);
                        // plane coordinate = qlo + q * qscale; t = (coordinate -/+ pad - o) * inv, folded into one FMA on
                        // the float 2^23 + q: t = (2^23 + q) * s + (c - 2^23 * s).  The near plane is the min plane for a
                        // positive direction component and the max plane for a negative one.
                        const float sx = sc.qscale[0] * ix, sy = sc.qscale[1] * iy, sz = sc.qscale[2] * iz;
                        const float px = copysignf(pad, ix), py = copysignf(pad, iy), pz = copysignf(pad, iz);
                        sxx = make_float2(sx, sx); syy = make_float2(sy, sy); szz = make_float2(sz, sz);
                        cxx = make_float2(fmaf(-8388608.0f, sx, (sc.qlo[0] - o.x - px) * ix), fmaf(-8388608.0f, sx, (sc.qlo[0] - o.x + px) * ix));
                        cyy = make_float2(fmaf(-8388608.0f, sy, (sc.qlo[1] - o.y - py) * iy), fmaf(-8388608.0f, sy, (sc.qlo[1] - o.y + py) * iy));
                        czz = make_float2(fmaf(-8388608.0f, sz, (sc.qlo[2] - o.z - pz) * iz), fmaf(-8388608.0f, sz, (sc.qlo[2] - o.z + pz) * iz));
                        snx = ix >= 0.f ? 0x7410u : 0x7432u; sny = iy >= 0.f ? 0x7410u : 0x7432u; snz = iz >= 0.f ? 0x7410u : 0x7432u;
                        sfx = snx ^ 0x22u; sfy = sny ^ 0x22u; sfz = snz ^ 0x22u;
                        best = kMode == kAnyHit ? d4.w : kTMax; bestp = -1;
                        sp = s_stack + threadIdx.x; DRB_PUSH(kSentinel);
                        node = 0;
                    }
                }
            }
        }
        // ---- kSteps descent steps per lane between warp votes ----------------------------------------------
#pragma unroll
        for (int step = 0; step < kSteps; ++step) {
        if (node >= 0) {
            const WideNode* np = sc.wnodes + node;
            const f8 nA = ldg256(np->bx), nB = ldg256(np->bz);          // the whole node: two 256-bit loads
            // (near, far) distance of one axis: both planes come from the same word and share the scale, so they go through
            // one packed FFMA2.  Each half is one IEEE fma rounded like fmaf.  (Only explicit fmas are packed: ptxas contracts
            // a packed mul followed by a packed add into FFMA2 even under -fmad=false.)
#define DRB_PLANES(w, sn, sf, s_, c_) __ffma2_rn(make_float2(prmt_exp23(__float_as_uint(w), (sn)), prmt_exp23(__float_as_uint(w), (sf))), (s_), (c_))
#define DRB_CHILD(c, wx, wy, wz)                                                                                              \
            const float2 x##c = DRB_PLANES(wx, snx, sfx, sxx, cxx), y##c = DRB_PLANES(wy, sny, sfy, syy, cyy), z##c = DRB_PLANES(wz, snz, sfz, szz, czz); \
            const float tn##c = fmaxf(fmaxf(x##c.x, y##c.x), fmaxf(z##c.x, 0.0f));                                            \
            const float tf##c = fminf(fminf(x##c.y, y##c.y), fminf(z##c.y, best));                                            \
            const uint32_t k##c = (tn##c <= tf##c) ? ((__float_as_uint(tn##c) & 0xFFFFFFFCu) | c##u) : 0xFFFFFFFFu;
            DRB_CHILD(0, nA.lo.x, nA.hi.x, nB.lo.x)
            DRB_CHILD(1, nA.lo.y, nA.hi.y, nB.lo.y)
            DRB_CHILD(2, nA.lo.z, nA.hi.z, nB.lo.z)
            DRB_CHILD(3, nA.lo.w, nA.hi.w, nB.lo.w)
#undef DRB_CHILD
#undef DRB_PLANES
            // t_near >= 0, so its bits order like unsigned integers; the two low bits carry the slot
            if constexpr (kMode == kClosestSorted) {
            // sort the four keys (5 compare-exchanges), push the hits far-to-near, continue with the nearest
            uint32_t a0 = min(k0, k1), a1 = max(k0, k1), a2 = min(k2, k3), a3 = max(k2, k3);
            const uint32_t s0 = min(a0, a2), t1 = max(a0, a2), t2 = min(a1, a3), s3 = max(a1, a3);
            const uint32_t s1 = min(t1, t2), s2 = max(t1, t2);
            if (s0 == 0xFFFFFFFFu) node = DRB_POP();
            else {
                const int c0 = __float_as_int(nB.hi.x), c1 = __float_as_int(nB.hi.y), c2 = __float_as_int(nB.hi.z), c3 = __float_as_int(nB.hi.w);
#define DRB_LINK(k) (((k) & 2u) ? (((k) & 1u) ? c3 : c2) : (((k) & 1u) ? c1 : c0))
                if (s3 != 0xFFFFFFFFu) DRB_PUSH(DRB_LINK(s3));
                if (s2 != 0xFFFFFFFFu) DRB_PUSH(DRB_LINK(s2));
                if (s1 != 0xFFFFFFFFu) DRB_PUSH(DRB_LINK(s1));
                node = DRB_LINK(s0);
#undef DRB_LINK
            }
            } else {
            const uint32_t kmin = min(min(k0, k1), min(k2, k3));
            if (kmin == 0xFFFFFFFFu) node = DRB_POP();
            else {
                const int c0 = __float_as_int(nB.hi.x), c1 = __float_as_int(nB.hi.y), c2 = __float_as_int(nB.hi.z), c3 = __float_as_int(nB.hi.w);
                if (k3 != kmin && k3 != 0xFFFFFFFFu) DRB_PUSH(c3);
                if (k2 != kmin && k2 != 0xFFFFFFFFu) DRB_PUSH(c2);
                if (k1 != kmin && k1 != 0xFFFFFFFFu) DRB_PUSH(c1);
                if (k0 != kmin && k0 != 0xFFFFFFFFu) DRB_PUSH(c0);
                node = (kmin & 2u) ? ((kmin & 1u) ? c3 : c2) : ((kmin & 1u) ? c1 : c0);
            }
            }
        }
        // a lane that arrives at a leaf stashes it and keeps descending
        if (node < 0 && node != kSentinel && leaf == 0) { leaf = node; node = DRB_POP(); }
        }
        // ---- postponed leaves -------------------------------------------------------------------------
        // The (long, divergent) primitive test runs for the whole warp at once when enough lanes hold a stashed
        // leaf, or when too few lanes can still step.  (Testing each leaf as soon as a lane reaches it is slower, for
        // any hit as well: DESIGN.md §5.)
        const unsigned mpend = __ballot_sync(0xffffffffu, leaf != 0);
        if (mpend) {
            const unsigned mstep = __ballot_sync(0xffffffffu, node >= 0);
            if (__popc(mpend) >= leaf_batch || __popc(mstep) < step_min) {
                if (leaf != 0) {
                    intersect_prim(sc.prims, ~leaf, o, d, best, bestp); leaf = 0;
                    if constexpr (kMode == kAnyHit) {
                        if (bestp >= 0) node = kSentinel;           // an accepted primitive ends the ray, whatever the lane holds next
                    }
                }
            }
        }
        // ---- retire -----------------------------------------------------------------------------------
        if (node == kSentinel && leaf == 0 && ray != 0xFFFFFFFFu) {
            if constexpr (kMode == kAnyHit) occluded[ray] = bestp >= 0 ? 1 : 0;
            else hit[ray] = bestp >= 0 ? make_uint2(__float_as_uint(best), (uint32_t)bestp) : make_uint2(__float_as_uint(-1.0f), 0xFFFFFFFFu);
            ray = 0xFFFFFFFFu;
        }
    }
#undef DRB_PUSH
#undef DRB_POP
}

#ifndef DRB_TRACE_MIN_BLOCKS
#define DRB_TRACE_MIN_BLOCKS 8
#endif
// closest hit of the rays of queue `cur`
template <bool kSortedPush>
__global__ void __launch_bounds__(kTraceThreads, DRB_TRACE_MIN_BLOCKS) k_trace(DevScene sc, float scene_scale, const float4* __restrict__ ro, const float4* __restrict__ rdv,
                                               uint2* __restrict__ hit, uint32_t* counters, int cur, int refill, int leaf_batch, int step_min)
{
    traverse<kSortedPush ? kClosestSorted : kClosest>(sc, scene_scale, ro, rdv, hit, nullptr, counters, counters[cur], refill, leaf_batch, step_min);
}

// any hit of a query chunk (ray count in counters[0])
__global__ void __launch_bounds__(kTraceThreads, DRB_TRACE_MIN_BLOCKS) k_occluded(DevScene sc, float scene_scale, const float4* __restrict__ ro,
                                                                                 const float4* __restrict__ rdv, uint8_t* __restrict__ occluded,
                                                                                 uint32_t* counters, int refill, int leaf_batch, int step_min)
{
    traverse<kAnyHit>(sc, scene_scale, ro, rdv, nullptr, occluded, counters, counters[0], refill, leaf_batch, step_min);
}

// ---- shading ---------------------------------------------------------------------------------------
// tex2D<uchar4> with the reference's descriptor (kernel.cu:1959-1964): normalised coordinates, wrap,
// point filter; rows top-down
DRB_D uchar4 tex_fetch(const DevTexture* __restrict__ table, int ntex, int k, float u, float v)
{
    uchar4 r = make_uchar4(0, 0, 0, 0);
    if (k < 0 || k >= ntex) return r;
    const DevTexture t = table[k];
    if (t.w <= 0 || t.h <= 0 || t.texels == nullptr) return r;
    const float fu = u - floorf(u), fv = v - floorf(v);
    int ix = (int)floorf(fu * (float)t.w), iy = (int)floorf(fv * (float)t.h);
    if (!(ix >= 0)) ix = 0;
    if (!(iy >= 0)) iy = 0;
    if (ix >= t.w) ix = t.w - 1;
    if (iy >= t.h) iy = t.h - 1;
    return __ldg(&t.texels[(size_t)iy * (size_t)t.w + (size_t)ix]);
}

DRB_D f3 reflect(f3 v, f3 n)
{
    const float k = 2.0f * dot(v, n);               // 2.0 * dot in double is the same float (kernel.cu:668)
    return v - mk3(k) * n;
}

DRB_D float reflectance(float cosine, float ref_idx)
{
    // Schlick, kernel.cu:686-691; the (1 - cosine)^5 term is evaluated in double there
    float r0 = (1.0f - ref_idx) / (1.0f + ref_idx);
    r0 = r0 * r0;
    const double x = (double)(1.0f - cosine);
    const double x2 = x * x;
    return (float)((double)r0 + (double)(1.0f - r0) * (x2 * x2 * x));
}

DRB_D f3 refract(f3 uv, f3 n, float etai_over_etat)
{
    // kernel.cu:678-683
    const float cos_theta = fminf(dot(uv * mk3(-1.0f), n), 1.0f);
    const f3 perp = mk3(etai_over_etat) * (uv + mk3(cos_theta) * n);
    const float lp = length(perp);
    const float k = (float)(-sqrt(fabs(1.0 - (double)(lp * lp))));
    return perp + mk3(k) * n;
}

// environment colour, kernel.cu:951-976 (the caller applies attenuation and intensity in the reference's order)
DRB_D f3 environment(const DevScene& sc, const FrameParams& fp, f3 raydir)
{
    const f3 ud = normalize(raydir);
    if (fp.backtex > -1) {
        const double dx = (double)ud.x, dy = (double)ud.y, dz = (double)ud.z + 1.0;
        const float m = (float)(2.0 * sqrt(dx * dx + dy * dy + dz * dz));
        f3 t = ud / mk3(m) + mk3(0.5f);
        t.y = -t.y;
        const uchar4 c = tex_fetch(sc.textures, sc.ntextures, fp.backtex, t.x, -t.y + 1.0f);
        return mk3((float)c.x / 255.0f, (float)c.y / 255.0f, (float)c.z / 255.0f);
    }
    const float t = (float)(0.5 * ((double)ud.y + 1.0));
    const float omt = (float)(1.0 - (double)t);
    return mk3(omt) * mk3(1.0f) + mk3(t) * mk3(0.5f, 0.7f, 1.0f);
}

// The unit-sphere rejection loop (kernel.cu:640-647) is ~60 % of the shading instructions and, run per ray inside a warp,
// keeps ~10 of 32 lanes busy: the warp waits for its unluckiest lane while each attempt costs a Philox block.  So a warp
// takes kShadeRays consecutive rays per iteration and works in three stages through shared memory:
//   1  (full width, once per 32 rays) loads, miss / emissive termination, normal, textures, material; a ray that scatters
//      leaves a record: its finished successor (mirror, glass), or what stage 3 needs plus a sampling request;
//   2  the requests form a pool that the 32 lanes drain with per-lane refill: a lane makes one attempt per iteration and
//      takes the next request as soon as its own is accepted, so the lanes stay busy until the pool is dry.  ONE Philox
//      call site serves the block a stream resumes in and the blocks after it.  The last few requests are finished by
//      TEAMS of lanes that try consecutive attempts of one stream side by side;
//   3  (full width) finishes the scatter from record + sample and appends the successors IN RAY ORDER with one atomic
//      for the whole group -- the next bounce sees the same queue order as a ray-per-lane pass would give it.
// Every path consumes exactly the words it always did (draw n of a path is word n of its Philox stream), so the image
// does not change by a bit.
#ifndef DRB_SHADE_GROUPS
#define DRB_SHADE_GROUPS 2
#endif
constexpr int kShadeGroups = DRB_SHADE_GROUPS;          // 32-ray groups per warp iteration
constexpr int kShadeRays = 32 * kShadeGroups;
#ifndef DRB_SHADE_TEAM_AT
#define DRB_SHADE_TEAM_AT 8
#endif
constexpr int kShadeTeamAt = DRB_SHADE_TEAM_AT;          // open requests from which the sampling pool is finished in teams
enum { REC_HX = 0, REC_HY, REC_HZ, REC_VX, REC_VY, REC_VZ, REC_AR, REC_AG, REC_AB, REC_ROUGH, REC_PID, REC_XY, REC_DRAWS, REC_MODE,
       REC_SX, REC_SY, REC_SZ, REC_WORDS };
enum { MODE_DEAD = 0, MODE_FINAL = 1, MODE_DIFFUSE = 2, MODE_DIFFUSE_UNIT = 3, MODE_METAL = 4 };

#ifndef DRB_SHADE_MIN_BLOCKS
#define DRB_SHADE_MIN_BLOCKS 8
#endif
__global__ void __launch_bounds__(128, DRB_SHADE_MIN_BLOCKS) k_shade(DevScene sc, FrameParams fp, const float4* __restrict__ ro, const float4* __restrict__ rdv,
                                                                           const float4* __restrict__ thr, const uint2* __restrict__ hit,
                                                                           float4* __restrict__ ro_next, float4* __restrict__ rdv_next,
                                                                           float4* __restrict__ thr_next, float4* __restrict__ contrib,
                                                                           uint32_t* counters, int cur, int last_bounce)
{
    __shared__ float s_rec[4][REC_WORDS][kShadeRays];           // [warp][field][slot]: conflict-free for slot = lane + 32 g
    __shared__ uint8_t s_req[4][kShadeRays];                    // slots that wait for a unit-sphere sample, in ray order
    const uint32_t count = counters[cur];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    float (*rec)[kShadeRays] = s_rec[warp];
    uint8_t* req = s_req[warp];
    uint32_t local_rays = 0;                                    // a warp shades rays of one queue (< 2^32): 32 bits hold its sum
    for (;;) {
        // the next kShadeRays rays of the queue: a ticket rather than a grid stride, so that warps whose groups are cheap
        // (all misses, no sampling) simply take more of them (frame 412 -> 404 ms)
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&counters[CNT_SHADE_TICKET], (uint32_t)kShadeRays);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= count) break;
        // ---- stage 1 ----------------------------------------------------------------------------------------------------
        int nreq = 0, nalive = 0;
#pragma unroll 1
        for (int g = 0; g < kShadeGroups; ++g) {
            const uint32_t i = base + (uint32_t)g * 32u + lane;
            const int slot = g * 32 + (int)lane;
            int mode = MODE_DEAD;
            if (i < count) {
                const float4 o4 = __ldg(&ro[i]);
                const uint32_t pid = __float_as_uint(o4.w);
                if (pid != kInvalidPid) {
                    local_rays++;
                    const float4 d4 = __ldg(&rdv[i]);
                    const float4 a4 = __ldg(&thr[i]);
                    const uint2 h = __ldg(&hit[i]);
                    const f3 rayo = xyz(o4), raydir = xyz(d4);
                    f3 atten = xyz(a4);
                    const float t = __uint_as_float(h.x);
                    const int prim = (int)h.y;
                    if (!(prim >= 0 && t > 0.0f)) {
                        const f3 c = atten * environment(sc, fp, raydir) * mk3(fp.bg_intensity);
                        contrib[pid] = make_float4(c.x, c.y, c.z, 0.f);
                    } else {
                        const ShadeRec* srec = sc.recs + prim;
                        const float4 r0 = __ldg(&srec->r[0]), r1 = __ldg(&srec->r[1]), r2 = __ldg(&srec->r[2]);
                        const uint32_t flags = __float_as_uint(r0.w);
                        const int mat = __float_as_int(r2.y), texnum = __float_as_int(r2.z), rtexnum = __float_as_int(r2.w);
                        const f3 hitpoint = rayo + mk3(t) * raydir;
                        f3 N; f3 texco = mk3(0.f);
                        if (flags & DRB_SF_SPHERE) {
                            const float4 pa = __ldg(&sc.prims[prim].a), pb = __ldg(&sc.prims[prim].b);
                            N = (hitpoint - xyz(pa)) / mk3(pb.x);                // kernel.cu:708, not normalised
                        } else {
                            // getnormal, kernel.cu:713-767
                            if ((flags & DRB_SF_NEEDS_UV) || !(flags & DRB_SF_FACE_NORMAL)) {
                                const float4 pa = __ldg(&sc.prims[prim].a), pb = __ldg(&sc.prims[prim].b), pc = __ldg(&sc.prims[prim].c);
                                const f3 v0 = xyz(pa), e1 = xyz(pb), e2 = xyz(pc);
                                N = cross(e1, e2);
                                if (flags & DRB_SF_NEEDS_UV) {
                                    const f3 pvec = cross(raydir, e2);
                                    const float det = dot(e1, pvec);
                                    const float inv_det = 1.0f / det;
                                    const f3 tvec = rayo - v0;
                                    const float bu = dot(tvec, pvec) * inv_det;
                                    const f3 qvec = cross(tvec, e1);
                                    const float bv = dot(raydir, qvec) * inv_det;
                                    const float bw = 1.0f - bu - bv;
                                    const float4 r3 = __ldg(&srec->r[3]), r4 = __ldg(&srec->r[4]), r5 = __ldg(&srec->r[5]), r6 = __ldg(&srec->r[6]);
                                    texco = mk3(bw) * mk3(r3.w, r6.x, 0.f) + mk3(bu) * mk3(r4.w, r6.y, 0.f) + mk3(bv) * mk3(r5.w, r6.z, 0.f);
                                    if (flags & DRB_SF_SMOOTH) N = mk3(bw) * xyz(r3) + mk3(bu) * xyz(r4) + mk3(bv) * xyz(r5);
                                    else if (flags & DRB_SF_FACE_NORMAL) N = xyz(r0);
                                }
                            } else {
                                N = xyz(r0);
                            }
                            N = normalize(N);
                        }
                        const bool front = dot(raydir, N) < 0.0f;                  // get_face_normal, kernel.cu:235-238
                        if (!front) N = N * mk3(-1.0f);

                        f3 ocolor = xyz(r1);
                        float rough = r1.w;
                        if (texnum >= 0) {
                            const uchar4 c = tex_fetch(sc.textures, sc.ntextures, texnum, texco.x, -texco.y + 1.0f);
                            ocolor = mk3((float)c.x / 255.0f, (float)c.y / 255.0f, (float)c.z / 255.0f);
                        } else if (flags & DRB_SF_CHECKER) {
                            // checker, kernel.cu:776-784
                            const float yes = floorf(texco.x * 10.0f) + floorf(texco.y * 10.0f);
                            if (fmodf(yes, 2.0f) == 0.0f) ocolor = mk3(0.8f);
                        }
                        if (rtexnum >= 0) {
                            const uchar4 c = tex_fetch(sc.textures, sc.ntextures, rtexnum, texco.x, -texco.y + 1.0f);
                            rough = (float)c.x / 255.0f / 2.0f;
                        }
                        if (!(mat == 0 || mat == 2 || mat == 3 || mat == 4 || mat == 5)) {
                            const f3 c = ocolor * atten;                            // emissive, kernel.cu:941-944
                            contrib[pid] = make_float4(c.x, c.y, c.z, 0.f);
                        } else if (last_bounce) {
                            contrib[pid] = make_float4(0.f, 0.f, 0.f, 0.f);       // depth exhausted: black (kernel.cu:981), nothing to scatter
                        } else {
                            uint32_t draws = __float_as_uint(d4.w);
                            f3 vec;                                                 // successor direction (FINAL), normal (diffuse lobe) or mirror direction (metal lobe)
                            atten = atten * ocolor;
                            if (mat == 2) {
                                vec = reflect(normalize(raydir), N);                // mirror, kernel.cu:867-874
                                mode = MODE_FINAL;
                            } else if (mat == 4) {
                                // glass, kernel.cu:914-939 (ior comes from addional.y even when a roughness map is bound)
                                const float ir = r1.w;
                                const float ratio = front ? (float)(1.0 / (double)ir) : ir;
                                const f3 unit = normalize(raydir);
                                const float cos_theta = fminf(dot(unit * mk3(-1.0f), N), 1.0f);
                                const float sin_theta = (float)sqrt(1.0 - (double)(cos_theta * cos_theta));
                                bool mirror = (ratio * sin_theta) > 1.0f;
                                if (!mirror) {
                                    const uint32_t xy = __float_as_uint(a4.w);
                                    PathRng rng;
                                    rng.init(fp.seed, xy & 0xFFFFu, xy >> 16, fp.sample_base + (pid >> 5) % fp.samples, draws);
                                    mirror = reflectance(cos_theta, ratio) > rng.uniform();
                                    draws = rng.draws;
                                }
                                if (mirror) vec = reflect(unit, N); else vec = refract(unit, N, ratio);
                                mode = MODE_FINAL;
                            } else {
                                bool metal_lobe = mat == 3;
                                if (mat == 5) {                                     // glossy picks its lobe first, kernel.cu:885
                                    const uint32_t xy = __float_as_uint(a4.w);
                                    PathRng rng;
                                    rng.init(fp.seed, xy & 0xFFFFu, xy >> 16, fp.sample_base + (pid >> 5) % fp.samples, draws);
                                    metal_lobe = rng.uniform() > 0.8f;
                                    draws = rng.draws;
                                }
                                if (metal_lobe) { vec = reflect(normalize(raydir), N); mode = MODE_METAL; }     // kernel.cu:875-883, 886-898
                                else { vec = N; mode = (mat == 0 && r2.x != 0.0f) ? MODE_DIFFUSE_UNIT : MODE_DIFFUSE; }   // kernel.cu:848-866, 900-910
                            }
                            rec[REC_HX][slot] = hitpoint.x; rec[REC_HY][slot] = hitpoint.y; rec[REC_HZ][slot] = hitpoint.z;
                            rec[REC_VX][slot] = vec.x; rec[REC_VY][slot] = vec.y; rec[REC_VZ][slot] = vec.z;
                            rec[REC_AR][slot] = atten.x; rec[REC_AG][slot] = atten.y; rec[REC_AB][slot] = atten.z;
                            rec[REC_ROUGH][slot] = rough;
                            rec[REC_PID][slot] = o4.w; rec[REC_XY][slot] = a4.w;
                            rec[REC_DRAWS][slot] = __uint_as_float(draws);
                        }
                    }
                }
            }
            rec[REC_MODE][slot] = __int_as_float(mode);
            nalive += __popc(__ballot_sync(0xffffffffu, mode != MODE_DEAD));
            const unsigned mreq = __ballot_sync(0xffffffffu, mode >= MODE_DIFFUSE);
            if (mode >= MODE_DIFFUSE) req[nreq + __popc(mreq & lt_mask)] = (uint8_t)slot;
            nreq += __popc(mreq);
        }
        if (nalive == 0) continue;                              // warp-uniform
        __syncwarp();
        // ---- stage 2: drain the request pool ------------------------------------------------------------------------------
        if (nreq > 0) {
            int next = 32;                                      // requests [0, 32) start on the lanes; the rest is handed out as lanes finish
            int mine = -1;
            uint32_t x = 0, y = 0, smp = 0, draws = 0, w1 = 0, w2 = 0, w3 = 0;    // w1..w3: the block's words not consumed yet (word 0 always is)
            bool regen = false;
#define DRB_TAKE(r_) do { mine = (int)req[(r_)]; const uint32_t xy_ = __float_as_uint(rec[REC_XY][mine]), pid_ = __float_as_uint(rec[REC_PID][mine]); \
                          x = xy_ & 0xFFFFu; y = xy_ >> 16; smp = fp.sample_base + (pid_ >> 5) % fp.samples; \
                          draws = __float_as_uint(rec[REC_DRAWS][mine]); regen = (draws & 3u) != 0u; } while (0)
            if ((int)lane < nreq) DRB_TAKE(lane);
            for (;;) {
                if (mine >= 0) {
                    const uint32_t ph = draws & 3u;
                    uint32_t n0 = 0, n1 = 0, n2 = 0, n3 = 0;
                    if (regen || ph != 1u) {                    // the block the stream resumes in, or the next one
                        const Philox4 p = philox4x32_10((uint32_t)fp.seed, (uint32_t)(fp.seed >> 32), x, y, smp, regen ? (draws >> 2) : ((draws + 3u) >> 2));
                        n0 = p.v[0]; n1 = p.v[1]; n2 = p.v[2]; n3 = p.v[3];
                    }
                    bool attempt = true;
                    if (regen) { w1 = n1; w2 = n2; w3 = n3; regen = false; attempt = (ph == 1u); }
                    if (attempt) {
                        // words draws, draws + 1, draws + 2 (PathRng::words3); the FIRST lands in the LAST component (see the sampling helpers)
                        const uint32_t wc = ph == 0u ? n0 : (ph == 1u ? w1 : (ph == 2u ? w2 : w3));
                        const uint32_t wb = ph == 0u ? n1 : (ph == 1u ? w2 : (ph == 2u ? w3 : n0));
                        const uint32_t wa = ph == 0u ? n2 : (ph == 1u ? w3 : (ph == 2u ? n0 : n1));
                        if (ph != 1u) { w1 = n1; w2 = n2; w3 = n3; }
                        draws += 3u;
                        const f3 p = mk3(PathRng::to_uniform(wa) * 2.0f - 1.0f, PathRng::to_uniform(wb) * 2.0f - 1.0f, PathRng::to_uniform(wc) * 2.0f - 1.0f);
                        if (!(dot(p, p) >= 1.0f)) {
                            rec[REC_SX][mine] = p.x; rec[REC_SY][mine] = p.y; rec[REC_SZ][mine] = p.z;
                            rec[REC_DRAWS][mine] = __uint_as_float(draws);
                            mine = -1;
                        }
                    }
                }
                const unsigned mfree = __ballot_sync(0xffffffffu, mine < 0);
                if (next < nreq) {                              // warp-uniform
                    if (mine < 0) {
                        const int r = next + __popc(mfree & lt_mask);
                        if (r < nreq) DRB_TAKE(r);
                    }
                    next += __popc(mfree);
                } else if (__popc(~mfree) <= kShadeTeamAt) break;   // the pool is dry and few requests are left: finish them in teams
            }
#undef DRB_TAKE
            // The tail.  The last requests would run alone for several more attempts; instead every one of them gets a
            // TEAM of lanes: helper h of a team generates block (draws >> 2) + h of the request's stream, borrows the first
            // two words of its right neighbour's block, and tries every attempt that STARTS in its block (attempt a starts at
            // word draws + 3 a).  The attempts of a team cover the stream in order, so the first accepting helper holds
            // exactly the sample the one-lane loop would have found, and writes it.
            unsigned act = __ballot_sync(0xffffffffu, mine >= 0);
            while (act) {
                const int u = __popc(act);
                const int tshift = u > 4 ? 2 : (u > 2 ? 3 : (u > 1 ? 4 : 5));          // team size 4, 8, 16 or 32 lanes
                const int tsize = 1 << tshift;
                const int j = (int)lane >> tshift, h = (int)lane & (tsize - 1);
                const bool serving = j < u;
                const int owner = (int)__fns(act, 0u, (serving ? j : 0) + 1);             // the j-th open request sits on this lane
                const uint32_t ox = __shfl_sync(0xffffffffu, x, owner), oy = __shfl_sync(0xffffffffu, y, owner);
                const uint32_t os = __shfl_sync(0xffffffffu, smp, owner), od = __shfl_sync(0xffffffffu, draws, owner);
                const int oslot = __shfl_sync(0xffffffffu, mine, owner);
                const uint32_t blk = (od >> 2) + (uint32_t)h;
                const Philox4 pb = philox4x32_10((uint32_t)fp.seed, (uint32_t)(fp.seed >> 32), ox, oy, os, blk);
                const uint32_t m0 = __shfl_down_sync(0xffffffffu, pb.v[0], 1), m1 = __shfl_down_sync(0xffffffffu, pb.v[1], 1);
                const bool has_next = h + 1 < tsize;
                const uint32_t base = blk << 2;
                uint32_t first;                                                             // offset in my block of the first attempt starting there
                if (h == 0) first = od & 3u; else { const uint32_t r = (base - od) % 3u; first = r ? 3u - r : 0u; }
                const uint32_t a0 = first == 0u ? pb.v[0] : (first == 1u ? pb.v[1] : (first == 2u ? pb.v[2] : pb.v[3]));
                const uint32_t a1 = first == 0u ? pb.v[1] : (first == 1u ? pb.v[2] : (first == 2u ? pb.v[3] : m0));
                const uint32_t a2 = first == 0u ? pb.v[2] : (first == 1u ? pb.v[3] : (first == 2u ? m0 : m1));
                const f3 pa = mk3(PathRng::to_uniform(a2) * 2.0f - 1.0f, PathRng::to_uniform(a1) * 2.0f - 1.0f, PathRng::to_uniform(a0) * 2.0f - 1.0f);
                const bool acc_a = serving && (first < 2u || has_next) && !(dot(pa, pa) >= 1.0f);
                // a second attempt starts at word 3 of my block when the first one started at word 0
                const f3 pc = mk3(PathRng::to_uniform(m1) * 2.0f - 1.0f, PathRng::to_uniform(m0) * 2.0f - 1.0f, PathRng::to_uniform(pb.v[3]) * 2.0f - 1.0f);
                const bool acc_c = serving && first == 0u && has_next && !(dot(pc, pc) >= 1.0f);
                const unsigned macc = __ballot_sync(0xffffffffu, acc_a || acc_c);
                const unsigned team = tsize == 32 ? 0xffffffffu : (((1u << tsize) - 1u) << (j << tshift));
                if ((acc_a || acc_c) && (macc & team & lt_mask) == 0u) {                    // the first accepting helper of its team
                    const f3 pw = acc_a ? pa : pc;
                    rec[REC_SX][oslot] = pw.x; rec[REC_SY][oslot] = pw.y; rec[REC_SZ][oslot] = pw.z;
                    rec[REC_DRAWS][oslot] = __uint_as_float(base + (acc_a ? first : 3u) + 3u);
                }
                if (mine >= 0) {
                    const int myj = __popc(act & lt_mask);
                    const unsigned myteam = tsize == 32 ? 0xffffffffu : (((1u << tsize) - 1u) << (myj << tshift));
                    if (macc & myteam) mine = -1;
                    else draws += 3u * (((uint32_t)(4 << tshift) - (draws & 3u)) / 3u);     // every attempt inside the team's blocks was rejected
                }
                act = __ballot_sync(0xffffffffu, mine >= 0);
            }
            __syncwarp();
        }
        // ---- stage 3: finish and append in ray order ---------------------------------------------------------------------------
        uint32_t dst0 = 0;
        if (lane == 0) dst0 = atomicAdd(&counters[cur ^ 1], (uint32_t)nalive);
        dst0 = __shfl_sync(0xffffffffu, dst0, 0);
#pragma unroll 1
        for (int g = 0; g < kShadeGroups; ++g) {
            const int slot = g * 32 + (int)lane;
            const int mode = __float_as_int(rec[REC_MODE][slot]);
            const unsigned malive = __ballot_sync(0xffffffffu, mode != MODE_DEAD);
            if (mode != MODE_DEAD) {
                const f3 hp = mk3(rec[REC_HX][slot], rec[REC_HY][slot], rec[REC_HZ][slot]);
                const f3 vec = mk3(rec[REC_VX][slot], rec[REC_VY][slot], rec[REC_VZ][slot]);
                f3 ndir = vec;
                if (mode >= MODE_DIFFUSE) {
                    const f3 rs = mk3(rec[REC_SX][slot], rec[REC_SY][slot], rec[REC_SZ][slot]);
                    if (mode == MODE_METAL) ndir = vec + mk3(rec[REC_ROUGH][slot]) * rs;
                    else {
                        f3 target = hp + vec;
                        if (mode == MODE_DIFFUSE) target = target + rs; else target = target + normalize(rs);
                        ndir = normalize(target - hp);
                    }
                }
                const uint32_t dst = dst0 + (uint32_t)__popc(malive & lt_mask);
                ro_next[dst] = make_float4(hp.x, hp.y, hp.z, rec[REC_PID][slot]);
                rdv_next[dst] = make_float4(ndir.x, ndir.y, ndir.z, rec[REC_DRAWS][slot]);
                thr_next[dst] = make_float4(rec[REC_AR][slot], rec[REC_AG][slot], rec[REC_AB][slot], rec[REC_XY][slot]);
            }
            dst0 += (uint32_t)__popc(malive);
        }
        __syncwarp();                                           // the records are rewritten by the next iteration
    }
    // ray statistics: one 64-bit atomic per warp
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) local_rays += __shfl_xor_sync(0xffffffffu, local_rays, off);
    if (lane == 0 && local_rays) atomicAdd(reinterpret_cast<unsigned long long*>(&counters[CNT_RAYS]), (unsigned long long)local_rays);
}

// counters for the next bounce: clear the queue that k_shade is about to fill and the trace ticket
__global__ void k_prepare(uint32_t* counters, int clear_queue, int set_queue, uint32_t set_value)
{
    if (threadIdx.x == 0) {
        if (clear_queue >= 0) counters[clear_queue] = 0u;
        if (set_queue >= 0) counters[set_queue] = set_value;
        counters[CNT_TICKET] = 0u;
        counters[CNT_SHADE_TICKET] = 0u;
    }
}

__global__ void __launch_bounds__(256) k_resolve(FrameParams fp, const float4* __restrict__ contrib, float* __restrict__ accum, int accumulate)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= fp.W || y >= fp.H) return;
    const uint32_t gtile = (uint32_t)(y >> 2) * (uint32_t)fp.tiles_x + (uint32_t)(x >> 3);
    if (gtile % fp.tile_count != fp.tile_rank) return;                              // another shard's pixel: left untouched
    const uint32_t tile = gtile / fp.tile_count;
    const uint32_t lane = (uint32_t)((y & 3) * 8 + (x & 7));
    // One running sum per pixel, continued from what is already there: the value depends on the sample range only,
    // not on how it was cut into wavefront batches, progressive chunks or tile shards (0 + c is c, so a fresh frame
    // is the plain left-to-right sum of the reference).
    float* dst = accum + ((size_t)y * fp.W + x) * 3;
    f3 sum = accumulate ? mk3(dst[0], dst[1], dst[2]) : mk3(0.f);
    for (uint32_t s = 0; s < fp.samples; ++s) {
        const float4 c = contrib[(size_t)(tile * fp.samples + s) * 32u + lane];
        sum = sum + mk3(c.x, c.y, c.z);                              // ColorOutput += raycolor(...), kernel.cu:1076
    }
    dst[0] = sum.x; dst[1] = sum.y; dst[2] = sum.z;
}

// one chunk of a ray query: caller's float3 arrays -> query streams (index in chunk; tmax of an occlusion query in d.w,
// clamped to hit()'s 10000 -- a NaN stays NaN and is never occluded)
__global__ void __launch_bounds__(256) k_load_query(const float* __restrict__ o3, const float* __restrict__ d3, const float* __restrict__ tmax,
                                                     uint32_t n, float4* __restrict__ ro, float4* __restrict__ rdv)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const size_t k = (size_t)i * 3;
    const float tm = tmax ? tmax[i] : kTMax;
    ro[i] = make_float4(o3[k], o3[k + 1], o3[k + 2], __uint_as_float(i));
    rdv[i] = make_float4(d3[k], d3[k + 1], d3[k + 2], tm > kTMax ? kTMax : tm);
}
// closest-hit results of one chunk -> caller's arrays.  (u, v) of a triangle hit is recomputed with intersect_prim's
// operations in its order (same __frcp_rn, same left-associated dot / cross, no contraction in this TU): the values the
// acceptance test used, bit for bit.
__global__ void __launch_bounds__(256) k_store_query(const Prim* __restrict__ prims, const float4* __restrict__ ro, const float4* __restrict__ rdv,
                                                      const uint2* __restrict__ hit, const int32_t* __restrict__ orig, uint32_t n,
                                                      int32_t* __restrict__ ids, float* __restrict__ t, float* __restrict__ uv)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint2 h = hit[i];
    const int p = (int)h.y;
    ids[i] = p >= 0 ? orig[p] : -1;
    if (t) t[i] = __uint_as_float(h.x);
    if (!uv) return;
    float u = 0.0f, v = 0.0f;
    if (p >= 0) {
        const float4 pa = prims[p].a;
        if (__float_as_int(pa.w) == DRB_KIND_TRI) {
            const f3 o = xyz(ro[i]), d = xyz(rdv[i]);
            const f3 v0 = xyz(pa), e1 = xyz(prims[p].b), e2 = xyz(prims[p].c);
            const f3 hv = cross(d, e2);
            const float a = dot(e1, hv);
            const float f = __frcp_rn(a);
            const f3 sv = o - v0;
            u = f * dot(sv, hv);
            const f3 qv = cross(sv, e1);
            v = f * dot(d, qv);
        }
    }
    uv[2 * (size_t)i] = u;
    uv[2 * (size_t)i + 1] = v;
}
// camera rays of queue 0 (slot order) -> row-major arrays
__global__ void k_store_rays(FrameParams fp, uint32_t nslots, Queues q, float* __restrict__ o3, float* __restrict__ d3)
{
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= nslots) return;
    int x, y; uint32_t s;
    if (!slot_to_pixel(fp, slot, x, y, s)) return;
    const float4 o = q.ray_o[0][slot], d = q.ray_d[0][slot];
    const size_t k = ((size_t)y * fp.W + x) * 3;
    o3[k] = o.x; o3[k+1] = o.y; o3[k+2] = o.z;
    d3[k] = d.x; d3[k+1] = d.y; d3[k+2] = d.z;
}

__global__ void k_tonemap(const float* __restrict__ accum, size_t n, float scale, uint8_t* __restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = accum[i] * 255.0f * scale;
    const int qv = (v != v) ? 0 : (v >= 255.0f ? 255 : (v <= 0.0f ? 0 : (int)v));
    out[i] = (uint8_t)qv;
}

// Kernel's integer output (kernel.cu:1083-1085) from a float sum: out[x*H + y] = trunc(sum * 255 * (1/spp))
__global__ void k_frame_i3(const float* __restrict__ accum, int w, int h, int full_h, float scale, int32_t* __restrict__ out)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const float* src = accum + ((size_t)y * w + x) * 3;
    int32_t* dst = out + ((size_t)x * full_h + y) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float v = src[c] * 255.0f * scale;
        dst[c] = (v != v) ? 0 : (v >= 2147483648.0f ? INT32_MAX : (v <= -2147483648.0f ? INT32_MIN : (int32_t)v));
    }
}

} // namespace

// ---- host side ---------------------------------------------------------------------------------------
struct RenderBuffers {
    size_t capacity = 0;                // path slots
    DevArray<float4> ray_o[2], ray_d[2], thr[2], contrib;
    DevArray<uint2> hit;
    DevArray<uint32_t> counters;
    int trace_blocks = 0, shade_blocks = 0;
    size_t trace_smem = 0;              // dynamic shared memory of k_trace: (tree height + 2) stack levels x 128 lanes
    Queues queues() const
    {
        return Queues{ { ray_o[0].get(), ray_o[1].get() }, { ray_d[0].get(), ray_d[1].get() }, { thr[0].get(), thr[1].get() }, hit.get(), contrib.get(),
                       counters.get() };
    }
};

// Scratch of the ray-query entry points (drb_trace_ids, drb_trace_device, drb_occluded_device), apart from the render's queues: a query
// never reallocates or overwrites what the next frame uses.  Sized to one chunk of rays (40 B each).
struct QueryBuffers {
    size_t capacity = 0;                // rays per chunk
    DevArray<float4> ray_o, ray_d;
    DevArray<uint2> hit;
    DevArray<uint32_t> counters;
    int trace_blocks = 0, occluded_blocks = 0;
    size_t trace_smem = 0;              // stack of k_trace / k_occluded: (tree height + 2) levels x 128 lanes
    Queues queues() const { return Queues{ { ray_o.get(), nullptr }, { ray_d.get(), nullptr }, {}, hit.get(), nullptr, counters.get() }; }
};

void BuffersDelete::operator()(RenderBuffers* p) const { delete p; }
void BuffersDelete::operator()(QueryBuffers* p) const { delete p; }

namespace {

// Camera basis exactly as Kernel derives it per thread (kernel.cu:1016-1052), once on the host.
Camera make_camera(const drb_settings& st, int W, int H, int divisor)
{
    auto n3 = [](float x, float y, float z, float out[3]) {
        const float inv = 1.0f / sqrtf(x * x + y * y + z * z);
        out[0] = x * inv; out[1] = y * inv; out[2] = z * inv;
    };
    const float div = (float)divisor;
    Camera c;
    c.wdiv = (float)((float)W / div);
    c.hdiv = (float)((float)H / div);
    const float aspect = c.wdiv / c.hdiv;
    const float fov = (float)((double)(float)st.fov * M_PI / 180);
    const float vh = (float)(2.0 * (double)tanf(fov / 2));
    const float vw = aspect * vh;
    float wu[3], uu[3], vu[3];
    n3(st.cam[0] - st.look[0], st.cam[1] - st.look[1], st.cam[2] - st.look[2], wu);
    // cross(vup, wu), vup = (0,1,0)
    const float cx = 1.0f * wu[2] - 0.0f * wu[1], cy = 0.0f * wu[0] - 0.0f * wu[2], cz = 0.0f * wu[1] - 1.0f * wu[0];
    n3(cx, cy, cz, uu);
    vu[0] = wu[1] * uu[2] - wu[2] * uu[1];
    vu[1] = wu[2] * uu[0] - wu[0] * uu[2];
    vu[2] = wu[0] * uu[1] - wu[1] * uu[0];
    float hor[3], ver[3], llc[3];
    for (int a = 0; a < 3; ++a) {
        hor[a] = (st.focus * vw) * uu[a];
        ver[a] = (st.focus * vh) * vu[a];
    }
    for (int a = 0; a < 3; ++a) llc[a] = ((st.cam[a] - hor[a] / 2.0f) - ver[a] / 2.0f) - st.focus * wu[a];
    c.from = f3{ st.cam[0], st.cam[1], st.cam[2] };
    c.llc = f3{ llc[0], llc[1], llc[2] };
    c.horizontal = f3{ hor[0], hor[1], hor[2] };
    c.vertical = f3{ ver[0], ver[1], ver[2] };
    c.uu = f3{ uu[0], uu[1], uu[2] };
    c.vu = f3{ vu[0], vu[1], vu[2] };
    c.lens_radius = st.aperture / 2;
    return c;
}

// SMs x resident blocks per SM of a persistent kernel launched with `threads` per block and `smem` bytes of dynamic shared
// memory (both asked once per process and device, drb_occupancy)
int resident_grid(const void* kernel, int threads, int device, size_t smem, int* blocks)
{
    int sms = 0, per_sm = 0;
    if (int rc = drb_occupancy(kernel, threads, smem, device, &sms, &per_sm)) return rc;
    *blocks = sms * std::max(per_sm, 1);
    return DRB_OK;
}

// one grid for k_trace whichever push order the scene uses: the smaller of the two instantiations' grids
int trace_grid(int device, size_t smem, int* blocks)
{
    int sorted = 0;
    if (int rc = resident_grid((const void*)k_trace<false>, kTraceThreads, device, smem, blocks)) return rc;
    if (int rc = resident_grid((const void*)k_trace<true>, kTraceThreads, device, smem, &sorted)) return rc;
    *blocks = std::min(*blocks, sorted);
    return DRB_OK;
}

// dynamic shared memory of a traversal's stack: the exact bound the collapse computed (pushes along the worst root-to-leaf
// chain + sentinel + 1), not 3 per level, for each of the block's lanes
size_t trace_stack_bytes(const drb_scene* s)
{
    return (size_t)std::max(s->stack_levels, 3) * kTraceThreads * sizeof(int);
}

int ensure_buffers(drb_scene* s, size_t slots)
{
    if (s->rb && s->rb->capacity >= slots) return DRB_OK;
    cudaDeviceSynchronize();                         // renders may have run on caller streams
    s->rb.reset(new RenderBuffers());                // the old buffers go back before the new ones are allocated
    RenderBuffers& rb = *s->rb;
    cudaStream_t st = s->stream;
    for (int k = 0; k < 2; ++k) {
        if (int rc = rb.ray_o[k].alloc(slots, st)) return rc;
        if (int rc = rb.ray_d[k].alloc(slots, st)) return rc;
        if (int rc = rb.thr[k].alloc(slots, st)) return rc;
    }
    if (int rc = rb.hit.alloc(slots, st)) return rc;
    if (int rc = rb.contrib.alloc(slots, st)) return rc;
    if (int rc = rb.counters.alloc(CNT_WORDS, st)) return rc;
    const Queues q = rb.queues();
    if (getenv("DOGERAY_B200_DEBUG"))
        fprintf(stderr, "[dogeray_b200] queues for %zu slots: o %p %p d %p %p thr %p %p hit %p contrib %p\n", slots, (void*)q.ray_o[0], (void*)q.ray_o[1],
                (void*)q.ray_d[0], (void*)q.ray_d[1], (void*)q.thr[0], (void*)q.thr[1], (void*)q.hit, (void*)q.contrib);
    DRB_CUDA(cudaMemsetAsync(q.counters, 0, CNT_WORDS * sizeof(uint32_t), st));
    DRB_CUDA(cudaStreamSynchronize(st));             // the buffers may be used from a caller-provided stream next
    rb.capacity = slots;
    rb.trace_smem = trace_stack_bytes(s);
    if (int rc = trace_grid(s->device, rb.trace_smem, &rb.trace_blocks)) return rc;
    return resident_grid((const void*)k_shade, 128, s->device, 0, &rb.shade_blocks);
}

DevScene dev_scene(const drb_scene* s)
{
    DevScene d;
    for (int a = 0; a < 3; ++a) drb_quant_grid(s->info.bounds_min[a], s->info.bounds_max[a], &d.qlo[a], &d.qscale[a]);
    d.pad_cap = 0.49f * 65527.0f * std::max(d.qscale[0], std::max(d.qscale[1], d.qscale[2]));
    d.wnodes = s->wnodes.get(); d.prims = s->prims.get(); d.recs = s->recs.get(); d.textures = s->textures.get();
    d.nprims = (int)s->nprims; d.ntextures = s->ntextures;
    return d;
}

float scene_scale(const drb_scene* s)
{
    float m = 0.f;
    for (int a = 0; a < 3; ++a) m = std::max(m, std::max(fabsf(s->info.bounds_min[a]), fabsf(s->info.bounds_max[a])));
    return s->nprims ? m : 0.f;
}

int check_settings(const drb_settings* st)
{
    if (!st) { drb_set_error("null settings"); return DRB_ERR_ARG; }
    if (st->width <= 0 || st->height <= 0 || st->width > 32768 || st->height > 32768) { drb_set_error("bad image size %dx%d", st->width, st->height); return DRB_ERR_ARG; }
    if (st->max_depth < 0) { drb_set_error("bad max_depth %d", st->max_depth); return DRB_ERR_ARG; }
    return DRB_OK;
}

// samples per pixel a call traces: opts->sample_count, where 0 means "the settings' spp" unless the caller says it is exact
uint32_t requested_samples(const drb_opts& o, const drb_settings& st)
{
    if (o.sample_count || (o.flags & DRB_FLAG_EXACT_SAMPLES)) return o.sample_count;
    return (uint32_t)std::max(st.spp, 0);
}

// lanes-still-traversing threshold below which a warp refills its idle lanes (tunable for experiments)
int g_refill = []() { const char* e = getenv("DOGERAY_B200_REFILL"); int v = e ? atoi(e) : 24; return v < 0 ? 0 : (v > 33 ? 33 : v); }();

// stashed leaves are intersected when at least g_leaf_batch lanes hold one, or fewer than g_step_min lanes can descend
int g_leaf_batch = []() { const char* e = getenv("DOGERAY_B200_LEAF_BATCH"); int v = e ? atoi(e) : 12; return v < 1 ? 1 : v; }();
int g_step_min = []() { const char* e = getenv("DOGERAY_B200_STEP_MIN"); int v = e ? atoi(e) : 20; return v < 1 ? 1 : v; }();

// the closest-hit kernel for this scene: large scenes push the other hit children far-to-near (see DRB_SORTED_PUSH_FROM)
void launch_trace(const drb_scene* s, int blocks, size_t smem, cudaStream_t stream, const DevScene& sc, float scale, const Queues& q, int cur)
{
    auto kernel = s->nprims >= (int64_t)DRB_SORTED_PUSH_FROM ? k_trace<true> : k_trace<false>;
    kernel<<<blocks, kTraceThreads, smem, stream>>>(sc, scale, q.ray_o[cur], q.ray_d[cur], q.hit, q.counters, cur, g_refill, g_leaf_batch, g_step_min);
}

// rays per chunk of a ray query (DOGERAY_B200_QUERY_CHUNK, default 64 Mi: 2.6 GB of query scratch)
size_t g_query_chunk = []() { const char* e = getenv("DOGERAY_B200_QUERY_CHUNK"); long v = e ? atol(e) : (64L << 20); return (size_t)std::min(std::max(v, 1L), 1L << 30); }();

int ensure_query_buffers(drb_scene* s, size_t rays)
{
    if (s->qb && s->qb->capacity >= rays) return DRB_OK;
    if (s->qb) cudaDeviceSynchronize();              // queries run on caller streams
    s->qb.reset(new QueryBuffers());                 // the old scratch goes back before the new one is allocated
    QueryBuffers* qb = s->qb.get();
    cudaStream_t st = s->stream;
    if (int rc = qb->ray_o.alloc(rays, st)) return rc;
    if (int rc = qb->ray_d.alloc(rays, st)) return rc;
    if (int rc = qb->hit.alloc(rays, st)) return rc;
    if (int rc = qb->counters.alloc(CNT_WORDS, st)) return rc;
    DRB_CUDA(cudaMemsetAsync(qb->counters.get(), 0, CNT_WORDS * sizeof(uint32_t), st));
    DRB_CUDA(cudaStreamSynchronize(st));             // the buffers are used from the caller's stream next
    qb->trace_smem = trace_stack_bytes(s);
    if (int rc = trace_grid(s->device, qb->trace_smem, &qb->trace_blocks)) return rc;
    if (int rc = resident_grid((const void*)k_occluded, kTraceThreads, s->device, qb->trace_smem, &qb->occluded_blocks)) return rc;
    qb->capacity = rays;
    return DRB_OK;
}

// Both ray queries, chunk by chunk on one stream without a host synchronisation: load, set the counters, traverse, store.
// tmax == nullptr with occluded != nullptr: 10000 for every ray.
int run_query(drb_scene* s, const float* o3, const float* d3, const float* tmax, int64_t n, int32_t* ids, float* t, float* uv,
              uint8_t* occluded, void* stream)
{
    DRB_CUDA(cudaSetDevice(s->device));
    const size_t chunk = std::min<size_t>((size_t)n, g_query_chunk);
    if (int rc = ensure_query_buffers(s, chunk)) return rc;
    const QueryBuffers* qb = s->qb.get();
    const Queues q = qb->queues();
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    const DevScene sc = dev_scene(s);
    const float scale = scene_scale(s);
    for (int64_t done = 0; done < n; done += (int64_t)chunk) {
        const uint32_t m = (uint32_t)std::min<int64_t>((int64_t)chunk, n - done);
        const unsigned grid = (m + 255u) / 256u;
        k_load_query<<<grid, 256, 0, st>>>(o3 + 3 * done, d3 + 3 * done, tmax ? tmax + done : nullptr, m, q.ray_o[0], q.ray_d[0]);
        k_prepare<<<1, 32, 0, st>>>(q.counters, -1, 0, m);
        if (occluded) {
            // one byte per ray, written by the traversal itself: there is nothing to map back
            k_occluded<<<qb->occluded_blocks, kTraceThreads, qb->trace_smem, st>>>(sc, scale, q.ray_o[0], q.ray_d[0], occluded + done, q.counters,
                                                                                  g_refill, g_leaf_batch, g_step_min);
        } else {
            launch_trace(s, qb->trace_blocks, qb->trace_smem, st, sc, scale, q, 0);
            k_store_query<<<grid, 256, 0, st>>>(s->prims.get(), q.ray_o[0], q.ray_d[0], q.hit, s->orig_id.get(), m, ids + done, t ? t + done : nullptr,
                                                uv ? uv + 2 * done : nullptr);
        }
    }
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}



struct EventPool {
    std::vector<cudaEvent_t> ev;
    ~EventPool() { for (auto e : ev) cudaEventDestroy(e); }
    cudaEvent_t get() { cudaEvent_t e; cudaEventCreate(&e); ev.push_back(e); return e; }
};

// the wavefront loop for a W x H grid; accum is a device buffer of W*H*3 floats
int render_core(drb_scene* s, const drb_settings* st, const drb_opts* opts, int W, int H, int divisor, float* accum, drb_stats* stats)
{
    const auto t_enter = std::chrono::steady_clock::now();
    drb_opts o; if (opts) o = *opts; else drb_opts_default(&o);
    const uint32_t total_samples = requested_samples(o, *st);
    cudaStream_t stream = o.stream ? (cudaStream_t)o.stream : s->stream;
    DRB_CUDA(cudaSetDevice(s->device));
    if (st->backtex >= s->ntextures) { drb_set_error("settings.backtex %d out of range (scene has %d textures)", st->backtex, s->ntextures); return DRB_ERR_ARG; }

    const int tiles_x = (W + 7) / 8, tiles_y = (H + 3) / 4;
    const uint32_t tile_count = o.tile_count ? o.tile_count : 1u, tile_rank = o.tile_count ? o.tile_rank : 0u;
    if (tile_rank >= tile_count) { drb_set_error("tile_rank %u out of range (tile_count %u)", tile_rank, tile_count); return DRB_ERR_ARG; }
    const size_t tiles_total = (size_t)tiles_x * tiles_y;
    const size_t my_tiles = tiles_total > tile_rank ? (tiles_total - tile_rank + tile_count - 1) / tile_count : 0;
    const size_t slots_per_sample = std::max<size_t>(my_tiles, 1) * 32;
    // Paths in flight per wavefront batch.  The last bounces of a batch hold few rays and run at the latency floor, and
    // every launch has a tail, so bigger batches amortise both (1080p, 256 spp, 1 M triangles: 16 M paths per batch 509 ms
    // per frame, 128 M 424 ms, 531 M -- the whole frame in one batch -- 417 ms).  A path slot costs 120 B of queues; by
    // default a batch may take 40 % of the device memory (B200: 73 GB, 610 M slots).  The samples are then cut into
    // EQUAL batches (no small last one), and the batch is halved on allocation failure.
    size_t want = o.batch_paths;
    if (!want) {
        want = (size_t)128 << 20;
        const size_t device_mem = drb_device_total_mem(s->device);
        if (device_mem) want = std::max<size_t>((size_t)(0.40 * (double)device_mem) / 120, (size_t)1 << 20);
    }
    uint32_t per_batch = 1;
    for (;;) {
        per_batch = (uint32_t)std::max<size_t>(1, want / slots_per_sample);
        per_batch = std::min<uint32_t>(per_batch, std::max<uint32_t>(total_samples, 1u));
        if (slots_per_sample * per_batch >= 0xFFFFFFF0ull) { want /= 2; continue; }
        if (total_samples > per_batch) {
            const uint32_t nbatches = (total_samples + per_batch - 1) / per_batch;
            per_batch = (total_samples + nbatches - 1) / nbatches;
        }
        const int rc = ensure_buffers(s, slots_per_sample * per_batch);
        if (rc == DRB_OK) break;
        if (per_batch == 1) return rc;                  // not even one sample per pixel fits
        cudaGetLastError();                              // out of memory: try half the batch
        want = slots_per_sample * (size_t)(per_batch / 2);
    }
    const RenderBuffers* rb = s->rb.get();
    const Queues q = rb->queues();

    FrameParams fp;
    fp.W = W; fp.H = H; fp.tiles_x = tiles_x; fp.tiles_y = tiles_y; fp.tile_rank = tile_rank; fp.tile_count = tile_count;
    fp.seed = o.seed; fp.backtex = st->backtex; fp.bg_intensity = st->bg_intensity;
    fp.scene_scale = scene_scale(s);
    fp.cam = make_camera(*st, st->width, st->height, divisor);     // aspect and u/v denominators come from the FULL size
    const DevScene sc = dev_scene(s);

    const bool debug = getenv("DOGERAY_B200_DEBUG") != nullptr;
    const auto t_setup = std::chrono::steady_clock::now();
    EventPool pool;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> trace_ev;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    if (stats) {
        ev_begin = pool.get(); ev_end = pool.get();
        DRB_CUDA(cudaMemsetAsync(q.counters + CNT_RAYS, 0, 8, stream));
        DRB_CUDA(cudaEventRecord(ev_begin, stream));
    }
    uint32_t launches = 0, trace_launches = 0;
    const bool accumulate_first = (o.flags & DRB_FLAG_ACCUMULATE) != 0;
    if (total_samples == 0 && !accumulate_first) {
        // an empty share: this call's pixels (its tiles) become 0, everything else stays as it is
        fp.samples = 0; fp.sample_base = o.sample_base;
        dim3 rb_block(32, 8), rb_grid((W + 31) / 32, (H + 7) / 8);
        k_resolve<<<rb_grid, rb_block, 0, stream>>>(fp, q.contrib, accum, 0);
        launches += 1;
    }

    for (uint32_t done = 0; done < total_samples; done += per_batch) {
        fp.samples = std::min(per_batch, total_samples - done);
        fp.sample_base = o.sample_base + done;
        const uint32_t nslots = (uint32_t)(slots_per_sample * fp.samples);
        // no clearing of contrib[]: every path ends exactly once (miss, emissive hit, or black at the depth limit) and
        // writes its slot then; slots of pixels outside the image are never read.  (No bounce at all: everything is black.)
        if (st->max_depth == 0) DRB_CUDA(cudaMemsetAsync(q.contrib, 0, (size_t)nslots * sizeof(float4), stream));
        k_generate<<<(nslots + 255) / 256, 256, 0, stream>>>(fp, nslots, q);
        k_prepare<<<1, 32, 0, stream>>>(q.counters, 1, 0, nslots);
        launches += 2;
        int cur = 0;
        uint32_t live = nslots;
        for (int b = 0; b < st->max_depth; ++b) {
            // The queue size ends the batch early and sizes the shade grid.  Reading it back drains the stream, so it is read
            // every fourth bounce only (queues never grow from one bounce to the next: the last value read is an upper bound).
            if (b > 0 && (b & 3) == 0) {
                DRB_CUDA(cudaMemcpyAsync(&live, q.counters + cur, sizeof live, cudaMemcpyDeviceToHost, stream));
                DRB_CUDA(cudaStreamSynchronize(stream));
                if (live == 0) break;
            }
            if (stats) { auto e0 = pool.get(), e1 = pool.get(); trace_ev.push_back({ e0, e1 }); DRB_CUDA(cudaEventRecord(e0, stream)); }
            launch_trace(s, rb->trace_blocks, rb->trace_smem, stream, sc, fp.scene_scale, q, cur);
            if (stats) DRB_CUDA(cudaEventRecord(trace_ev.back().second, stream));
            k_shade<<<std::min<uint32_t>((uint32_t)rb->shade_blocks, (live + 4u * kShadeRays - 1u) / (4u * kShadeRays)), 128, 0, stream>>>(
                sc, fp, q.ray_o[cur], q.ray_d[cur], q.thr[cur], q.hit, q.ray_o[cur ^ 1], q.ray_d[cur ^ 1], q.thr[cur ^ 1], q.contrib, q.counters, cur,
                b == st->max_depth - 1 ? 1 : 0);
            k_prepare<<<1, 32, 0, stream>>>(q.counters, cur, -1, 0u);
            launches += 3; trace_launches += 1;
            cur ^= 1;
        }
        dim3 rb_block(32, 8), rb_grid((W + 31) / 32, (H + 7) / 8);
        k_resolve<<<rb_grid, rb_block, 0, stream>>>(fp, q.contrib, accum, (accumulate_first || done > 0) ? 1 : 0);
        launches += 1;
    }
    DRB_CUDA(cudaGetLastError());
    if (debug) {
        const double setup_ms = std::chrono::duration<double, std::milli>(t_setup - t_enter).count();
        const double loop_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_setup).count();
        fprintf(stderr, "[dogeray_b200] render_core host time: setup %.2f ms, launch loop %.2f ms\n", setup_ms, loop_ms);
    }
    if (stats) {
        DRB_CUDA(cudaEventRecord(ev_end, stream));
        uint64_t rays = 0;
        DRB_CUDA(cudaMemcpyAsync(&rays, q.counters + CNT_RAYS, 8, cudaMemcpyDeviceToHost, stream));
        DRB_CUDA(cudaStreamSynchronize(stream));
        memset(stats, 0, sizeof *stats);
        stats->paths = tile_count == 1 ? (uint64_t)W * H * total_samples : 0;   // with tile sharding the caller sums paths over shards
        if (tile_count > 1) {
            uint64_t px = 0;
            for (size_t t = tile_rank; t < tiles_total; t += tile_count) {
                const int tx = (int)(t % tiles_x) * 8, ty = (int)(t / tiles_x) * 4;
                px += (uint64_t)std::min(8, W - tx) * (uint64_t)std::min(4, H - ty);
            }
            stats->paths = px * total_samples;
        }
        stats->rays = rays;
        float ms = 0;
        cudaEventElapsedTime(&ms, ev_begin, ev_end); stats->total_ms = ms;
        double tms = 0;
        for (auto& pr : trace_ev) { cudaEventElapsedTime(&ms, pr.first, pr.second); tms += ms; }
        stats->trace_ms = (float)tms;
        stats->trace_launches = trace_launches;
        stats->kernel_launches = launches;
    }
    return DRB_OK;
}

} // namespace

extern "C" {

void drb_opts_default(drb_opts* o)
{
    if (!o) return;
    memset(o, 0, sizeof *o);
}

int drb_render_device(drb_scene* s, const drb_settings* settings, const drb_opts* opts, float* accum_dev, drb_stats* stats)
{
    if (!s || !accum_dev) { drb_set_error("drb_render_device: null argument"); return DRB_ERR_ARG; }
    if (int rc = check_settings(settings)) return rc;
    return render_core(s, settings, opts, settings->width, settings->height, 1, accum_dev, stats);
}

int drb_render(drb_scene* s, const drb_settings* settings, const drb_opts* opts, float* accum_host, drb_stats* stats)
{
    if (!s || !accum_host) { drb_set_error("drb_render: null argument"); return DRB_ERR_ARG; }
    if (int rc = check_settings(settings)) return rc;
    DRB_CUDA(cudaSetDevice(s->device));
    const size_t n = (size_t)settings->width * settings->height * 3;
    drb_opts o; if (opts) o = *opts; else drb_opts_default(&o);
    cudaStream_t stream = o.stream ? (cudaStream_t)o.stream : s->stream;
    DevArray<float> buf;
    StreamDrain drain{ stream };                     // the image goes back to the cache idle, also when the render fails part-way
    if (int rc = buf.alloc(n, stream)) return rc;
    float* d = buf.get();
    // accumulate adds to the caller's values; with tile sharding the pixels of other shards must come back as they were
    if ((o.flags & DRB_FLAG_ACCUMULATE) || o.tile_count > 1) DRB_CUDA(cudaMemcpyAsync(d, accum_host, n * sizeof(float), cudaMemcpyHostToDevice, stream));
    if (int rc = render_core(s, settings, &o, settings->width, settings->height, 1, d, stats)) return rc;
    DRB_CUDA(cudaMemcpyAsync(accum_host, d, n * sizeof(float), cudaMemcpyDeviceToHost, stream));
    DRB_CUDA(cudaStreamSynchronize(stream));
    return DRB_OK;
}

} // extern "C"

// ---- one frame over several handles (devices) from one process ------------------------------------------------------
namespace {

struct ShardParts { const float* p[32]; };

// dst = (accumulate ? dst : 0) + parts[0] + parts[1] + ... in handle order; the parts live on peer devices (NVLink reads)
__global__ void __launch_bounds__(256) k_sum_shards(float* __restrict__ dst, ShardParts parts, int nparts, size_t n, int accumulate)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float v = accumulate ? dst[i] : 0.0f;
    for (int k = 0; k < nparts; ++k) v = v + parts.p[k][i];
    dst[i] = v;
}

thread_local std::vector<float> t_multi_ms;           // per-handle device time of this thread's last drb_render_multi

void add_stats(drb_stats& into, const drb_stats& t)
{
    into.paths += t.paths; into.rays += t.rays;
    into.trace_launches += t.trace_launches; into.kernel_launches += t.kernel_launches;
    into.trace_ms += t.trace_ms; into.total_ms += t.total_ms;
}

// the pre-P2P path: every shard starts from the caller's image in host memory and changes only its own tiles, the shards are
// merged on the host by pixel ownership.  Used when some handle's device cannot reach the first handle's device.
int render_multi_through_host(drb_scene* const* scenes, int nscenes, const drb_settings* settings, const drb_opts& base, float* accum_host,
                              std::vector<drb_stats>& sts)
{
    const int W = settings->width, H = settings->height;
    const size_t n = (size_t)W * H * 3;
    std::vector<std::vector<float>> shard((size_t)nscenes - 1);
    std::vector<int> rcs((size_t)nscenes, DRB_OK);
    std::vector<std::string> errs((size_t)nscenes);
    auto work = [&](int k, float* dst) {
        drb_opts o = base;
        o.flags &= ~(DRB_FLAG_DYNAMIC_TILES | DRB_FLAG_SHARD_SAMPLES);
        o.tile_rank = (uint32_t)k; o.tile_count = (uint32_t)nscenes;
        rcs[(size_t)k] = drb_render(scenes[k], settings, &o, dst, &sts[(size_t)k]);
        if (rcs[(size_t)k] != DRB_OK) errs[(size_t)k] = drb_last_error();       // the message is thread-local
    };
    std::vector<std::thread> pool;
    for (int k = 1; k < nscenes; ++k) {
        shard[(size_t)k - 1].assign(accum_host, accum_host + n);
        pool.emplace_back(work, k, shard[(size_t)k - 1].data());
    }
    work(0, accum_host);                                                        // shard 0 renders in place
    for (auto& th : pool) th.join();
    for (int k = 0; k < nscenes; ++k)
        if (rcs[(size_t)k] != DRB_OK) { drb_set_error("drb_render_multi: scene %d: %s", k, errs[(size_t)k].c_str()); return rcs[(size_t)k]; }
    const int tiles_x = (W + 7) / 8;
    for (int y = 0; y < H; ++y)
        for (int tx = 0; tx < tiles_x; ++tx) {
            const uint32_t owner = ((uint32_t)(y >> 2) * (uint32_t)tiles_x + (uint32_t)tx) % (uint32_t)nscenes;
            if (owner == 0) continue;
            const size_t at = ((size_t)y * W + (size_t)tx * 8) * 3;
            const size_t len = (size_t)std::min(8, W - tx * 8) * 3;
            memcpy(accum_host + at, shard[owner - 1].data() + at, len * sizeof(float));
        }
    return DRB_OK;
}

} // namespace

extern "C" int drb_render_multi_times(float* ms, int n)
{
    for (int k = 0; k < n && k < (int)t_multi_ms.size(); ++k) ms[k] = t_multi_ms[(size_t)k];
    return (int)t_multi_ms.size();
}

extern "C" int drb_render_multi(drb_scene* const* scenes, int nscenes, const drb_settings* settings, const drb_opts* opts, float* accum_host, drb_stats* stats)
{
    if (!scenes || nscenes < 1 || !accum_host) { drb_set_error("drb_render_multi: bad argument"); return DRB_ERR_ARG; }
    for (int k = 0; k < nscenes; ++k)
        if (!scenes[k]) { drb_set_error("drb_render_multi: scene %d is null", k); return DRB_ERR_ARG; }
    if (int rc = check_settings(settings)) return rc;
    drb_opts base; if (opts) base = *opts; else drb_opts_default(&base);
    if (base.stream) { drb_set_error("drb_render_multi: opts->stream must be NULL (each handle renders on its own stream)"); return DRB_ERR_ARG; }
    const bool by_samples = (base.flags & DRB_FLAG_SHARD_SAMPLES) != 0, dynamic = (base.flags & DRB_FLAG_DYNAMIC_TILES) != 0 && !by_samples;
    if (by_samples && nscenes > 32) { drb_set_error("drb_render_multi: at most 32 handles with DRB_FLAG_SHARD_SAMPLES"); return DRB_ERR_ARG; }
    t_multi_ms.assign((size_t)nscenes, 0.0f);
    std::vector<drb_stats> sts((size_t)nscenes);
    for (auto& t : sts) memset(&t, 0, sizeof t);
    auto finish_stats = [&]() {
        if (stats) memset(stats, 0, sizeof *stats);
        for (int k = 0; k < nscenes; ++k) {
            t_multi_ms[(size_t)k] = sts[(size_t)k].total_ms;
            if (!stats) continue;
            stats->paths += sts[(size_t)k].paths; stats->rays += sts[(size_t)k].rays;
            stats->trace_launches += sts[(size_t)k].trace_launches; stats->kernel_launches += sts[(size_t)k].kernel_launches;
            stats->trace_ms = std::max(stats->trace_ms, sts[(size_t)k].trace_ms);            // the handles run side by side
            stats->total_ms = std::max(stats->total_ms, sts[(size_t)k].total_ms);
        }
    };
    if (nscenes == 1) {
        base.flags &= ~(DRB_FLAG_DYNAMIC_TILES | DRB_FLAG_SHARD_SAMPLES);
        base.tile_rank = 0; base.tile_count = 1;
        const int rc = drb_render(scenes[0], settings, &base, accum_host, &sts[0]);
        if (rc == DRB_OK) finish_stats();
        return rc;
    }
    const int W = settings->width, H = settings->height;
    const size_t n = (size_t)W * H * 3;
    drb_scene* first = scenes[0];
    const int dev0 = first->device;
    // tiles: every handle's kernels must be able to WRITE the image on dev0; samples: dev0's kernel must READ the parts
    bool peers = true;
    for (int k = 1; k < nscenes; ++k)
        peers = peers && (by_samples ? drb_peer_access(scenes[k]->device, dev0) : drb_peer_access(dev0, scenes[k]->device));
    if (!peers && !by_samples) {
        const int rc = render_multi_through_host(scenes, nscenes, settings, base, accum_host, sts);
        if (rc == DRB_OK) finish_stats();
        return rc;
    }
    DRB_CUDA(cudaSetDevice(dev0));
    DevArray<float> image;                                  // THE image, on the first handle's device
    if (int rc = image.alloc(n, first->stream)) return rc;
    float* d_image = image.get();
    const bool accumulate = (base.flags & DRB_FLAG_ACCUMULATE) != 0;
    if (accumulate) DRB_CUDA(cudaMemcpyAsync(d_image, accum_host, n * sizeof(float), cudaMemcpyHostToDevice, first->stream));
    DRB_CUDA(cudaStreamSynchronize(first->stream));        // the other devices' streams may touch it from here on

    std::vector<int> rcs((size_t)nscenes, DRB_OK);
    std::vector<std::string> errs((size_t)nscenes);
    std::vector<DevArray<float>> parts((size_t)(by_samples ? nscenes : 0));
    std::atomic<uint32_t> next_shard{ 0 };
    const uint32_t nshards = dynamic ? 4u * (uint32_t)nscenes : (uint32_t)nscenes;
    const uint32_t total_samples = requested_samples(base, *settings);
    auto fail = [&](int k, int rc) { rcs[(size_t)k] = rc; errs[(size_t)k] = drb_last_error(); };
    auto work = [&](int k) {
        drb_scene* sc = scenes[k];
        drb_opts o = base;
        o.flags &= ~(DRB_FLAG_DYNAMIC_TILES | DRB_FLAG_SHARD_SAMPLES);
        if (cudaSetDevice(sc->device) != cudaSuccess) { drb_set_error("cudaSetDevice(%d) failed", sc->device); return fail(k, DRB_ERR_CUDA); }
        if (by_samples) {
            // sample range k of nscenes (the same split as distributed.shard_samples), into this device's own buffer
            const uint32_t q = total_samples / (uint32_t)nscenes, r = total_samples % (uint32_t)nscenes;
            o.sample_base = base.sample_base + (uint32_t)k * q + std::min<uint32_t>((uint32_t)k, r);
            o.sample_count = q + ((uint32_t)k < r ? 1u : 0u);
            o.flags = (o.flags & ~DRB_FLAG_ACCUMULATE) | DRB_FLAG_EXACT_SAMPLES;
            o.tile_rank = 0; o.tile_count = 1;
            if (parts[(size_t)k].alloc(n, sc->stream) != DRB_OK) { drb_set_error("out of device memory for a sample shard"); return fail(k, DRB_ERR_NOMEM); }
            if (int rc = render_core(sc, settings, &o, W, H, 1, parts[(size_t)k].get(), &sts[(size_t)k])) return fail(k, rc);
            return;
        }
        // tiles: claim shards (static: exactly shard k) and resolve them straight into the image on dev0
        for (;;) {
            const uint32_t j = dynamic ? next_shard.fetch_add(1u) : (uint32_t)k;
            if (j >= nshards) break;
            o.tile_rank = j; o.tile_count = nshards;
            drb_stats t;
            if (int rc = render_core(sc, settings, &o, W, H, 1, d_image, &t)) return fail(k, rc);
            add_stats(sts[(size_t)k], t);
            if (!dynamic) break;
        }
    };
    {
        std::vector<std::thread> pool;
        for (int k = 1; k < nscenes; ++k) pool.emplace_back(work, k);
        work(0);
        for (auto& th : pool) th.join();
    }
    // the image and the parts go back to the cache idle, also when a handle failed part-way
    for (int k = 0; k < nscenes; ++k)
        if (cudaSetDevice(scenes[k]->device) == cudaSuccess) cudaStreamSynchronize(scenes[k]->stream);
    for (int k = 0; k < nscenes; ++k)
        if (rcs[(size_t)k] != DRB_OK) { drb_set_error("drb_render_multi: scene %d: %s", k, errs[(size_t)k].c_str()); return rcs[(size_t)k]; }
    DRB_CUDA(cudaSetDevice(dev0));
    if (by_samples) {
        if (peers) {
            ShardParts sp;
            for (int k = 0; k < nscenes; ++k) sp.p[k] = parts[(size_t)k].get();
            k_sum_shards<<<(unsigned)((n + 255) / 256), 256, 0, first->stream>>>(d_image, sp, nscenes, n, accumulate ? 1 : 0);
            DRB_CUDA(cudaGetLastError());
            DRB_CUDA(cudaMemcpyAsync(accum_host, d_image, n * sizeof(float), cudaMemcpyDeviceToHost, first->stream));
            DRB_CUDA(cudaStreamSynchronize(first->stream));
        } else {
            // no peer access: the parts come back one by one and are added on the host, in the same order
            std::vector<float> tmp(n);
            for (int k = 0; k < nscenes; ++k) {
                DRB_CUDA(cudaSetDevice(scenes[k]->device));
                DRB_CUDA(cudaMemcpy(tmp.data(), parts[(size_t)k].get(), n * sizeof(float), cudaMemcpyDeviceToHost));
                if (k == 0 && !accumulate) memcpy(accum_host, tmp.data(), n * sizeof(float));
                else for (size_t i = 0; i < n; ++i) accum_host[i] = accum_host[i] + tmp[i];
            }
        }
    } else {
        DRB_CUDA(cudaMemcpyAsync(accum_host, d_image, n * sizeof(float), cudaMemcpyDeviceToHost, first->stream));
        DRB_CUDA(cudaStreamSynchronize(first->stream));
    }
    finish_stats();
    return DRB_OK;
}

extern "C" {

int drb_frame_i3(drb_scene* s, const drb_settings* settings, const drb_opts* opts, int divisor, int32_t* out)
{
    if (!s || !out || divisor < 1) { drb_set_error("drb_frame_i3: bad argument"); return DRB_ERR_ARG; }
    if (int rc = check_settings(settings)) return rc;
    DRB_CUDA(cudaSetDevice(s->device));
    // the grid CudaStarter launches: (W/div/8) x (H/div/8) blocks of 8x8 (kernel.cu:2634-2636)
    const int W = settings->width / divisor / 8 * 8, H = settings->height / divisor / 8 * 8;
    if (W <= 0 || H <= 0) return DRB_OK;
    drb_opts o; if (opts) o = *opts; else drb_opts_default(&o);
    o.flags &= ~DRB_FLAG_ACCUMULATE;
    cudaStream_t stream = o.stream ? (cudaStream_t)o.stream : s->stream;
    const uint32_t spp = requested_samples(o, *settings);
    const size_t nfull = (size_t)settings->width * settings->height * 3;
    DevArray<float> b_acc;
    DevArray<int32_t> b_out;
    StreamDrain drain{ stream };
    if (int rc = b_acc.alloc((size_t)W * H * 3, stream)) return rc;
    if (int rc = b_out.alloc(nfull, stream)) return rc;
    float* d_acc = b_acc.get();
    int32_t* d_out = b_out.get();
    // entries outside the launched grid stay as the caller left them
    DRB_CUDA(cudaMemcpyAsync(d_out, out, nfull * sizeof(int32_t), cudaMemcpyHostToDevice, stream));
    if (int rc = render_core(s, settings, &o, W, H, divisor, d_acc, nullptr)) return rc;
    const float scale = (float)(1.0 / (double)(float)spp);          // kernel.cu:1081
    dim3 block(8, 8), grid(W / 8, H / 8);
    k_frame_i3<<<grid, block, 0, stream>>>(d_acc, W, H, settings->height, scale, d_out);
    DRB_CUDA(cudaGetLastError());
    DRB_CUDA(cudaMemcpyAsync(out, d_out, nfull * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    DRB_CUDA(cudaStreamSynchronize(stream));
    return DRB_OK;
}

int drb_trace_ids(drb_scene* s, const float* o3, const float* d3, int64_t n, int32_t* ids, float* t)
{
    if (!s || n < 0 || (n && (!o3 || !d3 || !ids))) { drb_set_error("drb_trace_ids: bad argument"); return DRB_ERR_ARG; }
    if (n == 0) return DRB_OK;
    if (n >= 0x7FFFFFF0ll) { drb_set_error("too many rays"); return DRB_ERR_ARG; }
    DRB_CUDA(cudaSetDevice(s->device));
    cudaStream_t stream = s->stream;
    DevArray<float> b_o, b_d, b_t;
    DevArray<int32_t> b_ids;
    StreamDrain drain{ stream };
    if (int rc = b_o.alloc((size_t)n * 3, stream)) return rc;
    if (int rc = b_d.alloc((size_t)n * 3, stream)) return rc;
    if (int rc = b_ids.alloc((size_t)n, stream)) return rc;
    if (t) { if (int rc = b_t.alloc((size_t)n, stream)) return rc; }
    DRB_CUDA(cudaMemcpyAsync(b_o.get(), o3, (size_t)n * 12, cudaMemcpyHostToDevice, stream));
    DRB_CUDA(cudaMemcpyAsync(b_d.get(), d3, (size_t)n * 12, cudaMemcpyHostToDevice, stream));
    if (int rc = run_query(s, b_o.get(), b_d.get(), nullptr, n, b_ids.get(), b_t.get(), nullptr, nullptr, nullptr)) return rc;
    DRB_CUDA(cudaMemcpyAsync(ids, b_ids.get(), (size_t)n * 4, cudaMemcpyDeviceToHost, stream));
    if (t) DRB_CUDA(cudaMemcpyAsync(t, b_t.get(), (size_t)n * 4, cudaMemcpyDeviceToHost, stream));
    DRB_CUDA(cudaStreamSynchronize(stream));
    return DRB_OK;
}

int drb_trace_device(drb_scene* s, const float* o3_dev, const float* d3_dev, int64_t n, int32_t* ids_dev, float* t_dev, float* uv_dev, void* stream)
{
    if (!s || n < 0 || (n && (!o3_dev || !d3_dev || !ids_dev))) { drb_set_error("drb_trace_device: bad argument"); return DRB_ERR_ARG; }
    if (n == 0) return DRB_OK;
    return run_query(s, o3_dev, d3_dev, nullptr, n, ids_dev, t_dev, uv_dev, nullptr, stream);
}

int drb_occluded_device(drb_scene* s, const float* o3_dev, const float* d3_dev, const float* tmax_dev, int64_t n, uint8_t* occluded_dev, void* stream)
{
    if (!s || n < 0 || (n && (!o3_dev || !d3_dev || !occluded_dev))) { drb_set_error("drb_occluded_device: bad argument"); return DRB_ERR_ARG; }
    if (n == 0) return DRB_OK;
    return run_query(s, o3_dev, d3_dev, tmax_dev, n, nullptr, nullptr, nullptr, occluded_dev, stream);
}

int drb_primary_rays(drb_scene* s, const drb_settings* settings, const drb_opts* opts, uint32_t sample, float* o3, float* d3)
{
    if (!s || !o3 || !d3) { drb_set_error("drb_primary_rays: null argument"); return DRB_ERR_ARG; }
    if (int rc = check_settings(settings)) return rc;
    DRB_CUDA(cudaSetDevice(s->device));
    const int W = settings->width, H = settings->height;
    FrameParams fp;
    fp.W = W; fp.H = H; fp.tiles_x = (W + 7) / 8; fp.tiles_y = (H + 3) / 4; fp.tile_rank = 0; fp.tile_count = 1;
    fp.samples = 1; fp.sample_base = sample; fp.seed = opts ? opts->seed : 0;
    fp.backtex = -1; fp.bg_intensity = 1; fp.scene_scale = scene_scale(s);
    fp.cam = make_camera(*settings, W, H, 1);
    const size_t nslots = (size_t)fp.tiles_x * fp.tiles_y * 32;
    if (int rc = ensure_buffers(s, nslots)) return rc;
    cudaStream_t stream = s->stream;
    const size_t n = (size_t)W * H * 3;
    DevArray<float> b_o, b_d;
    StreamDrain drain{ stream };
    if (int rc = b_o.alloc(n, stream)) return rc;
    if (int rc = b_d.alloc(n, stream)) return rc;
    float *d_o = b_o.get(), *d_d = b_d.get();
    const Queues q = s->rb->queues();
    k_generate<<<(unsigned)((nslots + 255) / 256), 256, 0, stream>>>(fp, (uint32_t)nslots, q);
    k_store_rays<<<(unsigned)((nslots + 255) / 256), 256, 0, stream>>>(fp, (uint32_t)nslots, q, d_o, d_d);
    DRB_CUDA(cudaGetLastError());
    DRB_CUDA(cudaMemcpyAsync(o3, d_o, n * 4, cudaMemcpyDeviceToHost, stream));
    DRB_CUDA(cudaMemcpyAsync(d3, d_d, n * 4, cudaMemcpyDeviceToHost, stream));
    DRB_CUDA(cudaStreamSynchronize(stream));
    return DRB_OK;
}

int drb_tonemap_device(const float* accum_dev, int width, int height, double nsamples, uint8_t* rgb8_dev, void* stream)
{
    if (!accum_dev || !rgb8_dev || width <= 0 || height <= 0 || !(nsamples > 0)) { drb_set_error("drb_tonemap_device: bad argument"); return DRB_ERR_ARG; }
    const size_t n = (size_t)width * height * 3;
    k_tonemap<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(accum_dev, n, (float)(1.0 / nsamples), rgb8_dev);
    DRB_CUDA(cudaGetLastError());
    return DRB_OK;
}

uint32_t drb_philox_word(uint64_t seed, uint32_t x, uint32_t y, uint32_t sample, uint32_t n)
{
    Philox4 p = philox4x32_10((uint32_t)seed, (uint32_t)(seed >> 32), x, y, sample, n >> 2);
    return p.v[n & 3u];
}

} // extern "C"
