// Device scene construction: upload + GPU LBVH build.  Replaces readtextures, build_bvh and the
// per-frame scene upload inside CudaStarter (raygpu/kernel.cu:1915-1976, 1534-1909, 2604-2629).
//
// The reference builds a median-split tree on the host in ~4 s for 1 M triangles and re-uploads the
// whole scene every frame.  Here the object lines are uploaded once and everything else happens on
// the device:
//   flag renderable objects -> exclusive scan (slot = rank among renderable objects, file order)
//   pack Prim / ShadeRec / bounds per slot, reduce scene bounds (ordered-int atomics)
//   63-bit Morton key of the box centre -> stable radix sort of (key, slot)
//   Karras 2012 hierarchy over the sorted keys (ties broken by position)
//   bottom-up refit with one atomic flag per internal node
//   SAH-guided re-clustering of the sorted leaves, then a breadth-first collapse to 64 B four-wide nodes whose
//   child boxes are quantised to 16 bits on a scene-wide grid (both loops inside cooperative kernels)
// All floating-point steps that feed integer outputs (keys) use single IEEE operations (this TU is
// compiled with -fmad=false), so oracle/lbvh_host.c reproduces keys, order and topology bit-exactly.
#include "drb_internal.h"
#include "device_scene.cuh"

#include <cooperative_groups.h>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <chrono>
#include <cstring>
#include <map>
#include <mutex>
#include <thread>
#include <tuple>
#include <unordered_map>

namespace cg = cooperative_groups;

namespace {

constexpr int kBuildThreads = 256;      // block size of the cooperative build kernels

// what the host needs to know about a finished build, written by the build kernels and read back once
struct BuildCtl {
    int packed;                         // renderable objects k_pack saw (must equal the host scene's count)
    int rounds, ploc_n, error;          // clustering rounds; clusters left; 1 = no progress, 2 = collapse overran
    int nwide, wide_levels, stack_need; // four-wide nodes, their levels, exact bound of traversal pushes
    int height;                         // height of the binary tree the nodes were emitted from
};

__device__ __forceinline__ int float_to_ordered(float f)
{
    int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7FFFFFFF;
}
__host__ __device__ __forceinline__ float ordered_to_float(int i)
{
    int b = i >= 0 ? i : i ^ 0x7FFFFFFF;
#ifdef __CUDA_ARCH__
    return __int_as_float(b);
#else
    float f; memcpy(&f, &b, 4); return f;
#endif
}

__global__ void k_flag(const drb_object* __restrict__ objs, int64_t n, int* __restrict__ flag)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = drb_object_renderable(objs[i]) ? 1 : 0;
}

__global__ void k_init_bounds(int* b)
{
    if (threadIdx.x < 3) b[threadIdx.x] = 0x7FFFFFFF;            // min
    else if (threadIdx.x < 6) b[threadIdx.x] = (int)0x80000000;  // max
}

// One renderable object line -> its primitive and float box (from the vertices, or centre +- |radius|) and the flags of its
// shading record (or-ed into `flags`); pack_rec then makes the record.  The build (k_pack) and the refit (k_refit_check, k_refit_pack) share
// both, so a refitted primitive is bit for bit what a fresh build packs from the same line.
__device__ __forceinline__ void pack_prim(const drb_object& o, Prim& p, uint32_t& flags, float lo[3], float hi[3])
{
    if (o.type == 0) {
        const float r = fabsf(o.dim[0]);
        p.a = make_float4(o.pos[0], o.pos[1], o.pos[2], __int_as_float(DRB_KIND_SPHERE));
        p.b = make_float4(o.dim[0], 0.f, 0.f, 0.f);
        p.c = make_float4(0.f, 0.f, 0.f, 0.f);
        p.d = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int a = 0; a < 3; ++a) { lo[a] = o.pos[a] - r; hi[a] = o.pos[a] + r; }
        flags |= DRB_SF_SPHERE;
    } else {
        p.a = make_float4(o.pos[0], o.pos[1], o.pos[2], __int_as_float(DRB_KIND_TRI));
        p.b = make_float4(o.dim[0] - o.pos[0], o.dim[1] - o.pos[1], o.dim[2] - o.pos[2], 0.f);
        p.c = make_float4(o.rot[0] - o.pos[0], o.rot[1] - o.pos[1], o.rot[2] - o.pos[2], 0.f);
        p.d = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int a = 0; a < 3; ++a) {
            lo[a] = fminf(o.pos[a], fminf(o.dim[a], o.rot[a]));
            hi[a] = fmaxf(o.pos[a], fmaxf(o.dim[a], o.rot[a]));
        }
        const bool face = o.norm[2] != -20.0f;
        const bool smooth = face && o.n1[2] != -20.0f && o.smooth;
        if (face) flags |= DRB_SF_FACE_NORMAL;
        if (smooth) flags |= DRB_SF_SMOOTH;
        if (o.checker) flags |= DRB_SF_CHECKER;
        if (smooth || o.checker || o.texnum >= 0 || o.rtexnum >= 0) flags |= DRB_SF_NEEDS_UV;
    }
}
__device__ __forceinline__ void pack_rec(const drb_object& o, uint32_t flags, ShadeRec& r)
{
    r.r[0] = make_float4(o.norm[0], o.norm[1], o.norm[2], __uint_as_float(flags));
    r.r[1] = make_float4(o.col[0], o.col[1], o.col[2], o.add_y);
    r.r[2] = make_float4(o.add_x, __int_as_float(o.mat), __int_as_float(o.texnum), __int_as_float(o.rtexnum));
    r.r[3] = make_float4(o.n1[0], o.n1[1], o.n1[2], o.t1[0]);
    r.r[4] = make_float4(o.n2[0], o.n2[1], o.n2[2], o.t2[0]);
    r.r[5] = make_float4(o.n3[0], o.n3[1], o.n3[2], o.t3[0]);
    r.r[6] = make_float4(o.t1[1], o.t2[1], o.t3[1], 0.f);
    r.r[7] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// warp-reduce per-lane boxes into the ordered-int scene bounds, one atomic per warp and component
__device__ __forceinline__ void reduce_bounds(const float lo[3], const float hi[3], int* __restrict__ scene_bounds)
{
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        float l = lo[a], h = hi[a];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            l = fminf(l, __shfl_xor_sync(0xffffffffu, l, off));
            h = fmaxf(h, __shfl_xor_sync(0xffffffffu, h, off));
        }
        if ((threadIdx.x & 31) == 0 && l <= h) {
            atomicMin(&scene_bounds[a], float_to_ordered(l));
            atomicMax(&scene_bounds[3 + a], float_to_ordered(h));
        }
    }
}

// one thread per object line
__global__ void k_pack(const drb_object* __restrict__ objs, int64_t n, const int* __restrict__ flag, const int* __restrict__ slot, int nprims,
                       Prim* __restrict__ prims, ShadeRec* __restrict__ recs, int32_t* __restrict__ orig,
                       float4* __restrict__ bmin, float4* __restrict__ bmax, int* __restrict__ scene_bounds, int* __restrict__ packed)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float lo[3] = { 3.0e38f, 3.0e38f, 3.0e38f }, hi[3] = { -3.0e38f, -3.0e38f, -3.0e38f };
    bool live = i < n && flag[i];
    // the arrays were sized from the host's count of renderable objects; the device counts too and the build fails if
    // they disagree (never writes past the arrays)
    const unsigned mlive = __ballot_sync(0xffffffffu, live);
    if ((threadIdx.x & 31) == 0 && mlive) atomicAdd(packed, __popc(mlive));
    if (live && slot[i] >= nprims) live = false;
    if (live) {
        const drb_object o = objs[i];
        const int k = slot[i];
        uint32_t flags = 0;
        Prim p;
        pack_prim(o, p, flags, lo, hi);
        prims[k] = p;
        ShadeRec r;
        pack_rec(o, flags, r);
        recs[k] = r;
        orig[k] = (int32_t)i;
        bmin[k] = make_float4(lo[0], lo[1], lo[2], 0.f);
        bmax[k] = make_float4(hi[0], hi[1], hi[2], 0.f);
    }
    reduce_bounds(lo, hi, scene_bounds);
}

__device__ __forceinline__ uint64_t spread21(uint32_t v)
{
    uint64_t x = v & 0x1FFFFFull;
    x = (x | (x << 32)) & 0x1F00000000FFFFull;
    x = (x | (x << 16)) & 0x1F0000FF0000FFull;
    x = (x | (x << 8)) & 0x100F00F00F00F00Full;
    x = (x | (x << 4)) & 0x10C30C30C30C30C3ull;
    x = (x | (x << 2)) & 0x1249249249249249ull;
    return x;
}

// 63-bit Morton key of the box centre, 21 bits per axis, x most significant
__global__ void k_keys(const float4* __restrict__ bmin, const float4* __restrict__ bmax, int n, const int* __restrict__ scene_bounds,
                       uint64_t* __restrict__ keys, int32_t* __restrict__ idx)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 lo = bmin[i], hi = bmax[i];
    const float c[3] = { (lo.x + hi.x) * 0.5f, (lo.y + hi.y) * 0.5f, (lo.z + hi.z) * 0.5f };
    uint32_t q[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float slo = ordered_to_float(scene_bounds[a]), shi = ordered_to_float(scene_bounds[3 + a]);
        const float clo = slo, chi = shi;
        float ext = chi - clo;
        if (!(ext > 0.0f)) ext = 1.0f;
        float x = ((c[a] - clo) / ext) * 2097152.0f;
        x = fminf(fmaxf(x, 0.0f), 2097151.0f);
        q[a] = (uint32_t)x;
    }
    keys[i] = (spread21(q[0]) << 2) | (spread21(q[1]) << 1) | spread21(q[2]);
    idx[i] = i;
}

__global__ void k_gather(const int32_t* __restrict__ order, int n, const Prim* __restrict__ prims_u, const ShadeRec* __restrict__ recs_u,
                         const int32_t* __restrict__ orig_u, const float4* __restrict__ bmin_u, const float4* __restrict__ bmax_u,
                         Prim* __restrict__ prims, ShadeRec* __restrict__ recs, int32_t* __restrict__ orig,
                         float4* __restrict__ lmin, float4* __restrict__ lmax)
{
    // 8 threads move one primitive: 4 + 8 float4 of payload
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    int k = t >> 3, part = t & 7;
    if (k >= n) return;
    const int src = order[k];
    const float4* rs = reinterpret_cast<const float4*>(recs_u + src);
    float4* rd = reinterpret_cast<float4*>(recs + k);
    rd[part] = rs[part];
    if (part < 4) {
        const float4* ps = reinterpret_cast<const float4*>(prims_u + src);
        float4* pd = reinterpret_cast<float4*>(prims + k);
        pd[part] = ps[part];
    } else if (part == 4) {
        orig[k] = orig_u[src];
    } else if (part == 5) {
        lmin[k] = bmin_u[src];
    } else if (part == 6) {
        lmax[k] = bmax_u[src];
    }
}

// common-prefix length of sorted positions i and j; ties on the key fall back to the position
__device__ __forceinline__ int delta(const uint64_t* __restrict__ keys, int n, int i, int j)
{
    if (j < 0 || j >= n) return -1;
    const uint64_t a = keys[i], b = keys[j];
    if (a != b) return __clzll((long long)(a ^ b));
    return 64 + __clz(i ^ j);
}

// Karras, "Maximizing Parallelism in the Construction of BVHs, Octrees, and k-d Trees", HPG 2012, section 4
__global__ void k_karras(const uint64_t* __restrict__ keys, int n, int32_t* __restrict__ left, int32_t* __restrict__ right,
                         int32_t* __restrict__ parent, int32_t* __restrict__ leaf_parent)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    const int dmin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = delta(keys, n, i, j);
    int s = 0;
    for (int t = (l + 1) >> 1; ; t = (t + 1) >> 1) {
        if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
        if (t <= 1) break;
    }
    const int gamma = i + s * d + min(d, 0);
    const int lo = min(i, j), hi = max(i, j);
    const int lc = (lo == gamma) ? ~gamma : gamma;
    const int rc = (hi == gamma + 1) ? ~(gamma + 1) : gamma + 1;
    left[i] = lc; right[i] = rc;
    if (lc < 0) leaf_parent[gamma] = i; else parent[gamma] = i;
    if (rc < 0) leaf_parent[gamma + 1] = i; else parent[gamma + 1] = i;
    if (i == 0) parent[0] = -1;
}

// one thread per leaf climbs; the second arrival at a node owns it
__global__ void k_refit(int n, const float4* __restrict__ lmin, const float4* __restrict__ lmax, const int32_t* __restrict__ left,
                        const int32_t* __restrict__ right, const int32_t* __restrict__ parent, const int32_t* __restrict__ leaf_parent,
                        int* __restrict__ visits, float4* node_min, float4* node_max, int* __restrict__ height)
{
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    int node = leaf_parent[k];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(&visits[node], 1) == 0) return;       // first arrival: sibling subtree not ready
        __threadfence();
        const int lc = left[node], rc = right[node];
        const volatile float4* vmin = node_min; const volatile float4* vmax = node_max;
        float4 a0, a1, b0, b1; int ha, hb;
        if (lc < 0) { a0 = lmin[~lc]; a1 = lmax[~lc]; ha = 0; }
        else { a0.x = vmin[lc].x; a0.y = vmin[lc].y; a0.z = vmin[lc].z; a0.w = vmin[lc].w; a1.x = vmax[lc].x; a1.y = vmax[lc].y; a1.z = vmax[lc].z; a1.w = 0; ha = __float_as_int(a0.w); }
        if (rc < 0) { b0 = lmin[~rc]; b1 = lmax[~rc]; hb = 0; }
        else { b0.x = vmin[rc].x; b0.y = vmin[rc].y; b0.z = vmin[rc].z; b0.w = vmin[rc].w; b1.x = vmax[rc].x; b1.y = vmax[rc].y; b1.z = vmax[rc].z; b1.w = 0; hb = __float_as_int(b0.w); }
        const int h = max(ha, hb) + 1;
        node_min[node] = make_float4(fminf(a0.x, b0.x), fminf(a0.y, b0.y), fminf(a0.z, b0.z), __int_as_float(h));   // .w carries the subtree height
        node_max[node] = make_float4(fmaxf(a1.x, b1.x), fmaxf(a1.y, b1.y), fmaxf(a1.z, b1.z), 0.f);
        if (node == 0) *height = h;
        node = parent[node];
    }
}


// ---- SAH-guided rebuild of the hierarchy: agglomerative clustering over the Morton order ---------------
// (Meister & Bittner, "Parallel Locally-Ordered Clustering for BVH Construction", TVCG 2018.)
// The Karras tree above splits where the Morton prefix changes, which ignores surface area; traversal
// of it visits ~1.5x more nodes than a SAH-quality tree.  Starting from the same sorted leaves, every
// cluster looks `radius` positions left and right for the neighbour whose union box has the smallest
// surface area; mutually nearest pairs merge into a new node, the survivors are compacted in order, and
// the process repeats until one cluster is left.  All steps are deterministic (ties go to the lower
// position; node ids come from a prefix sum, not from atomics), so oracle/lbvh_host.c reproduces the
// topology bit for bit.
#ifndef DRB_PLOC_RADIUS
#define DRB_PLOC_RADIUS 16
#endif
constexpr int kPlocRadius = DRB_PLOC_RADIUS;
constexpr int kPlocSoloClusters = 2048;     // from here on one block finishes the clustering (block barriers instead of grid barriers)

__device__ __forceinline__ float union_half_area(const float4& alo, const float4& ahi, const float4& blo, const float4& bhi)
{
    const float ex = fmaxf(ahi.x, bhi.x) - fminf(alo.x, blo.x);
    const float ey = fmaxf(ahi.y, bhi.y) - fminf(alo.y, blo.y);
    const float ez = fmaxf(ahi.z, bhi.z) - fminf(alo.z, blo.z);
    return ex * ey + ey * ez + ez * ex;
}

// block-wide exclusive scan of one 64-bit value per thread (two packed 32-bit counters); every thread also gets the block total
__device__ __forceinline__ unsigned long long block_excl_scan(unsigned long long v, unsigned long long* total)
{
    __shared__ unsigned long long s_warp[kBuildThreads / 32];
    __shared__ unsigned long long s_total;
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    unsigned long long x = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned long long y = __shfl_up_sync(0xffffffffu, x, off);
        if (lane >= (unsigned)off) x += y;
    }
    __syncthreads();                                      // the previous call's readers are done with s_warp / s_total
    if (lane == 31u) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = lane < kBuildThreads / 32 ? s_warp[lane] : 0ull;
#pragma unroll
        for (int off = 1; off < kBuildThreads / 32; off <<= 1) {
            const unsigned long long y = __shfl_up_sync(0xffffffffu, w, off);
            if (lane >= (unsigned)off) w += y;
        }
        if (lane < kBuildThreads / 32) s_warp[lane] = w;              // inclusive over warps
        if (lane == kBuildThreads / 32 - 1) s_total = w;
    }
    __syncthreads();
    *total = s_total;
    return (x - v) + (warp ? s_warp[warp - 1] : 0ull);
}

// The whole clustering loop in ONE cooperative launch (it used to be four launches and a host read-back per round,
// ~43 rounds for a million leaves).  Every block owns a contiguous chunk of the cluster array; a round is
//   A  nearest neighbour of every cluster                                            | grid sync
//   B  survive / merge flags, per-block totals                                       | grid sync
//   C  positions and node ids from (prefix over block totals) + (scan inside block); emit the next cluster array;
//      every block sums all block totals, so all agree on the next n without another exchange | grid sync
// Positions and node ids are the same prefix sums the host mirror computes, so the topology is unchanged bit for bit.
__global__ void __launch_bounds__(kBuildThreads) k_ploc_all(int n0, const float4* __restrict__ lmin, const float4* __restrict__ lmax,
                                                            int32_t* cid0, int32_t* cid1, float4* cmn0, float4* cmn1, float4* cmx0, float4* cmx1,
                                                            int32_t* nn, unsigned long long* f, unsigned long long* blk_tot,
                                                            int32_t* left, int32_t* right, float4* node_min, float4* node_max, BuildCtl* ctl)
{
    cg::grid_group grid = cg::this_grid();
    const int b = (int)blockIdx.x, t = (int)threadIdx.x;
    int32_t* cid[2] = { cid0, cid1 }; float4* cmn[2] = { cmn0, cmn1 }; float4* cmx[2] = { cmx0, cmx1 };
    for (int i = b * kBuildThreads + t; i < n0; i += (int)gridDim.x * kBuildThreads) {
        cid0[i] = ~i;
        float4 lo = lmin[i]; lo.w = 0.f;
        cmn0[i] = lo; cmx0[i] = lmax[i];
    }
    grid.sync();
    int n = n0, node_base = 0, cur = 0, rounds = 0, err = 0;
    // Once few clusters are left (most of the ~60 rounds), block 0 finishes alone: a block barrier costs a fraction of a
    // grid barrier and the work no longer fills more than one block anyway.  The switch depends on n only, which every
    // block knows, so the others leave after the grid barrier that ends their last common round.
    bool solo = false;
    int nb = (int)gridDim.x;
    auto barrier = [&]() { if (solo) __syncthreads(); else grid.sync(); };
    while (n > 1) {
        if (!solo && n <= kPlocSoloClusters) {
            if (b != 0) break;
            solo = true; nb = 1;
        }
        const int chunk = max((n + nb - 1) / nb, kBuildThreads);
        const int c0 = min(n, b * chunk), c1 = min(n, c0 + chunk);
        const float4* cmin = cmn[cur]; const float4* cmax = cmx[cur];
        // A
        for (int i = c0 + t; i < c1; i += kBuildThreads) {
            const float4 lo = cmin[i], hi = cmax[i];
            float best = 3.4e38f; int bj = -1;
            const int j0 = max(0, i - kPlocRadius), j1 = min(n - 1, i + kPlocRadius);
            for (int j = j0; j <= j1; ++j) {
                if (j == i) continue;
                const float a = union_half_area(lo, hi, cmin[j], cmax[j]);
                if (a < best) { best = a; bj = j; }
            }
            if (bj < 0) bj = (i ^ 1) < n ? (i ^ 1) : i - 1;        // non-finite boxes: pair neighbours so the loop still ends
            nn[i] = bj;
        }
        barrier();
        // B: low word = the cluster survives at this position, high word = it is the lower half of a merging pair
        unsigned long long mine = 0ull;
        for (int i = c0 + t; i < c1; i += kBuildThreads) {
            const int j = nn[i];
            const bool mutual = j >= 0 && j < n && nn[j] == i;
            const unsigned long long valid = !(mutual && i > j), merge = (mutual && i < j);
            const unsigned long long fi = valid | (merge << 32);
            f[i] = fi;
            mine += fi;
        }
        unsigned long long tot;
        block_excl_scan(mine, &tot);
        if (t == 0) blk_tot[b] = tot;
        barrier();
        // C
        unsigned long long before = 0ull, all = 0ull;
        for (int k = t; k < nb; k += kBuildThreads) { const unsigned long long v = blk_tot[k]; all += v; if (k < b) before += v; }
        { unsigned long long sum; block_excl_scan(all, &sum); all = sum; block_excl_scan(before, &sum); before = sum; }
        unsigned long long running = before;
        for (int base = c0; base < c1; base += kBuildThreads) {
            const int i = base + t;
            const unsigned long long fi = i < c1 ? f[i] : 0ull;
            unsigned long long tile;
            const unsigned long long si = running + block_excl_scan(fi, &tile);
            running += tile;
            if (fi & 1ull) {
                const int pos = (int)(uint32_t)si;
                if (fi >> 32) {
                    const int j = nn[i];
                    const int node = node_base + (int)(si >> 32);
                    const int a = cid[cur][i], bb = cid[cur][j];
                    const float4 alo = cmin[i], ahi = cmax[i], blo = cmin[j], bhi = cmax[j];
                    const int ha = a < 0 ? 0 : __float_as_int(alo.w), hb = bb < 0 ? 0 : __float_as_int(blo.w);
                    const float4 lo = make_float4(fminf(alo.x, blo.x), fminf(alo.y, blo.y), fminf(alo.z, blo.z), __int_as_float(max(ha, hb) + 1));
                    const float4 hi = make_float4(fmaxf(ahi.x, bhi.x), fmaxf(ahi.y, bhi.y), fmaxf(ahi.z, bhi.z), 0.f);
                    left[node] = a; right[node] = bb;
                    node_min[node] = lo; node_max[node] = hi;
                    cid[cur ^ 1][pos] = node; cmn[cur ^ 1][pos] = lo; cmx[cur ^ 1][pos] = hi;
                } else {
                    cid[cur ^ 1][pos] = cid[cur][i]; cmn[cur ^ 1][pos] = cmin[i]; cmx[cur ^ 1][pos] = cmax[i];
                }
            }
        }
        const int survivors = (int)(uint32_t)all, merges = (int)(all >> 32);
        ++rounds;
        if (merges <= 0 || survivors != n - merges) { err = 1; break; }          // same totals in every block: all leave together
        node_base += merges; n = survivors; cur ^= 1;
        barrier();
    }
    if (b == 0 && t == 0) { ctl->rounds = rounds; ctl->error = err; ctl->ploc_n = n; }
}

// both planes of one axis of a child box -> min_q | max_q << 16, rounded outwards + 1 quantum
__device__ __forceinline__ uint32_t quant_axis(float lo, float hi, float qlo, float qscale)
{
    int a = (int)floorf((lo - qlo) / qscale) - 1;
    int b = (int)ceilf((hi - qlo) / qscale) + 1;
    a = max(0, min(65535, a)); b = max(0, min(65535, b));
    return (uint32_t)a | ((uint32_t)b << 16);
}
__device__ __forceinline__ void quant_child(const float4& lo, const float4& hi, const int* __restrict__ scene_bounds, uint32_t out[3])
{
    const float l[3] = { lo.x, lo.y, lo.z }, h[3] = { hi.x, hi.y, hi.z };
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        float qlo, qs;
        drb_quant_grid(ordered_to_float(scene_bounds[a]), ordered_to_float(scene_bounds[3 + a]), &qlo, &qs);
        out[a] = quant_axis(l[a], h[a], qlo, qs);
    }
}

// final labelling: node created k-th becomes (n - 2) - k, so the root is node 0 and parents precede children
__global__ void k_relabel(int n, const int32_t* __restrict__ left,
                                  const int32_t* __restrict__ right, const float4* __restrict__ node_min, const float4* __restrict__ node_max,
                                  int32_t* __restrict__ fleft, int32_t* __restrict__ fright, float4* __restrict__ fmin,
                                  float4* __restrict__ fmax)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int lc = left[i], rc = right[i];
    const int dst = (n - 2) - i;
    const int flc = lc < 0 ? lc : (n - 2) - lc, frc = rc < 0 ? rc : (n - 2) - rc;
    fleft[dst] = flc; fright[dst] = frc;
    fmin[dst] = node_min[i]; fmax[dst] = node_max[i];
}

// ---- collapse to four-wide nodes ------------------------------------------------------------------------
// Breadth first over the final binary tree (root = node 0).  A wide node starts from a binary node's two
// children and twice replaces the internal child of largest surface area by that child's own two children
// (ties: lowest slot), giving up to four children.  Ids are assigned level by level from prefix sums, so the
// result is deterministic and oracle/lbvh_host.c reproduces it bit for bit.
__device__ __forceinline__ float box_half_area(const float4& lo, const float4& hi)
{
    const float ex = hi.x - lo.x, ey = hi.y - lo.y, ez = hi.z - lo.z;
    return ex * ey + ey * ez + ez * ex;
}

// The breadth-first collapse in ONE cooperative launch (was: three launches and a host read-back per level).  Per level
//   A  expand every queued binary node into up to four slots, count its internal children, per-block totals | grid sync
//   B  child ids from (prefix over block totals) + (scan inside the block); emit the wide nodes and the next queue | grid sync
// and afterwards, bottom-up over the recorded levels, the exact stack bound of the traversal kernel: visiting a node
// pushes all but one of its children, so need(node) = (children - 1) + max over internal children of need(child).
constexpr int kMaxWideLevels = 512;
__global__ void __launch_bounds__(kBuildThreads) k_wide_all(const int32_t* __restrict__ left, const int32_t* __restrict__ right,
                                                            const float4* __restrict__ node_min, const float4* __restrict__ node_max,
                                                            const float4* __restrict__ lmin, const float4* __restrict__ lmax,
                                                            const int* __restrict__ scene_bounds, int max_nodes,
                                                            int32_t* wq0, int32_t* wq1, int4* slots, int* counts, unsigned long long* blk_tot,
                                                            WideNode* out, int* need, int* level_start, BuildCtl* ctl)
{
    cg::grid_group grid = cg::this_grid();
    __shared__ int s_level_start[kMaxWideLevels + 1];
    const int nb = (int)gridDim.x, b = (int)blockIdx.x, t = (int)threadIdx.x;
    int32_t* wq[2] = { wq0, wq1 };
    if (b == 0 && t == 0) wq0[0] = 0;                               // level 0 = { binary root 0 }
    grid.sync();
    int nq = 1, level_base = 0, cur = 0, levels = 0, err = 0;
    while (nq > 0) {
        if (levels >= kMaxWideLevels || level_base + nq > max_nodes) { err = 2; break; }
        if (t == 0) s_level_start[levels] = level_base;
        const int chunk = max((nq + nb - 1) / nb, kBuildThreads);
        const int c0 = min(nq, b * chunk), c1 = min(nq, c0 + chunk);
        // A
        unsigned long long mine = 0ull;
        for (int i = c0 + t; i < c1; i += kBuildThreads) {
            const int bn = wq[cur][i];
            int s[4] = { left[bn], right[bn], DRB_WIDE_EMPTY, DRB_WIDE_EMPTY };
            int n = 2;
            for (int it = 0; it < 2; ++it) {
                int pick = -1; float best = -1.0f;
                for (int k = 0; k < n; ++k)
                    if (s[k] >= 0) {
                        const float a = box_half_area(node_min[s[k]], node_max[s[k]]);
                        if (a > best) { best = a; pick = k; }
                    }
                if (pick < 0) break;
                const int c = s[pick];
                s[pick] = left[c];
                s[n++] = right[c];
            }
            int internal = 0;
            for (int k = 0; k < 4; ++k) internal += (s[k] >= 0) ? 1 : 0;
            slots[i] = make_int4(s[0], s[1], s[2], s[3]);
            counts[i] = internal;
            mine += (unsigned long long)internal;
        }
        unsigned long long tot;
        block_excl_scan(mine, &tot);
        if (t == 0) blk_tot[b] = tot;
        grid.sync();
        // B
        unsigned long long before = 0ull, all = 0ull;
        for (int k = t; k < nb; k += kBuildThreads) { const unsigned long long v = blk_tot[k]; all += v; if (k < b) before += v; }
        { unsigned long long sum; block_excl_scan(all, &sum); all = sum; block_excl_scan(before, &sum); before = sum; }
        const int next_base = level_base + nq;
        unsigned long long running = before;
        for (int base = c0; base < c1; base += kBuildThreads) {
            const int i = base + t;
            const unsigned long long ci = i < c1 ? (unsigned long long)counts[i] : 0ull;
            unsigned long long tile;
            const int off = (int)(running + block_excl_scan(ci, &tile));
            running += tile;
            if (i < c1) {
                const int4 s4 = slots[i];
                const int s[4] = { s4.x, s4.y, s4.z, s4.w };
                WideNode nd;
                int j = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    uint32_t q[3] = { 0x0000FFFFu, 0x0000FFFFu, 0x0000FFFFu };          // min 65535 > max 0: never hit
                    int link = DRB_WIDE_EMPTY;
                    if (s[k] != DRB_WIDE_EMPTY) {
                        if (s[k] < 0) { quant_child(lmin[~s[k]], lmax[~s[k]], scene_bounds, q); link = s[k]; }
                        else {
                            quant_child(node_min[s[k]], node_max[s[k]], scene_bounds, q);
                            link = next_base + off + j;
                            wq[cur ^ 1][off + j] = s[k];
                            ++j;
                        }
                    }
                    nd.bx[k] = q[0]; nd.by[k] = q[1]; nd.bz[k] = q[2]; nd.child[k] = link;
                }
                out[level_base + i] = nd;
            }
        }
        level_base += nq; nq = (int)all; cur ^= 1; ++levels;
        grid.sync();
    }
    if (t == 0) s_level_start[min(levels, kMaxWideLevels)] = level_base;
    __syncthreads();
    if (b == 0)                                                     // the level boundaries stay with the scene for refits
        for (int L = t; L <= min(levels, kMaxWideLevels); L += kBuildThreads) level_start[L] = s_level_start[L];
    // exact stack bound, deepest level first (children live on the next level, so they are done)
    if (!err)
        for (int L = levels - 1; L >= 0; --L) {
            const int l0 = s_level_start[L], l1 = s_level_start[L + 1];
            for (int i = l0 + b * kBuildThreads + t; i < l1; i += nb * kBuildThreads) {
                int kids = 0, deepest = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int c = out[i].child[k];
                    if (c == DRB_WIDE_EMPTY) continue;
                    ++kids;
                    if (c >= 0) deepest = max(deepest, need[c]);
                }
                need[i] = max(kids - 1, 0) + deepest;
            }
            grid.sync();
        }
    if (b == 0 && t == 0) {
        ctl->nwide = level_base; ctl->wide_levels = levels; ctl->stack_need = err ? 0 : need[0];
        ctl->height = __float_as_int(node_min[0].w);
        if (err) ctl->error = err;
    }
}

__global__ void k_wide_single(const float4* __restrict__ lmin, const float4* __restrict__ lmax, const int* __restrict__ scene_bounds, WideNode* __restrict__ out,
                              int* __restrict__ level_start)
{
    level_start[0] = 0; level_start[1] = 1;
    WideNode nd;
    uint32_t q[3];
    quant_child(lmin[0], lmax[0], scene_bounds, q);
    for (int k = 0; k < 4; ++k) { nd.bx[k] = nd.by[k] = nd.bz[k] = 0x0000FFFFu; nd.child[k] = DRB_WIDE_EMPTY; }
    nd.bx[0] = q[0]; nd.by[0] = q[1]; nd.bz[0] = q[2]; nd.child[0] = ~0;
    out[0] = nd;
}

// ---- refit: new object lines, same tree ----------------------------------------------------------------
// quant_axis is monotone (float subtract, divide by a positive scale, floor / ceil and the clamp each are), so the
// quantised box of a union is the integer union of the quantised boxes: min of the low halves, max of the high halves,
// with an empty slot (min 65535, max 0) neutral.  An internal child's box is therefore the integer union of the four
// boxes of the wide node it links to -- bit for bit what k_wide_all quantises from the float union of the same leaves --
// and the refit never needs the binary tree: leaf boxes on the new grid, then the integer union level by level, deepest
// first.
struct RefitCtl {
    int bounds[6];                      // scene bounds of the new leaf boxes (ordered ints, as in the build)
    unsigned long long bad;             // (first offending line << 2) | reason, ~0 when every line passed
};
constexpr unsigned kRefitKindChanged = 1u, kRefitNonFinite = 2u;
constexpr uint32_t kRefitNoSlot = 0xFFFFFFFFu;

__global__ void k_refit_init(RefitCtl* ctl)
{
    if (threadIdx.x < 3) ctl->bounds[threadIdx.x] = 0x7FFFFFFF;
    else if (threadIdx.x < 6) ctl->bounds[threadIdx.x] = (int)0x80000000;
    else if (threadIdx.x == 6) ctl->bad = ~0ull;
}

// object line -> slot << 1 | (sphere) of its primitive, kRefitNoSlot for lines outside the tree; built once per scene
__global__ void k_refit_inverse(const int32_t* __restrict__ orig, const Prim* __restrict__ prims, int nprims, uint32_t* __restrict__ inv)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < nprims) inv[orig[k]] = ((uint32_t)k << 1) | (__float_as_int(prims[k].a.w) == DRB_KIND_SPHERE ? 1u : 0u);
}

__device__ __forceinline__ bool finite3(const float v[3]) { return isfinite(v[0]) && isfinite(v[1]) && isfinite(v[2]); }

// one thread per object line: validate, leaf box (k_pack's operations) into scratch, scene bounds.  Writes nothing of the
// scene, so a refused refit leaves it as it was.
__global__ void k_refit_check(const drb_object* __restrict__ objs, int64_t n, const uint32_t* __restrict__ inv,
                              float4* __restrict__ lmin, float4* __restrict__ lmax, RefitCtl* __restrict__ ctl)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float lo[3] = { 3.0e38f, 3.0e38f, 3.0e38f }, hi[3] = { -3.0e38f, -3.0e38f, -3.0e38f };
    if (i < n) {
        const drb_object& o = objs[i];
        const uint32_t e = inv[i];
        unsigned bad = 0;
        if (drb_object_renderable(o) != (e != kRefitNoSlot) || (e != kRefitNoSlot && (o.type == 0) != ((e & 1u) != 0)))
            bad = kRefitKindChanged;
        else if (e != kRefitNoSlot) {
            Prim p;
            uint32_t flags = 0;
            pack_prim(o, p, flags, lo, hi);
            const bool ok = o.type == 0 ? finite3(o.pos) && isfinite(o.dim[0]) && finite3(lo) && finite3(hi)
                                        : finite3(o.pos) && finite3(o.dim) && finite3(o.rot);
            if (ok) {
                lmin[e >> 1] = make_float4(lo[0], lo[1], lo[2], 0.f);
                lmax[e >> 1] = make_float4(hi[0], hi[1], hi[2], 0.f);
            } else bad = kRefitNonFinite;
        }
        if (bad) {
            atomicMin(&ctl->bad, ((unsigned long long)i << 2) | bad);
            for (int a = 0; a < 3; ++a) { lo[a] = 3.0e38f; hi[a] = -3.0e38f; }
        }
    }
    reduce_bounds(lo, hi, ctl->bounds);
}

// one thread per object line: primitive and shading record of every line in the tree, once k_refit_check passed them all
__global__ void k_refit_pack(const drb_object* __restrict__ objs, int64_t n, const uint32_t* __restrict__ inv, const RefitCtl* __restrict__ ctl,
                             Prim* __restrict__ prims, ShadeRec* __restrict__ recs)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || ctl->bad != ~0ull) return;
    const uint32_t e = inv[i];
    if (e == kRefitNoSlot) return;
    const drb_object o = objs[i];
    const int k = (int)(e >> 1);
    float lo[3], hi[3];
    uint32_t flags = 0;
    Prim p;
    pack_prim(o, p, flags, lo, hi);
    prims[k] = p;
    ShadeRec r;
    pack_rec(o, flags, r);
    recs[k] = r;
}

// The node boxes in ONE cooperative launch, deepest level first (the shape of k_wide_all's stack-bound pass): a leaf child
// is quantised on the new grid, an internal child is the integer union of its node's four boxes, finished one level down.
__global__ void __launch_bounds__(kBuildThreads) k_refit_wide(const int* __restrict__ level_start, int levels, const float4* __restrict__ lmin,
                                                              const float4* __restrict__ lmax, const RefitCtl* ctl, WideNode* nodes)
{
    cg::grid_group grid = cg::this_grid();
    if (ctl->bad != ~0ull) return;                                  // the same in every block: nobody waits at a barrier
    const int nb = (int)gridDim.x, b = (int)blockIdx.x, t = (int)threadIdx.x;
    for (int L = levels - 1; L >= 0; --L) {
        const int l0 = level_start[L], l1 = level_start[L + 1];
        for (int i = l0 + b * kBuildThreads + t; i < l1; i += nb * kBuildThreads) {
            WideNode nd = nodes[i];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int c = nd.child[k];
                if (c == DRB_WIDE_EMPTY) continue;
                uint32_t q[3];
                if (c < 0) quant_child(lmin[~c], lmax[~c], ctl->bounds, q);
                else {
                    const WideNode& ch = nodes[c];
                    const uint32_t* w[3] = { ch.bx, ch.by, ch.bz };
#pragma unroll
                    for (int a = 0; a < 3; ++a) {
                        uint32_t mn = 0xFFFFu, mx = 0u;
#pragma unroll
                        for (int j = 0; j < 4; ++j) { mn = min(mn, w[a][j] & 0xFFFFu); mx = max(mx, w[a][j] >> 16); }
                        q[a] = mn | (mx << 16);
                    }
                }
                nd.bx[k] = q[0]; nd.by[k] = q[1]; nd.bz[k] = q[2];
            }
            nodes[i] = nd;
        }
        grid.sync();
    }
}

} // namespace

namespace {
struct BlockCache {
    std::mutex mu;
    std::unordered_map<void*, size_t> live;                     // every block handed out -> its size
    std::unordered_map<int, std::unordered_multimap<size_t, void*>> idle;   // device -> (size -> idle blocks)
    std::unordered_map<int, size_t> idle_bytes;
    static constexpr size_t kMaxIdleBytes = size_t(48) << 30;   // beyond this, blocks go back to the pool (and all of them do when an allocation fails)
} g_cache;
}

cudaError_t drb_dev_alloc(void** p, size_t bytes, cudaStream_t st)
{
    int dev = 0;
    cudaGetDevice(&dev);
    if (bytes == 0) bytes = 16;
    {
        std::lock_guard<std::mutex> g(g_cache.mu);
        auto& idle = g_cache.idle[dev];
        auto it = idle.find(bytes);
        if (it != idle.end()) {
            *p = it->second;
            idle.erase(it);
            g_cache.idle_bytes[dev] -= bytes;
            g_cache.live[*p] = bytes;
            return cudaSuccess;
        }
    }
    cudaError_t e = cudaMallocAsync(p, bytes, st);
    if (e == cudaErrorMemoryAllocation) {
        // idle blocks of other sizes may be holding the memory: give them back to the pool and try once more
        cudaGetLastError();
        std::vector<void*> blocks;
        {
            std::lock_guard<std::mutex> g(g_cache.mu);
            for (auto& kv : g_cache.idle[dev]) blocks.push_back(kv.second);
            g_cache.idle[dev].clear();
            g_cache.idle_bytes[dev] = 0;
        }
        if (!blocks.empty()) {
            for (void* b : blocks) cudaFreeAsync(b, st);       // idle blocks are not in use by any stream
            e = cudaMallocAsync(p, bytes, st);
        }
    }
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> g(g_cache.mu);
    g_cache.live[*p] = bytes;
    return cudaSuccess;
}

void drb_dev_free(void* p, cudaStream_t st)
{
    if (!p) return;
    int dev = 0;
    cudaGetDevice(&dev);
    size_t bytes = 0;
    {
        std::lock_guard<std::mutex> g(g_cache.mu);
        auto it = g_cache.live.find(p);
        if (it != g_cache.live.end()) { bytes = it->second; g_cache.live.erase(it); }
        if (bytes && g_cache.idle_bytes[dev] + bytes <= BlockCache::kMaxIdleBytes) {
            g_cache.idle[dev].emplace(bytes, p);
            g_cache.idle_bytes[dev] += bytes;
            return;
        }
    }
    cudaFreeAsync(p, st);
}

namespace {
struct FactsCache {                     // the per-device facts of device_scene.cuh
    std::mutex mu;
    std::map<int, int> sms;
    std::map<int, size_t> total_mem;
    std::map<std::tuple<const void*, int, int, size_t>, int> per_sm;   // (kernel, device, threads, dynamic smem) -> blocks per SM
    std::map<std::pair<const void*, int>, size_t> smem_set;          // (kernel, device) -> dynamic smem limit raised to so far
    std::map<std::pair<int, int>, bool> peer;                          // (owner, accessor) -> usable
} g_facts;
}

size_t drb_device_total_mem(int device)
{
    std::lock_guard<std::mutex> g(g_facts.mu);
    size_t& t = g_facts.total_mem[device];
    if (!t) {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) t = total_b; else cudaGetLastError();
    }
    return t;
}

int drb_occupancy(const void* kernel, int threads, size_t smem, int device, int* sms, int* per_sm)
{
    std::lock_guard<std::mutex> g(g_facts.mu);
    int& n = g_facts.sms[device];
    if (!n) DRB_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device));
    auto it = g_facts.per_sm.find({ kernel, device, threads, smem });
    if (it == g_facts.per_sm.end()) {
        size_t& set = g_facts.smem_set[{ kernel, device }];
        if (smem > set) {
            DRB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            set = smem;
        }
        int b = 0;
        DRB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kernel, threads, smem));
        it = g_facts.per_sm.emplace(std::make_tuple(kernel, device, threads, smem), b).first;
    }
    *sms = n;
    *per_sm = it->second;
    return DRB_OK;
}

bool drb_peer_access(int owner, int accessor)
{
    if (owner == accessor) return true;
    std::lock_guard<std::mutex> g(g_facts.mu);
    auto it = g_facts.peer.find({ owner, accessor });
    if (it != g_facts.peer.end()) return it->second;
    bool ok = false;
    int can = 0;
    if (cudaDeviceCanAccessPeer(&can, accessor, owner) == cudaSuccess && can) {
        // everything here comes from the stream-ordered pool, whose visibility is set per pool ...
        cudaMemPool_t pool;
        cudaMemAccessDesc d;
        memset(&d, 0, sizeof d);
        d.location.type = cudaMemLocationTypeDevice; d.location.id = accessor; d.flags = cudaMemAccessFlagsProtReadWrite;
        ok = cudaDeviceGetDefaultMemPool(&pool, owner) == cudaSuccess && cudaMemPoolSetAccess(pool, &d, 1) == cudaSuccess;
        // ... and classic peer access as well, so that peer copies take the direct NVLink path
        int cur = 0;
        cudaGetDevice(&cur);
        if (cudaSetDevice(accessor) == cudaSuccess) {
            const cudaError_t e = cudaDeviceEnablePeerAccess(owner, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) ok = false;
        }
        cudaSetDevice(cur);
    }
    cudaGetLastError();
    g_facts.peer[{ owner, accessor }] = ok;
    return ok;
}

extern "C" int drb_trim(int device)
{
    DRB_CUDA(cudaSetDevice(device));
    DRB_CUDA(cudaDeviceSynchronize());
    std::vector<void*> blocks;
    {
        std::lock_guard<std::mutex> g(g_cache.mu);
        for (auto& kv : g_cache.idle[device]) blocks.push_back(kv.second);
        g_cache.idle[device].clear();
        g_cache.idle_bytes[device] = 0;
    }
    for (void* p : blocks) DRB_CUDA(cudaFreeAsync(p, nullptr));
    DRB_CUDA(cudaDeviceSynchronize());
    cudaMemPool_t pool;
    DRB_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
    DRB_CUDA(cudaMemPoolTrimTo(pool, 0));
    return DRB_OK;
}

namespace {

int retain_pool(int device)
{
    cudaMemPool_t pool;
    DRB_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t keep = UINT64_MAX;
    DRB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    return DRB_OK;
}

// host-side stage times of a scene creation, printed with DOGERAY_B200_DEBUG set (how create's host overhead is found)
struct StageClock {
    bool on = getenv("DOGERAY_B200_DEBUG") != nullptr;
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    std::string log;
    void mark(const char* what)
    {
        if (!on) return;
        const auto now = std::chrono::steady_clock::now();
        char buf[96];
        snprintf(buf, sizeof buf, " %s %.2f", what, std::chrono::duration<double, std::milli>(now - t).count());
        log += buf; t = now;
    }
    void print(const char* who) { if (on) fprintf(stderr, "[dogeray_b200] %s host ms:%s\n", who, log.c_str()); }
};

struct EventTrio {
    cudaEvent_t e[3] = { nullptr, nullptr, nullptr };
    ~EventTrio() { for (auto x : e) if (x) cudaEventDestroy(x); }
    int create() { for (auto& x : e) DRB_CUDA(cudaEventCreate(&x)); return DRB_OK; }
};

// co-resident grid of a cooperative build kernel, at most max_per_sm blocks per SM: a grid barrier costs more the more
// blocks take part
int coop_grid(int device, const void* kernel, int want_blocks, int max_per_sm, int* blocks)
{
    int sms = 0, per_sm = 0;
    if (int rc = drb_occupancy(kernel, kBuildThreads, 0, device, &sms, &per_sm)) return rc;
    *blocks = std::max(1, std::min(sms * std::max(std::min(per_sm, max_per_sm), 1), want_blocks));
    return DRB_OK;
}

// Upload (unless the object lines are already on the device) + the whole tree build, enqueued on the scene's stream with
// ONE host synchronisation at the end: the number of renderable objects is known on the host (drb_host_scene counts
// them once), and both data-dependent loops -- clustering rounds, collapse levels -- run inside cooperative kernels.
int build_tree(drb_scene* s, const drb_host_scene* hs, const drb_object* objs_dev)
{
    const int64_t nobj = (int64_t)hs->objects.size();
    if (nobj >= (1ll << 31) - 8) { drb_set_error("too many objects (%lld)", (long long)nobj); return DRB_ERR_UNSUPPORTED; }
    cudaStream_t st = s->stream;
    StageClock clk;
    struct PrintOnExit { StageClock& c; ~PrintOnExit() { c.mark("scratch-free"); c.print("build_tree"); } };
    // scratch of the build, declared before `drain` so that the stream has drained when it goes back to the cache
    DevArray<drb_object> up;
    DevArray<int> d_flag, d_slot, d_bounds, d_levels, leaf_parent, visits, d_height, cid[2], nn, pl, pr, wq[2], wcounts, wneed, idx_u, orig_u;
    DevArray<float4> bmin_u, bmax_u, lmin, lmax, cmn[2], cmx[2], pmin, pmax;
    DevArray<unsigned long long> fl, btot, wtot;
    DevArray<uint64_t> keys_u;
    DevArray<BuildCtl> d_ctl;
    DevArray<Prim> prims_u;
    DevArray<ShadeRec> recs_u;
    DevArray<int4> wslots;
    DevArray<char> d_scan, d_sort;
    LbvhDebug dbg; FinalTree tree;                          // moved into the scene with DRB_BUILD_KEEP_DEBUG
    StreamDrain drain{ st };
    PrintOnExit print_on_exit{ clk };                         // destroyed before the scratch: "scratch-free" is then ~0; see drb_scene_create's own clock
    EventTrio ev;
    if (int rc = ev.create()) return rc;
    DRB_CUDA(cudaEventRecord(ev.e[0], st));
    clk.mark("events");

    const bool keep = (s->build_flags & DRB_BUILD_KEEP_DEBUG) != 0;
    const bool lbvh_only = (s->build_flags & DRB_BUILD_LBVH_ONLY) != 0;
    const int nprims = (int)drb_host_scene_num_renderable(hs);
    const drb_object* d_objs = objs_dev;
    if (!d_objs) {
        if (int rc = up.alloc((size_t)nobj, st)) return rc;
        if (nobj) DRB_CUDA(cudaMemcpyAsync(up.get(), hs->objects.data(), (size_t)nobj * sizeof(drb_object), cudaMemcpyHostToDevice, st));
        d_objs = up.get();
    }
    if (int rc = d_flag.alloc((size_t)nobj + 1, st)) return rc;
    if (int rc = d_slot.alloc((size_t)nobj + 1, st)) return rc;
    if (int rc = d_bounds.alloc(8, st)) return rc;
    if (int rc = d_ctl.alloc(1, st)) return rc;
    if (int rc = d_levels.alloc((size_t)kMaxWideLevels + 1, st)) return rc;
    DRB_CUDA(cudaMemsetAsync(d_ctl.get(), 0, sizeof(BuildCtl), st));
    DRB_CUDA(cudaEventRecord(ev.e[1], st));
    clk.mark("upload-enqueue");

    const int T = 256;
    s->nobjects = nobj;
    s->nprims = nprims;
    s->nnodes = nprims == 0 ? 0 : std::max(1, nprims - 1);
    memset(&s->info, 0, sizeof s->info);
    s->info.nprims = nprims; s->info.nnodes = s->nnodes;

    if (int rc = s->prims.alloc((size_t)nprims, st)) return rc;
    if (int rc = s->recs.alloc((size_t)nprims, st)) return rc;
    if (int rc = s->orig_id.alloc((size_t)nprims, st)) return rc;
    const size_t nint = nprims > 1 ? (size_t)nprims - 1 : 1;
    // the integer outputs of the build stay resident only on request (drb_scene_lbvh / drb_scene_tree); otherwise they
    // are scratch: ~100 B per primitive that rendering never reads
    if (int rc = dbg.keys.alloc((size_t)nprims, st)) return rc;
    if (int rc = dbg.order.alloc((size_t)nprims, st)) return rc;
    if (keep || lbvh_only) {
        if (int rc = dbg.parent.alloc(nint, st)) return rc;
        if (int rc = dbg.left.alloc(nint, st)) return rc;
        if (int rc = dbg.right.alloc(nint, st)) return rc;
        if (int rc = dbg.node_min.alloc(nint, st)) return rc;
        if (int rc = dbg.node_max.alloc(nint, st)) return rc;
    }
    if (int rc = tree.left.alloc(nint, st)) return rc;
    if (int rc = tree.right.alloc(nint, st)) return rc;
    if (int rc = tree.node_min.alloc(nint, st)) return rc;
    if (int rc = tree.node_max.alloc(nint, st)) return rc;

    BuildCtl ctl; memset(&ctl, 0, sizeof ctl);
    int hb[6] = { 0, 0, 0, 0, 0, 0 };
    if (nprims > 0) {
        if (int rc = prims_u.alloc((size_t)nprims, st)) return rc;
        if (int rc = recs_u.alloc((size_t)nprims, st)) return rc;
        if (int rc = orig_u.alloc((size_t)nprims, st)) return rc;
        if (int rc = bmin_u.alloc((size_t)nprims, st)) return rc;
        if (int rc = bmax_u.alloc((size_t)nprims, st)) return rc;
        if (int rc = lmin.alloc((size_t)nprims, st)) return rc;
        if (int rc = lmax.alloc((size_t)nprims, st)) return rc;
        if (int rc = keys_u.alloc((size_t)nprims, st)) return rc;
        if (int rc = idx_u.alloc((size_t)nprims, st)) return rc;

        k_flag<<<(unsigned)((nobj + T - 1) / T), T, 0, st>>>(d_objs, nobj, d_flag.get());
        size_t scan_bytes = 0;
        DRB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, d_flag.get(), d_slot.get(), (int)nobj, st));
        if (int rc = d_scan.alloc(scan_bytes, st)) return rc;
        DRB_CUDA(cub::DeviceScan::ExclusiveSum(d_scan.get(), scan_bytes, d_flag.get(), d_slot.get(), (int)nobj, st));
        k_init_bounds<<<1, 32, 0, st>>>(d_bounds.get());
        k_pack<<<(unsigned)((nobj + T - 1) / T), T, 0, st>>>(d_objs, nobj, d_flag.get(), d_slot.get(), nprims, prims_u.get(), recs_u.get(), orig_u.get(),
                                                             bmin_u.get(), bmax_u.get(), d_bounds.get(), &d_ctl.get()->packed);
        k_keys<<<(nprims + T - 1) / T, T, 0, st>>>(bmin_u.get(), bmax_u.get(), nprims, d_bounds.get(), keys_u.get(), idx_u.get());
        size_t sort_bytes = 0;
        DRB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, keys_u.get(), dbg.keys.get(), idx_u.get(), dbg.order.get(), nprims, 0, 63, st));
        if (int rc = d_sort.alloc(sort_bytes, st)) return rc;
        DRB_CUDA(cub::DeviceRadixSort::SortPairs(d_sort.get(), sort_bytes, keys_u.get(), dbg.keys.get(), idx_u.get(), dbg.order.get(), nprims, 0, 63, st));
        {
            const long long threads = (long long)nprims * 8;
            k_gather<<<(unsigned)((threads + T - 1) / T), T, 0, st>>>(dbg.order.get(), nprims, prims_u.get(), recs_u.get(), orig_u.get(), bmin_u.get(),
                                                                      bmax_u.get(), s->prims.get(), s->recs.get(), s->orig_id.get(), lmin.get(), lmax.get());
        }
        if (int rc = s->wnodes.alloc(nint, st)) return rc;
        if (nprims > 1) {
            if (keep || lbvh_only) {
                // the LBVH of north_star: Karras hierarchy + bottom-up refit (the traversal tree only with DRB_BUILD_LBVH_ONLY)
                if (int rc = leaf_parent.alloc((size_t)nprims, st)) return rc;
                if (int rc = visits.alloc(nint, st)) return rc;
                if (int rc = d_height.alloc(1, st)) return rc;
                DRB_CUDA(cudaMemsetAsync(visits.get(), 0, nint * sizeof(int), st));
                DRB_CUDA(cudaMemsetAsync(d_height.get(), 0, sizeof(int), st));
                k_karras<<<(nprims - 1 + T - 1) / T, T, 0, st>>>(dbg.keys.get(), nprims, dbg.left.get(), dbg.right.get(), dbg.parent.get(), leaf_parent.get());
                k_refit<<<(nprims + T - 1) / T, T, 0, st>>>(nprims, lmin.get(), lmax.get(), dbg.left.get(), dbg.right.get(), dbg.parent.get(), leaf_parent.get(),
                                                           visits.get(), dbg.node_min.get(), dbg.node_max.get(), d_height.get());
            }
            if (lbvh_only) {
                DRB_CUDA(cudaMemcpyAsync(tree.left.get(), dbg.left.get(), nint * 4, cudaMemcpyDeviceToDevice, st));
                DRB_CUDA(cudaMemcpyAsync(tree.right.get(), dbg.right.get(), nint * 4, cudaMemcpyDeviceToDevice, st));
                DRB_CUDA(cudaMemcpyAsync(tree.node_min.get(), dbg.node_min.get(), nint * 16, cudaMemcpyDeviceToDevice, st));
                DRB_CUDA(cudaMemcpyAsync(tree.node_max.get(), dbg.node_max.get(), nint * 16, cudaMemcpyDeviceToDevice, st));
            } else {
                // SAH-guided rebuild over the same sorted leaves
                for (int k = 0; k < 2; ++k) {
                    if (int rc = cid[k].alloc((size_t)nprims, st)) return rc;
                    if (int rc = cmn[k].alloc((size_t)nprims, st)) return rc;
                    if (int rc = cmx[k].alloc((size_t)nprims, st)) return rc;
                }
                if (int rc = nn.alloc((size_t)nprims, st)) return rc;
                if (int rc = fl.alloc((size_t)nprims, st)) return rc;
                if (int rc = pl.alloc(nint, st)) return rc;
                if (int rc = pr.alloc(nint, st)) return rc;
                if (int rc = pmin.alloc(nint, st)) return rc;
                if (int rc = pmax.alloc(nint, st)) return rc;
                int blocks = 1;
                if (int rc = coop_grid(s->device, (const void*)k_ploc_all, (nprims + kBuildThreads - 1) / kBuildThreads, 2, &blocks)) return rc;
                if (int rc = btot.alloc((size_t)blocks, st)) return rc;
                int n0 = nprims;
                void* args[] = { &n0, lmin.arg(), lmax.arg(), cid[0].arg(), cid[1].arg(), cmn[0].arg(), cmn[1].arg(), cmx[0].arg(), cmx[1].arg(), nn.arg(),
                                 fl.arg(), btot.arg(), pl.arg(), pr.arg(), pmin.arg(), pmax.arg(), d_ctl.arg() };
                DRB_CUDA(cudaLaunchCooperativeKernel((const void*)k_ploc_all, dim3(blocks), dim3(kBuildThreads), args, 0, st));
                k_relabel<<<(nprims - 1 + T - 1) / T, T, 0, st>>>(nprims, pl.get(), pr.get(), pmin.get(), pmax.get(), tree.left.get(), tree.right.get(),
                                                                 tree.node_min.get(), tree.node_max.get());
            }
            // ---- four-wide collapse of the final tree (tree.*, root 0)
            if (int rc = wq[0].alloc((size_t)nprims, st)) return rc;
            if (int rc = wq[1].alloc((size_t)nprims, st)) return rc;
            if (int rc = wslots.alloc((size_t)nprims, st)) return rc;
            if (int rc = wcounts.alloc((size_t)nprims, st)) return rc;
            if (int rc = wneed.alloc(nint, st)) return rc;
            int blocks = 1;
            if (int rc = coop_grid(s->device, (const void*)k_wide_all, (nprims / 2 + kBuildThreads - 1) / kBuildThreads, 1, &blocks)) return rc;
            if (int rc = wtot.alloc((size_t)blocks, st)) return rc;
            int max_nodes = (int)nint;
            void* args[] = { tree.left.arg(), tree.right.arg(), tree.node_min.arg(), tree.node_max.arg(), lmin.arg(), lmax.arg(), d_bounds.arg(), &max_nodes,
                             wq[0].arg(), wq[1].arg(), wslots.arg(), wcounts.arg(), wtot.arg(), s->wnodes.arg(), wneed.arg(), d_levels.arg(), d_ctl.arg() };
            DRB_CUDA(cudaLaunchCooperativeKernel((const void*)k_wide_all, dim3(blocks), dim3(kBuildThreads), args, 0, st));
        } else {
            k_wide_single<<<1, 1, 0, st>>>(lmin.get(), lmax.get(), d_bounds.get(), s->wnodes.get(), d_levels.get());
        }
        DRB_CUDA(cudaMemcpyAsync(hb, d_bounds.get(), sizeof hb, cudaMemcpyDeviceToHost, st));
        DRB_CUDA(cudaMemcpyAsync(&ctl, d_ctl.get(), sizeof ctl, cudaMemcpyDeviceToHost, st));
    }
    DRB_CUDA(cudaEventRecord(ev.e[2], st));
    clk.mark("build-enqueue");
    DRB_CUDA(cudaStreamSynchronize(st));                     // the one synchronisation of the build
    clk.mark("sync");
    DRB_CUDA(cudaGetLastError());
    if (keep) { s->dbg = std::move(dbg); s->tree = std::move(tree); }
    if (nprims > 0) {
        if (ctl.packed != nprims) { drb_set_error("the device packed %d renderable objects, the host scene counted %d", ctl.packed, nprims); return DRB_ERR_ARG; }
        if (ctl.error == 1) { drb_set_error("hierarchy rebuild made no progress (%d clusters left after %d rounds)", ctl.ploc_n, ctl.rounds); return DRB_ERR_CUDA; }
        if (ctl.error == 2) { drb_set_error("wide collapse overran (%d nodes, level %d)", ctl.nwide, ctl.wide_levels); return DRB_ERR_CUDA; }
        for (int a = 0; a < 3; ++a) { s->info.bounds_min[a] = ordered_to_float(hb[a]); s->info.bounds_max[a] = ordered_to_float(hb[3 + a]); }
        if (nprims > 1) { s->nwnodes = ctl.nwide; s->wide_levels = ctl.wide_levels; s->stack_levels = ctl.stack_need + 2; s->info.max_depth = ctl.height; }
        else { s->nwnodes = 1; s->wide_levels = 1; s->stack_levels = 3; s->info.max_depth = 1; }
        s->info.rebuild_iterations = ctl.rounds;
        s->info.nwide = s->nwnodes; s->info.wide_levels = s->wide_levels; s->info.stack_levels = s->stack_levels;
        if (int rc = s->wide_level_start.alloc((size_t)s->wide_levels + 1, st)) return rc;
        DRB_CUDA(cudaMemcpyAsync(s->wide_level_start.get(), d_levels.get(), ((size_t)s->wide_levels + 1) * sizeof(int), cudaMemcpyDeviceToDevice, st));
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, ev.e[0], ev.e[1]); s->info.upload_ms = ms;
    cudaEventElapsedTime(&ms, ev.e[1], ev.e[2]); s->info.build_ms = ms;
    // the traversal stack lives in shared memory, one column per lane: what limits a scene is that, not the tree height
    if ((size_t)s->stack_levels * 128 * sizeof(int) > (size_t)200 * 1024) {
        drb_set_error("traversal stack of %d levels does not fit in shared memory", s->stack_levels);
        return DRB_ERR_UNSUPPORTED;
    }
    return DRB_OK;
}

int upload_textures(drb_scene* s, const drb_host_scene* hs)
{
    const int nt = (int)hs->tex_paths.size();
    s->ntextures = nt;
    drb_host_scene_summarise(hs);                              // which textures the scene names: one pass per host scene, not per create
    std::vector<char> used((size_t)std::max(nt, 1), 0);
    for (int k = 0; k < nt && k < (int)hs->tex_used.size(); ++k) used[(size_t)k] = hs->tex_used[(size_t)k];
    std::vector<DevTexture> table((size_t)std::max(nt, 1));
    for (int i = 0; i < nt; ++i) {
        table[(size_t)i] = DevTexture{ nullptr, 0, 0 };
        drb_image img;
        int rc = drb_load_ppm(hs->tex_paths[(size_t)i], img);
        if (rc != DRB_OK) {
            if (used[(size_t)i]) return rc;             // a texture the scene names must load
            continue;                                   // the reference loads every .ppm it finds; unused ones may be anything
        }
        s->texture_storage.emplace_back();
        if ((rc = s->texture_storage.back().alloc(img.rgba.size(), s->stream)) != DRB_OK) return rc;
        uint8_t* d = s->texture_storage.back().get();
        DRB_CUDA(cudaMemcpyAsync(d, img.rgba.data(), img.rgba.size(), cudaMemcpyHostToDevice, s->stream));
        DRB_CUDA(cudaStreamSynchronize(s->stream));      // img goes out of scope
        table[(size_t)i] = DevTexture{ (const uchar4*)d, img.w, img.h };
    }
    if (int rc = s->textures.alloc(table.size(), s->stream)) return rc;
    DRB_CUDA(cudaMemcpyAsync(s->textures.get(), table.data(), table.size() * sizeof(DevTexture), cudaMemcpyHostToDevice, s->stream));
    DRB_CUDA(cudaStreamSynchronize(s->stream));
    drb_clear_error();
    return DRB_OK;
}

// New object lines into an existing tree, enqueued on `st` (already ordered after the caller's producer and the scene's
// own stream) with ONE host synchronisation, for the validation result and the new bounds.  Scratch comes from the block
// cache, so repeated refits make no allocator call after the first.
int refit_tree(drb_scene* s, const drb_object* d_objs, cudaStream_t st)
{
    const int64_t nobj = s->nobjects;
    const int nprims = (int)s->nprims;
    const int T = 256;
    DevArray<RefitCtl> d_ctl;
    DevArray<float4> lmin, lmax;
    StreamDrain drain{ st };                                 // the scratch goes back to the cache idle, whichever return is taken
    if (int rc = d_ctl.alloc(1, st)) return rc;
    if (int rc = lmin.alloc((size_t)nprims, st)) return rc;
    if (int rc = lmax.alloc((size_t)nprims, st)) return rc;
    const unsigned grid_lines = (unsigned)((nobj + T - 1) / T);
    k_refit_init<<<1, 32, 0, st>>>(d_ctl.get());
    k_refit_check<<<grid_lines, T, 0, st>>>(d_objs, nobj, s->refit_inv.get(), lmin.get(), lmax.get(), d_ctl.get());
    if (nprims > 0) {
        k_refit_pack<<<grid_lines, T, 0, st>>>(d_objs, nobj, s->refit_inv.get(), d_ctl.get(), s->prims.get(), s->recs.get());
        int blocks = 1;
        if (int rc = coop_grid(s->device, (const void*)k_refit_wide, (int)((s->nwnodes + kBuildThreads - 1) / kBuildThreads), 2, &blocks)) return rc;
        int levels = s->wide_levels;
        void* args[] = { s->wide_level_start.arg(), &levels, lmin.arg(), lmax.arg(), d_ctl.arg(), s->wnodes.arg() };
        DRB_CUDA(cudaLaunchCooperativeKernel((const void*)k_refit_wide, dim3(blocks), dim3(kBuildThreads), args, 0, st));
    }
    DRB_CUDA(cudaGetLastError());
    RefitCtl ctl;
    DRB_CUDA(cudaMemcpyAsync(&ctl, d_ctl.get(), sizeof ctl, cudaMemcpyDeviceToHost, st));
    DRB_CUDA(cudaStreamSynchronize(st));                     // the one synchronisation of the refit
    if (ctl.bad != ~0ull) {
        const long long line = (long long)(ctl.bad >> 2);
        if ((ctl.bad & 3ull) == kRefitKindChanged)
            drb_set_error("drb_scene_refit: object line %lld changed whether it is rendered, or its kind (sphere / triangle)", line);
        else
            drb_set_error("drb_scene_refit: object line %lld has a non-finite vertex, centre or radius", line);
        return DRB_ERR_ARG;
    }
    if (nprims > 0)
        for (int a = 0; a < 3; ++a) { s->info.bounds_min[a] = ordered_to_float(ctl.bounds[a]); s->info.bounds_max[a] = ordered_to_float(ctl.bounds[3 + a]); }
    return DRB_OK;
}

// The line -> slot map, made by the first refit on the scene's own stream: the stream it is freed on when the scene is.
int ensure_refit_inverse(drb_scene* s)
{
    if (s->refit_inv.get()) return DRB_OK;
    const int nprims = (int)s->nprims, T = 256;
    if (int rc = s->refit_inv.alloc((size_t)s->nobjects, s->stream)) return rc;
    DRB_CUDA(cudaMemsetAsync(s->refit_inv.get(), 0xFF, (size_t)s->nobjects * sizeof(uint32_t), s->stream));
    if (nprims > 0) k_refit_inverse<<<(nprims + T - 1) / T, T, 0, s->stream>>>(s->orig_id.get(), s->prims.get(), nprims, s->refit_inv.get());
    return DRB_OK;
}

int refit_args(const drb_scene* s, const void* objects, int64_t nobjects)
{
    if (!s || nobjects < 0 || (nobjects > 0 && !objects)) { drb_set_error("drb_scene_refit: bad argument"); return DRB_ERR_ARG; }
    if (nobjects != s->nobjects) {
        drb_set_error("drb_scene_refit: %lld object lines given, the scene has %lld", (long long)nobjects, (long long)s->nobjects);
        return DRB_ERR_ARG;
    }
    return DRB_OK;
}

} // namespace

void drb_host_scene_unpin(drb_host_scene* hs)
{
    if (hs && hs->pinned) { cudaHostUnregister((void*)hs->objects.data()); cudaGetLastError(); hs->pinned = false; }
}

extern "C" {

int drb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void drb_scene_free(drb_scene* s)
{
    if (!s) return;
    cudaSetDevice(s->device);
    cudaDeviceSynchronize();                                 // renders and queries may have run on caller streams
    cudaStream_t st = s->stream;
    delete s;                                                // every array goes back to the cache, some freed on the stream ...
    if (st) cudaStreamDestroy(st);                           // ... which therefore goes last
}

int drb_scene_create(const drb_host_scene* hs, int device, drb_scene** out) { return drb_scene_create_from_device(hs, device, 0u, nullptr, nullptr, out); }

int drb_scene_create_ex(const drb_host_scene* hs, int device, uint32_t build_flags, drb_scene** out)
{
    return drb_scene_create_from_device(hs, device, build_flags, nullptr, nullptr, out);
}

int drb_scene_create_from_device(const drb_host_scene* hs, int device, uint32_t build_flags, const void* objects_dev, void* stream, drb_scene** out)
{
    if (!hs || !out) { drb_set_error("drb_scene_create: null argument"); return DRB_ERR_ARG; }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        drb_set_error("no CUDA device available (dogeray_b200 has no CPU path)");
        return DRB_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) { drb_set_error("device %d out of range (0..%d)", device, ndev - 1); return DRB_ERR_ARG; }
    DRB_CUDA(cudaSetDevice(device));
    StageClock clk;
    auto s = new drb_scene();
    s->device = device;
    s->build_flags = build_flags;
    s->settings = hs->settings;
    cudaError_t ce = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    if (ce != cudaSuccess) { drb_set_error("cudaStreamCreate: %s", cudaGetErrorString(ce)); delete s; return DRB_ERR_CUDA; }
    if (int prc = retain_pool(device)) { cudaStreamDestroy(s->stream); delete s; return prc; }
    int rc = DRB_OK;
    if (objects_dev) {
        // the build runs on the scene's stream: order it after whatever produced the array
        cudaEvent_t ready = nullptr;
        if (cudaEventCreateWithFlags(&ready, cudaEventDisableTiming) != cudaSuccess || cudaEventRecord(ready, (cudaStream_t)stream) != cudaSuccess ||
            cudaStreamWaitEvent(s->stream, ready, 0) != cudaSuccess) {
            drb_set_error("cannot order the build after the caller's stream: %s", cudaGetErrorString(cudaGetLastError()));
            rc = DRB_ERR_CUDA;
        }
        if (ready) cudaEventDestroy(ready);
    } else if (!hs->objects.empty() && !hs->pinned) {
        // page-lock the object lines once per host scene so the upload runs at PCIe speed (and again for free next frame)
        if (cudaHostRegister((void*)hs->objects.data(), hs->objects.size() * sizeof(drb_object), cudaHostRegisterPortable) == cudaSuccess) hs->pinned = true;
        else cudaGetLastError();
    }
    clk.mark("stream+pool+pin");
    if (rc == DRB_OK) rc = upload_textures(s, hs);
    clk.mark("textures");
    if (rc == DRB_OK) rc = build_tree(s, hs, (const drb_object*)objects_dev);
    clk.mark("build_tree");
    clk.print("drb_scene_create");
    if (rc != DRB_OK) { std::string keep = drb_last_error(); drb_scene_free(s); drb_set_error("%s", keep.c_str()); return rc; }
    if (s->settings.backtex >= s->ntextures) s->settings.backtex = -1;
    *out = s;
    return DRB_OK;
}

int drb_scene_create_multi(const drb_host_scene* hs, const int* devices, int ndevices, uint32_t build_flags, drb_scene** out)
{
    if (!hs || !devices || ndevices < 1 || !out) { drb_set_error("drb_scene_create_multi: bad argument"); return DRB_ERR_ARG; }
    for (int k = 0; k < ndevices; ++k) out[k] = nullptr;
    if (ndevices == 1) return drb_scene_create_ex(hs, devices[0], build_flags, &out[0]);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); drb_set_error("no CUDA device available (dogeray_b200 has no CPU path)"); return DRB_ERR_CUDA; }
    for (int k = 0; k < ndevices; ++k)
        if (devices[k] < 0 || devices[k] >= ndev) { drb_set_error("device %d out of range (0..%d)", devices[k], ndev - 1); return DRB_ERR_ARG; }
    drb_host_scene_summarise(hs);                                   // before the threads: the cached counts are not thread-safe
    const size_t nobj = hs->objects.size();
    if (nobj && !hs->pinned) {
        if (cudaHostRegister((void*)hs->objects.data(), nobj * sizeof(drb_object), cudaHostRegisterPortable) == cudaSuccess) hs->pinned = true;
        else cudaGetLastError();
    }
    const bool debug = getenv("DOGERAY_B200_DEBUG") != nullptr;
    auto trace = [&](const char* fmt, int a, int b) { if (debug) { fprintf(stderr, "[dogeray_b200] create_multi: "); fprintf(stderr, fmt, a, b); fputc('\n', stderr); fflush(stderr); } };
    // share k = object lines [k * chunk, (k + 1) * chunk): uploaded by device k, pulled by all the others
    const size_t chunk = (nobj + (size_t)ndevices - 1) / (size_t)ndevices;
    struct Side { DevArray<drb_object> buf; cudaStream_t st = nullptr; cudaEvent_t uploaded = nullptr, pulled = nullptr; int rc = DRB_OK; std::string err; };
    std::vector<Side> side((size_t)ndevices);
    auto share = [&](int k, size_t* lo, size_t* hi) { *lo = std::min(nobj, (size_t)k * chunk); *hi = std::min(nobj, *lo + chunk); };
    // phase 1 (sequential, cheap): buffers, streams, events, and each device's own share on its way
    for (int k = 0; k < ndevices; ++k) {
        Side& sd = side[(size_t)k];
        auto bad = [&](const char* what) { sd.rc = DRB_ERR_CUDA; sd.err = std::string(what) + ": " + cudaGetErrorString(cudaGetLastError()); };
        if (cudaSetDevice(devices[k]) != cudaSuccess) { bad("cudaSetDevice"); break; }
        if (retain_pool(devices[k]) != DRB_OK) { sd.rc = DRB_ERR_CUDA; sd.err = drb_last_error(); break; }
        if (cudaStreamCreateWithFlags(&sd.st, cudaStreamNonBlocking) != cudaSuccess) { bad("cudaStreamCreate"); break; }
        if (cudaEventCreateWithFlags(&sd.uploaded, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&sd.pulled, cudaEventDisableTiming) != cudaSuccess) { bad("cudaEventCreate"); break; }
        if (sd.buf.alloc(nobj, sd.st) != DRB_OK) { bad("device memory for the object lines"); break; }
        size_t lo, hi; share(k, &lo, &hi);
        if (hi > lo && cudaMemcpyAsync(sd.buf.get() + lo, hs->objects.data() + lo, (hi - lo) * sizeof(drb_object), cudaMemcpyHostToDevice, sd.st) != cudaSuccess) { bad("upload"); break; }
        if (cudaEventRecord(sd.uploaded, sd.st) != cudaSuccess) { bad("cudaEventRecord"); break; }
        trace("share %d uploading on device %d", k, devices[k]);
    }
    bool ok = true;
    for (const Side& sd : side) ok = ok && sd.rc == DRB_OK;
    // phase 2: every device pulls the other shares from the device that uploaded them (NVLink where there is peer access,
    // staged by the driver otherwise), then builds; one host thread per device
    if (ok) {
        for (int k = 0; k < ndevices; ++k)
            for (int j = 0; j < ndevices; ++j) drb_peer_access(devices[j], devices[k]);
        auto work = [&](int k) {
            Side& sd = side[(size_t)k];
            auto bad = [&](const char* what) { sd.rc = DRB_ERR_CUDA; sd.err = std::string(what) + ": " + cudaGetErrorString(cudaGetLastError()); };
            if (cudaSetDevice(devices[k]) != cudaSuccess) return bad("cudaSetDevice");
            for (int d = 1; d < ndevices; ++d) {
                const int j = (k + d) % ndevices;                   // staggered, so the pulls do not all hit the same source at once
                size_t lo, hi; share(j, &lo, &hi);
                if (hi <= lo) continue;
                if (cudaStreamWaitEvent(sd.st, side[(size_t)j].uploaded, 0) != cudaSuccess) return bad("cudaStreamWaitEvent");
                const cudaError_t ce = devices[j] == devices[k]
                    ? cudaMemcpyAsync(sd.buf.get() + lo, side[(size_t)j].buf.get() + lo, (hi - lo) * sizeof(drb_object), cudaMemcpyDeviceToDevice, sd.st)
                    : cudaMemcpyPeerAsync(sd.buf.get() + lo, devices[k], side[(size_t)j].buf.get() + lo, devices[j], (hi - lo) * sizeof(drb_object), sd.st);
                if (ce != cudaSuccess) return bad("peer copy");
                trace("pulled share %d into %d", j, k);
            }
            if (cudaEventRecord(sd.pulled, sd.st) != cudaSuccess) return bad("cudaEventRecord");
            trace("building scene %d on device %d", k, devices[k]);
            sd.rc = drb_scene_create_from_device(hs, devices[k], build_flags, sd.buf.get(), sd.st, &out[k]);
            if (sd.rc != DRB_OK) sd.err = drb_last_error();
            trace("scene %d: rc %d", k, sd.rc);
        };
        std::vector<std::thread> pool;
        for (int k = 1; k < ndevices; ++k) pool.emplace_back(work, k);
        work(0);
        for (auto& th : pool) th.join();
    }
    trace("threads joined (%d devices, ok %d)", ndevices, ok ? 1 : 0);
    // a share may be freed only after every device has pulled it
    for (int k = 0; k < ndevices; ++k)
        if (side[(size_t)k].st && cudaSetDevice(devices[k]) == cudaSuccess) cudaStreamSynchronize(side[(size_t)k].st);
    for (int k = 0; k < ndevices; ++k) {
        Side& sd = side[(size_t)k];
        if (cudaSetDevice(devices[k]) != cudaSuccess) { cudaGetLastError(); continue; }
        sd.buf.reset();                                             // before its stream goes
        if (sd.uploaded) cudaEventDestroy(sd.uploaded);
        if (sd.pulled) cudaEventDestroy(sd.pulled);
        if (sd.st) cudaStreamDestroy(sd.st);
    }
    cudaGetLastError();
    for (int k = 0; k < ndevices; ++k)
        if (side[(size_t)k].rc != DRB_OK) {
            const int rc = side[(size_t)k].rc;
            const std::string msg = side[(size_t)k].err;
            for (int j = 0; j < ndevices; ++j) { if (out[j]) drb_scene_free(out[j]); out[j] = nullptr; }
            drb_set_error("drb_scene_create_multi: device %d: %s", devices[k], msg.c_str());
            return rc;
        }
    return DRB_OK;
}

int drb_scene_load(const char* rts_path, const char* tex_dir, int device, drb_scene** out)
{
    if (!out) { drb_set_error("drb_scene_load: null argument"); return DRB_ERR_ARG; }
    drb_host_scene* hs = nullptr;
    int rc = drb_host_scene_load(rts_path, tex_dir, &hs);
    if (rc != DRB_OK) return rc;
    rc = drb_scene_create(hs, device, out);
    drb_host_scene_free(hs);
    return rc;
}

int drb_scene_settings(const drb_scene* s, drb_settings* out)
{
    if (!s || !out) { drb_set_error("drb_scene_settings: null argument"); return DRB_ERR_ARG; }
    *out = s->settings;
    return DRB_OK;
}
int64_t drb_scene_num_prims(const drb_scene* s) { return s ? s->nprims : 0; }
int64_t drb_scene_num_objects(const drb_scene* s) { return s ? s->nobjects : 0; }
int drb_scene_build_info(const drb_scene* s, drb_build_info* out)
{
    if (!s || !out) { drb_set_error("drb_scene_build_info: null argument"); return DRB_ERR_ARG; }
    *out = s->info;
    return DRB_OK;
}

int drb_scene_refit_device(drb_scene* s, const void* objects_dev, int64_t nobjects, void* stream)
{
    if (int rc = refit_args(s, objects_dev, nobjects)) return rc;
    if (nobjects == 0) return DRB_OK;
    DRB_CUDA(cudaSetDevice(s->device));
    if (int rc = ensure_refit_inverse(s)) return rc;
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (st != s->stream) {
        // the refit runs on the caller's stream, after what is already enqueued on the scene's own
        cudaEvent_t done = nullptr;
        DRB_CUDA(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
        const cudaError_t e1 = cudaEventRecord(done, s->stream);
        const cudaError_t e2 = e1 == cudaSuccess ? cudaStreamWaitEvent(st, done, 0) : e1;
        cudaEventDestroy(done);
        DRB_CUDA(e2);
    }
    return refit_tree(s, (const drb_object*)objects_dev, st);
}

int drb_scene_refit(drb_scene* s, const drb_object* objects_host, int64_t nobjects)
{
    if (int rc = refit_args(s, objects_host, nobjects)) return rc;
    if (nobjects == 0) return DRB_OK;
    DRB_CUDA(cudaSetDevice(s->device));
    if (int rc = ensure_refit_inverse(s)) return rc;
    DevArray<drb_object> d;                                  // idle once refit_tree returns: it drains the same stream
    if (int rc = d.alloc((size_t)nobjects, s->stream)) return rc;
    DRB_CUDA(cudaMemcpyAsync(d.get(), objects_host, (size_t)nobjects * sizeof(drb_object), cudaMemcpyHostToDevice, s->stream));
    return refit_tree(s, d.get(), s->stream);
}

int drb_scene_lbvh(const drb_scene* s, uint64_t* keys, int32_t* order, int32_t* parent, int32_t* left, int32_t* right,
                   float* node_min, float* node_max)
{
    if (!s) { drb_set_error("drb_scene_lbvh: null scene"); return DRB_ERR_ARG; }
    if (!(s->build_flags & DRB_BUILD_KEEP_DEBUG)) { drb_set_error("drb_scene_lbvh: the scene was not created with DRB_BUILD_KEEP_DEBUG"); return DRB_ERR_UNSUPPORTED; }
    DRB_CUDA(cudaSetDevice(s->device));
    const size_t n = (size_t)s->nprims, ni = n > 1 ? n - 1 : 0;
    if (keys && n) DRB_CUDA(cudaMemcpy(keys, s->dbg.keys.get(), n * 8, cudaMemcpyDeviceToHost));
    if (order && n) DRB_CUDA(cudaMemcpy(order, s->dbg.order.get(), n * 4, cudaMemcpyDeviceToHost));
    if (parent && ni) DRB_CUDA(cudaMemcpy(parent, s->dbg.parent.get(), ni * 4, cudaMemcpyDeviceToHost));
    if (left && ni) DRB_CUDA(cudaMemcpy(left, s->dbg.left.get(), ni * 4, cudaMemcpyDeviceToHost));
    if (right && ni) DRB_CUDA(cudaMemcpy(right, s->dbg.right.get(), ni * 4, cudaMemcpyDeviceToHost));
    if ((node_min || node_max) && ni) {
        std::vector<float4> tmp(ni);
        if (node_min) {
            DRB_CUDA(cudaMemcpy(tmp.data(), s->dbg.node_min.get(), ni * 16, cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < ni; ++i) { node_min[3*i] = tmp[i].x; node_min[3*i+1] = tmp[i].y; node_min[3*i+2] = tmp[i].z; }
        }
        if (node_max) {
            DRB_CUDA(cudaMemcpy(tmp.data(), s->dbg.node_max.get(), ni * 16, cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < ni; ++i) { node_max[3*i] = tmp[i].x; node_max[3*i+1] = tmp[i].y; node_max[3*i+2] = tmp[i].z; }
        }
    }
    return DRB_OK;
}

int drb_scene_wide(const drb_scene* s, int32_t* child, uint32_t* boxes)
{
    if (!s) { drb_set_error("drb_scene_wide: null scene"); return DRB_ERR_ARG; }
    DRB_CUDA(cudaSetDevice(s->device));
    const size_t n = (size_t)s->nwnodes;
    if (!n) return DRB_OK;
    std::vector<WideNode> tmp(n);
    DRB_CUDA(cudaMemcpy(tmp.data(), s->wnodes.get(), n * sizeof(WideNode), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n; ++i)
        for (int k = 0; k < 4; ++k) {
            if (child) child[4 * i + k] = tmp[i].child[k];
            if (boxes) { boxes[12 * i + 3 * k] = tmp[i].bx[k]; boxes[12 * i + 3 * k + 1] = tmp[i].by[k]; boxes[12 * i + 3 * k + 2] = tmp[i].bz[k]; }
        }
    return DRB_OK;
}

int drb_scene_tree(const drb_scene* s, int32_t* left, int32_t* right, float* node_min, float* node_max)
{
    if (!s) { drb_set_error("drb_scene_tree: null scene"); return DRB_ERR_ARG; }
    if (!(s->build_flags & DRB_BUILD_KEEP_DEBUG)) { drb_set_error("drb_scene_tree: the scene was not created with DRB_BUILD_KEEP_DEBUG"); return DRB_ERR_UNSUPPORTED; }
    DRB_CUDA(cudaSetDevice(s->device));
    const size_t n = (size_t)s->nprims, ni = n > 1 ? n - 1 : 0;
    if (left && ni) DRB_CUDA(cudaMemcpy(left, s->tree.left.get(), ni * 4, cudaMemcpyDeviceToHost));
    if (right && ni) DRB_CUDA(cudaMemcpy(right, s->tree.right.get(), ni * 4, cudaMemcpyDeviceToHost));
    if ((node_min || node_max) && ni) {
        std::vector<float4> tmp(ni);
        if (node_min) {
            DRB_CUDA(cudaMemcpy(tmp.data(), s->tree.node_min.get(), ni * 16, cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < ni; ++i) { node_min[3*i] = tmp[i].x; node_min[3*i+1] = tmp[i].y; node_min[3*i+2] = tmp[i].z; }
        }
        if (node_max) {
            DRB_CUDA(cudaMemcpy(tmp.data(), s->tree.node_max.get(), ni * 16, cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < ni; ++i) { node_max[3*i] = tmp[i].x; node_max[3*i+1] = tmp[i].y; node_max[3*i+2] = tmp[i].z; }
        }
    }
    return DRB_OK;
}

} // extern "C"
