// Device-resident scene layout (HBM).  Everything the reference keeps as two AoS arrays --
// `singleobject` (164 B, raygpu/kernel.cu:48-74) and `bvh` (56 B, kernel.cu:79-96) -- re-laid for
// 128-bit loads.  See DESIGN.md "Data layout in HBM".
#pragma once
#include "dogeray_b200.h"
#include <cuda_runtime.h>
#include <cstdint>
#include <string>
#include <vector>

// 64 B four-wide node, two 256-bit loads: the binary hierarchy collapsed two levels at a time (k_wide_* in
// scene.cu).  Child boxes are quantised to 16 bits per plane on a scene-wide grid (drb_quant_grid), rounded outwards
// plus one quantum of margin, so a quantised box always contains the float box it came from.  Traversal never
// converts the integers: PRMT drops a 16-bit half under the exponent byte 0x4B (the float 2^23 + q) and one FMA with
// per-ray constants turns it into the plane's ray parameter.
//   bx[c], by[c], bz[c] = min_q | max_q << 16 of child c on each axis; an empty slot has min 65535 > max 0
//   child[c] >= 0: wide node index, < 0: leaf, ~child = primitive slot, kWideEmpty: no child
struct __align__(32) WideNode {
    uint32_t bx[4], by[4];
    uint32_t bz[4];
    int32_t child[4];
};
static_assert(sizeof(WideNode) == 64, "WideNode must be 64 bytes");
#define DRB_WIDE_EMPTY ((int32_t)0x80000000)

// The quantisation grid of one axis: 65528 quanta span the scene bounds, 4 spare quanta on each side so the
// outward margin never clamps.  Same single float operations on host and device.
#ifdef __CUDACC__
__host__ __device__
#endif
inline void drb_quant_grid(float lo, float hi, float* qlo, float* qscale)
{
    float ext = hi - lo;
    if (!(ext > 0.0f)) ext = 1.0f;
    const float sc = ext / 65527.0f;
    *qscale = sc;
    *qlo = lo - 4.0f * sc;
}

#ifdef __CUDACC__
// one 256-bit read-only global load (PTX ISA 8.8, sm_100+): half the L1 data-pipe wavefronts of two LDG.128
struct __align__(32) f8 { float4 lo, hi; };
__device__ __forceinline__ f8 ldg256(const void* p)
{
    f8 r;
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(r.lo.x), "=f"(r.lo.y), "=f"(r.lo.z), "=f"(r.lo.w), "=f"(r.hi.x), "=f"(r.hi.y), "=f"(r.hi.z), "=f"(r.hi.w)
                 : "l"(p));
    return r;
}
#endif

// 64 B primitive, in tree (Morton) order, fetched with two 256-bit loads (LDG.E.256 on sm_100).
//   triangle: a = (v0, kind 0), b = (v1 - v0, 0), c = (v2 - v0, 0), d = spare   (edges precomputed in float,
//             exactly the subtraction hit_tri does first, kernel.cu:287-288)
//   sphere:   a = (centre, kind 1), b = (radius, 0, 0, 0)
struct __align__(32) Prim {
    float4 a, b, c, d;
};
static_assert(sizeof(Prim) == 64, "Prim must be 64 bytes");
#define DRB_KIND_TRI 0
#define DRB_KIND_SPHERE 1

// 128 B shading record per primitive, same order as Prim; the first 48 B serve the common case.
//   r0 = (face normal xyz, flags)                      flags: DRB_SF_*
//   r1 = (col rgb, rough = addional.y)
//   r2 = (addional.x, mat, texnum, rtexnum)            (ints stored as bits)
//   r3 = (n1 xyz, t1.x)  r4 = (n2 xyz, t2.x)  r5 = (n3 xyz, t3.x)  r6 = (t1.y, t2.y, t3.y, 0)
//   r7 = spare
struct __align__(16) ShadeRec {
    float4 r[8];
};
static_assert(sizeof(ShadeRec) == 128, "ShadeRec must be 128 bytes");
#define DRB_SF_SPHERE 1u        // getnormal's type 0 branch, kernel.cu:707-710
#define DRB_SF_FACE_NORMAL 2u   // norm.z != -20, kernel.cu:750
#define DRB_SF_SMOOTH 4u        // face normal present && n1.z != -20 && smooth, kernel.cu:756
#define DRB_SF_CHECKER 8u       // `tex` flag, kernel.cu:834
#define DRB_SF_NEEDS_UV 16u     // barycentrics are needed (smooth, textured, checker)

struct DevTexture {
    const uchar4* texels;   // row-major, top-down
    int32_t w, h;
};

struct LbvhDebug {              // integer outputs of the build, kept for drb_scene_lbvh (DRB_BUILD_KEEP_DEBUG only)
    uint64_t* keys = nullptr;   // n, sorted
    int32_t* order = nullptr;   // n
    int32_t* parent = nullptr;  // n-1
    int32_t* left = nullptr;    // n-1
    int32_t* right = nullptr;   // n-1
    float4* node_min = nullptr; // n-1
    float4* node_max = nullptr; // n-1
};

struct FinalTree {              // the hierarchy the nodes were emitted from (root = node 0), for drb_scene_tree (DRB_BUILD_KEEP_DEBUG only)
    int32_t* left = nullptr;    // n-1
    int32_t* right = nullptr;   // n-1
    float4* node_min = nullptr; // n-1
    float4* node_max = nullptr; // n-1
};

struct drb_scene {
    int device = 0;
    uint32_t build_flags = 0;
    FinalTree tree;
    drb_settings settings;
    int64_t nobjects = 0;       // object lines
    int64_t nprims = 0;         // renderable primitives (in the tree)
    int64_t nnodes = 0;
    WideNode* wnodes = nullptr; // the traversal structure
    int64_t nwnodes = 0;
    int wide_levels = 0;        // height of the wide tree (levels of the breadth-first collapse)
    int* wide_level_start = nullptr; // first node of every level, wide_levels + 1 entries (the refit's bottom-up order)
    uint32_t* refit_inv = nullptr;   // object line -> slot << 1 | sphere, or ~0u; made by the first refit
    int stack_levels = 3;       // traversal stack entries a lane can need (exact bound from the collapse + sentinel + 1)
    Prim* prims = nullptr;
    ShadeRec* recs = nullptr;
    int32_t* orig_id = nullptr; // prim slot -> object line index
    DevTexture* textures = nullptr;
    int ntextures = 0;
    std::vector<void*> texture_storage;
    LbvhDebug dbg;
    drb_build_info info;
    cudaStream_t stream = nullptr;
    // render work buffers, grown on demand (render.cu)
    struct RenderBuffers* rb = nullptr;
    // ray-query scratch, separate from the render's queues (render.cu)
    struct QueryBuffers* qb = nullptr;
};

#define DRB_CUDA(call)                                                                                     \
    do {                                                                                                   \
        cudaError_t e__ = (call);                                                                          \
        if (e__ != cudaSuccess) {                                                                          \
            drb_set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e__));   \
            return DRB_ERR_CUDA;                                                                           \
        }                                                                                                  \
    } while (0)

void drb_render_buffers_free(drb_scene* s);
void drb_query_buffers_free(drb_scene* s);
// Lets kernels and copies running on device `accessor` address pool memory of device `owner` (NVLink peers); granted once
// per pair and process.  False when the devices cannot reach each other.
bool drb_peer_access(int owner, int accessor);

// Device memory for scenes and render buffers.  Blocks come from the device's stream-ordered pool (release
// threshold raised so nothing goes back to the driver) through an exact-size cache: a scene that is created,
// rendered and freed every frame -- the reference's CudaStarter pattern, kernel.cu:2604-2665 -- finds every block
// it needs in the cache and performs no allocator call at all.  Blocks must be idle (their stream synchronised)
// when they are handed back.
cudaError_t drb_dev_alloc(void** p, size_t bytes, cudaStream_t st);
void drb_dev_free(void* p, cudaStream_t st);
