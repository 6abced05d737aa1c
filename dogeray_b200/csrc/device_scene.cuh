// Device-resident scene layout (HBM).  Everything the reference keeps as two AoS arrays --
// `singleobject` (164 B, raygpu/kernel.cu:48-74) and `bvh` (56 B, kernel.cu:79-96) -- re-laid for
// 128-bit loads.  See DESIGN.md "Data layout in HBM".
#pragma once
#include "drb_internal.h"
#include <cuda_runtime.h>
#include <cstdint>
#include <memory>
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

#define DRB_CUDA(call)                                                                                     \
    do {                                                                                                   \
        cudaError_t e__ = (call);                                                                          \
        if (e__ != cudaSuccess) {                                                                          \
            drb_set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e__));   \
            return DRB_ERR_CUDA;                                                                           \
        }                                                                                                  \
    } while (0)

// Device memory for scenes and render buffers.  Blocks come from the device's stream-ordered pool (release
// threshold raised so nothing goes back to the driver) through an exact-size cache: a scene that is created,
// rendered and freed every frame -- the reference's CudaStarter pattern, kernel.cu:2604-2665 -- finds every block
// it needs in the cache and performs no allocator call at all.  Blocks must be idle (their stream synchronised)
// when they are handed back.  Called only by DevArray and the cache itself.
cudaError_t drb_dev_alloc(void** p, size_t bytes, cudaStream_t st);
void drb_dev_free(void* p, cudaStream_t st);

// The owner of one block of `count` T from the block cache, on the device that was current at alloc().  The block goes
// back to that device's cache when the owner is reset or destroyed, freed on the stream it was allocated on, so that
// stream must outlive the owner.  The owner does not synchronise: whoever holds it synchronises the stream (or the
// device) first, so that the block is idle.
template <typename T> class DevArray {
public:
    DevArray() = default;
    DevArray(DevArray&& o) noexcept : p_(o.p_), dev_(o.dev_), st_(o.st_) { o.p_ = nullptr; }
    DevArray& operator=(DevArray&& o) noexcept
    {
        if (this != &o) { reset(); p_ = o.p_; dev_ = o.dev_; st_ = o.st_; o.p_ = nullptr; }
        return *this;
    }
    ~DevArray() { reset(); }

    // releases the block held so far first; a count of 0 still yields a valid one-element block
    int alloc(size_t count, cudaStream_t st)
    {
        reset();
        void* p = nullptr;
        DRB_CUDA(drb_dev_alloc(&p, (count ? count : 1) * sizeof(T), st));
        cudaGetDevice(&dev_);
        p_ = static_cast<T*>(p);
        st_ = st;
        return DRB_OK;
    }
    void reset()
    {
        if (!p_) return;
        int cur = -1;
        cudaGetDevice(&cur);
        if (cur != dev_) cudaSetDevice(dev_);
        drb_dev_free(p_, st_);
        if (cur != dev_ && cur >= 0) cudaSetDevice(cur);
        p_ = nullptr;
    }
    T* get() const { return p_; }
    void* arg() { return &p_; }         // an entry of a kernel-argument array (cudaLaunchCooperativeKernel)

private:
    T* p_ = nullptr;
    int dev_ = -1;
    cudaStream_t st_ = nullptr;
};

// Synchronises a stream when it goes out of scope.  A call declares it after its scratch owners, so that it runs before
// they hand their blocks back: an error can return while work is still queued on them.
struct StreamDrain {
    cudaStream_t st;
    ~StreamDrain() { cudaStreamSynchronize(st); }
};

struct LbvhDebug {              // integer outputs of the build, kept for drb_scene_lbvh (DRB_BUILD_KEEP_DEBUG only)
    DevArray<uint64_t> keys;    // n, sorted
    DevArray<int32_t> order;    // n
    DevArray<int32_t> parent;   // n-1
    DevArray<int32_t> left;     // n-1
    DevArray<int32_t> right;    // n-1
    DevArray<float4> node_min;  // n-1
    DevArray<float4> node_max;  // n-1
};

struct FinalTree {              // the hierarchy the nodes were emitted from (root = node 0), for drb_scene_tree (DRB_BUILD_KEEP_DEBUG only)
    DevArray<int32_t> left;     // n-1
    DevArray<int32_t> right;    // n-1
    DevArray<float4> node_min;  // n-1
    DevArray<float4> node_max;  // n-1
};

// the render's work buffers and the ray queries' scratch, defined in render.cu
struct RenderBuffers;
struct QueryBuffers;
struct BuffersDelete {
    void operator()(RenderBuffers* p) const;
    void operator()(QueryBuffers* p) const;
};

// Every device array of a scene is owned by a member: deleting the scene (after a synchronisation, drb_scene_free)
// returns them all.  `stream` is not owned here: the blocks are freed on it, so drb_scene_free destroys it last.
struct drb_scene {
    int device = 0;
    uint32_t build_flags = 0;
    FinalTree tree;
    drb_settings settings;
    int64_t nobjects = 0;       // object lines
    int64_t nprims = 0;         // renderable primitives (in the tree)
    int64_t nnodes = 0;
    DevArray<WideNode> wnodes;  // the traversal structure
    int64_t nwnodes = 0;
    int wide_levels = 0;        // height of the wide tree (levels of the breadth-first collapse)
    DevArray<int> wide_level_start;  // first node of every level, wide_levels + 1 entries (the refit's bottom-up order)
    DevArray<uint32_t> refit_inv;    // object line -> slot << 1 | sphere, or ~0u; made by the first refit
    int stack_levels = 3;       // traversal stack entries a lane can need (exact bound from the collapse + sentinel + 1)
    DevArray<Prim> prims;
    DevArray<ShadeRec> recs;
    DevArray<int32_t> orig_id;  // prim slot -> object line index
    DevArray<DevTexture> textures;
    int ntextures = 0;
    std::vector<DevArray<uint8_t>> texture_storage;
    LbvhDebug dbg;
    drb_build_info info;
    cudaStream_t stream = nullptr;
    // render work buffers, grown on demand (render.cu)
    std::unique_ptr<RenderBuffers, BuffersDelete> rb;
    // ray-query scratch, separate from the render's queues (render.cu)
    std::unique_ptr<QueryBuffers, BuffersDelete> qb;
};

// Facts of a device, asked of the driver once per process and device (and kernel): each of these queries takes a
// device-wide lock, and asked once per scene handle they stalled frames by tens of milliseconds whenever a monitoring
// process polled the GPU (DESIGN.md section 8).  One cache under one mutex answers them all, for every host thread.
// SMs of `device`, and resident blocks per SM of `kernel` at `threads` per block and `smem` bytes of dynamic shared memory
// there (`device` current), whose limit is raised first when it lies below `smem`
int drb_occupancy(const void* kernel, int threads, size_t smem, int device, int* sms, int* per_sm);
// total memory of `device`, which must be current; 0 when it cannot be asked
size_t drb_device_total_mem(int device);
// Lets kernels and copies running on device `accessor` address pool memory of device `owner` (NVLink peers); granted once
// per pair and process.  False when the devices cannot reach each other.
bool drb_peer_access(int owner, int accessor);
