// sm_100a kernels of the hot path: batch queries, the unit predicates, and the wavefront renderer.
// Strict build: -fmad=false, IEEE div/sqrt. No tensor cores (the path is not a dense contraction), no OptiX.
#include "cgrt_kernels.h"
#include "cgrt_device.cuh"

#include <float.h>
#include <stdlib.h>
#include <string>

namespace cgrt {

// =================================================================================================================
// Scene set-up: planes of all triangles (trianglePlane, src/ray_tracing.cpp:74-82) computed once, on the device.
// =================================================================================================================
__global__ void k_setup_planes(const float4* __restrict__ v0, const float4* __restrict__ v1, const float4* __restrict__ v2,
                               float4* __restrict__ pl, float4* __restrict__ tri4, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 a = v0[i], b = v1[i], c = v2[i];
    const float4 p = trianglePlaneDev(mk3(a), mk3(b), mk3(c));
    pl[i] = p;
    tri4[4 * (size_t)i + 0] = p;
    tri4[4 * (size_t)i + 1] = a;
    tri4[4 * (size_t)i + 2] = b;
    tri4[4 * (size_t)i + 3] = c;
}

// tri4f[k] = tri4[fastOrder[k]] with the position in tri4 in v2.w (fastOrder == nullptr: identity)
__global__ void k_permute_tri4(const float4* __restrict__ tri4, const int* __restrict__ fastOrder, float4* __restrict__ tri4f, int n)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int p = fastOrder ? fastOrder[k] : k;
    float4 c = tri4[4 * (size_t)p + 3];
    c.w = __int_as_float(p);
    tri4f[4 * (size_t)k + 0] = tri4[4 * (size_t)p + 0];
    tri4f[4 * (size_t)k + 1] = tri4[4 * (size_t)p + 1];
    tri4f[4 * (size_t)k + 2] = tri4[4 * (size_t)p + 2];
    tri4f[4 * (size_t)k + 3] = c;
}

// =================================================================================================================
// Batch closest hit: one thread per ray.  BoundingVolumeHierarchy::intersect, src/bounding_volume_hierarchy.cpp:850-881
// =================================================================================================================
RT_DEV void writeHit(const DevScene& S, const V3& o, const V3& d, float tIn, bool hit, const TraceResult& R, float4* out)
{
    float4 h0 = make_float4(hit ? R.t : tIn, i2f(-1), 0.0f, 0.0f);
    float4 h1 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (hit) {
        if (R.sphere >= 0) {
            const int srcTri = R.tri >= 0 ? f2i(__ldg(S.triV0 + R.tri).w) : -1;
            h0.y = i2f(-2 - R.sphere);
            h0.z = i2f(srcTri);
            h1.y = R.sphereN.x; h1.z = R.sphereN.y; h1.w = R.sphereN.z;
        } else {
            const int i = R.tri;
            const float4 v0 = __ldg(S.triV0 + i), v1 = __ldg(S.triV1 + i), v2 = __ldg(S.triV2 + i);
            const float4 n0 = __ldg(S.triN0 + i), n1 = __ldg(S.triN1 + i), n2 = __ldg(S.triN2 + i);
            const float4 pl = __ldg(S.triPl + i);
            float al, be, ga;
            V3 nn;
            hitEpilogue(mk3(v0), mk3(v1), mk3(v2), mk3(n0), mk3(n1), mk3(n2), mk3(pl), o, d, R.t, al, be, ga, nn);
            h0.y = v0.w; // global id bits
            h0.z = al; h0.w = be;
            h1.x = ga; h1.y = nn.x; h1.z = nn.y; h1.w = nn.z;
        }
    }
    out[0] = h0;
    out[1] = h1;
}

template <bool COUNT>
__global__ void __launch_bounds__(128) k_closest_batch(DevScene S, const float4* __restrict__ rays, size_t n,
                                                       float4* __restrict__ hits, uint32_t* __restrict__ counts)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float4 r0 = __ldg(rays + 2 * i), r1 = __ldg(rays + 2 * i + 1);
        const V3 o = mk3(r0), d = mk3(r1);
        TraceResult R;
        uint32_t nBox = 0, nTri = 0;
        const bool hit = COUNT ? traverseStrict<false, true>(S, o, d, r0.w, 0.0f, 0.0f, R, nBox, nTri)
                               : traverseSpec<false>(S, o, d, r0.w, 0.0f, 0.0f, R);
        writeHit(S, o, d, r0.w, hit, R, hits + 2 * i);
        if (COUNT) {
            counts[2 * i] = nBox;
            counts[2 * i + 1] = nTri;
        }
    }
}

__global__ void __launch_bounds__(128) k_any_batch(DevScene S, const float4* __restrict__ rays,
                                                   const float* __restrict__ maxDist, float eps, size_t n,
                                                   uint8_t* __restrict__ occluded)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float4 r0 = __ldg(rays + 2 * i), r1 = __ldg(rays + 2 * i + 1);
        TraceResult R;
        const bool sh = traverseSpec<true>(S, mk3(r0), mk3(r1), r0.w, eps, __ldg(maxDist + i), R);
        occluded[i] = sh ? 1 : 0;
    }
}

// intersectRayWithShape(const Mesh&, ...) over every mesh in scene order, src/ray_tracing.cpp:202-213
__global__ void __launch_bounds__(128) k_brute_batch(DevScene S, const float4* __restrict__ rays, size_t n,
                                                     float4* __restrict__ hits)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float4 r0 = __ldg(rays + 2 * i), r1 = __ldg(rays + 2 * i + 1);
        const V3 o = mk3(r0), d = mk3(r1);
        TraceResult R;
        R.sphere = -1;
        R.tri = -1;
        float t = r0.w;
        for (int g = 0; g < S.nTris; g++) {
            const int k = __ldg(S.origToLeaf + g);
            const float4 pl = __ldg(S.triPl + k);
            float tt;
            if (planeTest(mk3(pl), pl.w, o, d, t, tt)) {
                const float4 v0 = __ldg(S.triV0 + k), v1 = __ldg(S.triV1 + k), v2 = __ldg(S.triV2 + k);
                if (pointInTriangleDev(mk3(v0), mk3(v1), mk3(v2), mk3(pl), o + d * tt)) {
                    t = tt;
                    R.tri = k;
                }
            }
        }
        R.t = t;
        writeHit(S, o, d, r0.w, R.tri >= 0, R, hits + 2 * i);
    }
}

// =================================================================================================================
// Unit predicates (src/ray_tracing.h:10-20), one element per thread
// =================================================================================================================
__global__ void k_unit_aabb(const float* __restrict__ boxes, const float4* __restrict__ rays, size_t n,
                            uint8_t* __restrict__ hit, float* __restrict__ t)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* b = boxes + 6 * i;
    const float4 r0 = rays[2 * i], r1 = rays[2 * i + 1];
    float th;
    const bool h = slabTest(mk3(b[0], b[1], b[2]), mk3(b[3], b[4], b[5]), mk3(r0), mk3(r1), r0.w, th);
    hit[i] = h;
    t[i] = h ? th : r0.w;
}

__global__ void k_unit_triangle(const float* __restrict__ tris, const float4* __restrict__ rays, size_t n,
                                float4* __restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* q = tris + 18 * i;
    const V3 v0 = mk3(q[0], q[1], q[2]), v1 = mk3(q[3], q[4], q[5]), v2 = mk3(q[6], q[7], q[8]);
    const V3 n0 = mk3(q[9], q[10], q[11]), n1 = mk3(q[12], q[13], q[14]), n2 = mk3(q[15], q[16], q[17]);
    const float4 r0 = rays[2 * i], r1 = rays[2 * i + 1];
    const V3 o = mk3(r0), d = mk3(r1);
    const float4 pl = trianglePlaneDev(v0, v1, v2);
    float4 h0 = make_float4(r0.w, i2f(0), 0.0f, 0.0f), h1 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    float tt;
    if (planeTest(mk3(pl), pl.w, o, d, r0.w, tt) && pointInTriangleDev(v0, v1, v2, mk3(pl), o + d * tt)) {
        float al, be, ga;
        V3 nn;
        hitEpilogue(v0, v1, v2, n0, n1, n2, mk3(pl), o, d, tt, al, be, ga, nn);
        h0 = make_float4(tt, i2f(1), al, be);
        h1 = make_float4(ga, nn.x, nn.y, nn.z);
    }
    out[2 * i] = h0;
    out[2 * i + 1] = h1;
}

__global__ void k_unit_plane(const float4* __restrict__ planes, const float4* __restrict__ rays, size_t n,
                             uint8_t* __restrict__ hit, float* __restrict__ t)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 pl = planes[i], r0 = rays[2 * i], r1 = rays[2 * i + 1];
    float tt;
    const bool h = planeTest(mk3(pl), pl.w, mk3(r0), mk3(r1), r0.w, tt);
    hit[i] = h;
    t[i] = h ? tt : r0.w;
}

__global__ void k_unit_triangle_plane(const float* __restrict__ tris, size_t n, float4* __restrict__ planes)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* q = tris + 9 * i;
    planes[i] = trianglePlaneDev(mk3(q[0], q[1], q[2]), mk3(q[3], q[4], q[5]), mk3(q[6], q[7], q[8]));
}

__global__ void k_unit_point_in_triangle(const float* __restrict__ in, size_t n, uint8_t* __restrict__ inside)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* q = in + 15 * i;
    inside[i] = pointInTriangleDev(mk3(q[0], q[1], q[2]), mk3(q[3], q[4], q[5]), mk3(q[6], q[7], q[8]),
                                   mk3(q[9], q[10], q[11]), mk3(q[12], q[13], q[14]));
}

__global__ void k_unit_sphere(const float4* __restrict__ spheres, const float4* __restrict__ rays, size_t n,
                              float* __restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 s = spheres[i], r0 = rays[2 * i], r1 = rays[2 * i + 1];
    float ts;
    V3 nn = mk3(0.0f, 0.0f, 0.0f);
    const bool h = sphereTest(mk3(s), s.w, mk3(r0), mk3(r1), r0.w, ts, nn);
    float* o = out + 5 * i;
    o[0] = h ? ts : r0.w;
    o[1] = i2f(h ? 1 : 0);
    o[2] = nn.x; o[3] = nn.y; o[4] = nn.z;
}

// =================================================================================================================
// Wavefront renderer.  renderRayTracing + getFinalColor/trace/shade/shading/pointInShadow (src/main.cpp:61-310, 648-697)
// One of four kernel sets renders a frame (choosePipeline, cgrt_capi.cu); all four give the same pixels and ray counts:
//   counting wavefront  CGRT_RENDER_COUNT: level by level, counting the reference's box / triangle tests (launchCountingFrame)
//   path pipeline       scenes without a fast tree, and frames too large for the round pipeline (launchPathPipeline)
//   round pipeline      large shallow frames of scenes with a fast tree (launchRoundPipeline)
//   k_wave              every other frame of a scene with a fast tree (launchWavePipeline, cgrt_wave.cuh; DESIGN 4.4)
// =================================================================================================================
// Trackball::generateRay (framework/src/trackball.cpp:92-103) with the host-evaluated constants of FrameParams; the pixel ->
// NDC mapping is main.cpp:691-693 (pixel corners, left-to-right evaluation).
RT_DEV V3 quatRotate(const float4& q /* x,y,z,w */, const V3& v)
{
    const V3 qv = mk3(q.x, q.y, q.z);
    const V3 uv = cross3(qv, v);
    const V3 uuv = cross3(qv, uv);
    return v + ((uv * q.w) + uuv) * 2.0f;
}
// camera constants of one view (host-evaluated, cgrt_capi.cu cameraConstants)
struct ViewCamera {
    V3 o;                // Trackball::position()
    float halfW, halfH;
    float4 q;            // x, y, z, w
};
// view v of the frame: its CGRT_VIEW_F4 float4s follow the point and spherical lights in the parameter block
RT_DEV ViewCamera viewCamera(const FrameParams& P, const float4* __restrict__ lights, int v)
{
    const float4* c = lights + 2 * (P.nLights + P.nSph) + CGRT_VIEW_F4 * v;
    const float4 a = __ldg(c), q = __ldg(c + 1), h = __ldg(c + 2);
    return ViewCamera{mk3(a), a.w, h.x, q};
}
RT_DEV V3 primaryDirection(const FrameParams& P, const ViewCamera& C, int x, int y)
{
    const float px = float(x) / P.width * 2.0f - 1.0f;
    const float py = float(y) / P.height * 2.0f - 1.0f;
    const V3 cam = normalize3(mk3(-px * C.halfW, py * C.halfH, 1.0f));
    return quatRotate(C.q, cam);
}
RT_DEV V3 primaryDirection(const FrameParams& P, int x, int y)
{
    return primaryDirection(P, ViewCamera{mk3(P.camX, P.camY, P.camZ), P.halfW, P.halfH, make_float4(P.qx, P.qy, P.qz, P.qw)}, x, y);
}

// local pixel slot -> (x, y, output index). Slots enumerate this rank's tiles (8x4 pixel patches per warp for coherence).
RT_DEV bool slotToPixel(const FrameParams& P, const int* __restrict__ tileList, int slot, int& x, int& y, int& outIdx)
{
    const int tpx = P.tileW * P.tileH;
    const int lt = slot / tpx, q = slot - lt * tpx;
    const int g = tileList ? __ldg(tileList + lt) : lt;
    const int ty = g / P.tilesX, tx = g - ty * P.tilesX;
    x = tx * P.tileW + q % P.tileW;
    y = ty * P.tileH + q / P.tileW;
    if (x >= P.width || y >= P.height) return false;
    outIdx = (P.world == 1) ? ((P.height - 1 - y) * P.width + x) : slot; // Screen::setPixel row flip, src/screen.cpp:34
    return true;
}

// Slots of a frame of K = P.nViews views (cgrt_render_views): the views are interleaved tile by tile in the centre-out tile
// order, slot s = (k * K + v) * tpx + q with k the position in the one-view tile sequence, v the view and q the pixel in the
// tile, so the centre tiles of every view start first. K = 1 is the one-view numbering. Returns k; `single` = k * tpx + q is
// the slot of the same pixel in a frame of view v alone. VIEWS = false: a kernel instantiated for frames of one view only
// (K = 1 at compile time, no decode work).
template <bool VIEWS = true>
RT_DEV int decodeSlot(const FrameParams& P, int slot, int& v, int& q, int& single)
{
    const int tpx = P.tileW * P.tileH;
    const int K = VIEWS ? P.nViews : 1;
    const int kv = slot / tpx;
    q = slot - kv * tpx;
    const int k = kv / K;
    v = kv - k * K;
    single = k * tpx + q;
    return k;
}

// production form: processing position -> (global tile id, local tile index) through the per-frame tile sequence (tiles in
// centre-out order so that the long mirror chains of the object start first and the trivially missing border pixels fill the
// end of the launch). outIdx: Screen layout when P.screenLayout (single GPU, or direct writes into the peer-mapped frame of
// rank 0; view v's frame starts at pixel v * W * H), else the position in this rank's tile-major buffer; `local` is that
// position in either case. v = the view of the slot.
template <bool VIEWS = true>
RT_DEV bool seqToPixel(const FrameParams& P, const int2* __restrict__ tileSeq, int slot, int& x, int& y, int& outIdx, int& local,
                       int& v)
{
    const int tpx = P.tileW * P.tileH;
    int q, single;
    const int k = decodeSlot<VIEWS>(P, slot, v, q, single);
    const int2 e = __ldg(tileSeq + k);
    const int ty = e.x / P.tilesX, tx = e.x - ty * P.tilesX;
    x = tx * P.tileW + q % P.tileW;
    y = ty * P.tileH + q / P.tileW;
    local = e.y * tpx + q;
    if (x >= P.width || y >= P.height) return false;
    // Screen::setPixel row flip, src/screen.cpp:34
    outIdx = P.screenLayout ? (v * P.height + (P.height - 1 - y)) * P.width + x : local;
    return true;
}
RT_DEV bool seqToPixel(const FrameParams& P, const int2* __restrict__ tileSeq, int slot, int& x, int& y, int& outIdx, int& local)
{
    int v;
    return seqToPixel(P, tileSeq, slot, x, y, outIdx, local, v);
}

// warp-aggregated queue push: one atomic per warp, slots handed out by lane rank (ballot / popc / shfl)
RT_DEV int warpPush(int* counter, bool want)
{
    const unsigned mask = __ballot_sync(0xffffffffu, want);
    if (mask == 0u) return -1;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(mask) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(counter, __popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    return want ? base + __popc(mask & ((1u << lane) - 1u)) : -1;
}

// bounding box of the coloured pixels (CGRT_CNT_BBOX): one atomic per warp and bound
RT_DEV void noteColoured(int* bbox, bool wrote, int x, int row, int W, int H)
{
    const unsigned m = __ballot_sync(0xffffffffu, wrote);
    if (m == 0u) return;
    const int a = __reduce_max_sync(0xffffffffu, wrote ? x + 1 : 0), b = __reduce_max_sync(0xffffffffu, wrote ? row + 1 : 0);
    const int c = __reduce_max_sync(0xffffffffu, wrote ? W - x : 0), d = __reduce_max_sync(0xffffffffu, wrote ? H - row : 0);
    if ((threadIdx.x & 31) == 0) {
        if (a > bbox[0]) atomicMax(bbox + 0, a);
        if (b > bbox[1]) atomicMax(bbox + 1, b);
        if (c > bbox[2]) atomicMax(bbox + 2, c);
        if (d > bbox[3]) atomicMax(bbox + 3, d);
    }
}
RT_DEV void storeRGB(float* fb, int idx, const V3& c)
{
    fb[3 * (size_t)idx + 0] = c.x;
    fb[3 * (size_t)idx + 1] = c.y;
    fb[3 * (size_t)idx + 2] = c.z;
}

// ---- counting wavefront (CGRT_RENDER_COUNT): one launch per ray class and level, sequential leaf scans -----------------------
// colour of a path whose trace() at `level` returned `c`: unwind shade() of the levels above,
// color = directColor + reflectedColor * ks  (src/main.cpp:263), innermost first, exactly as the recursion returns.
RT_DEV V3 foldPath(const float4* __restrict__ pathState, size_t cap, int level, int pathId, V3 c)
{
    for (int j = level - 1; j >= 0; j--) {
        const float4 dr = pathState[((size_t)j * cap + pathId) * 2];
        const float4 ks = pathState[((size_t)j * cap + pathId) * 2 + 1];
        c = mk3(dr) + c * mk3(ks);
    }
    return c;
}

// Hit record (3 x float4) of the shade queue:  [P | matId] [N | outIdx] [D | pathId]
RT_DEV void pushHitRecord(const DevScene& S, const CountBuffers& B, int level, bool hit, const TraceResult& R, const V3& o,
                          const V3& d, int outIdx, int pathId)
{
    const int slot = warpPush(B.counts + CGRT_CNT_HIT + level, hit);
    if (!hit) return;
    V3 nn;
    int mat;
    if (R.sphere >= 0) {
        nn = R.sphereN;
        // hitInfo.material stays at the last accepted triangle's material (or the default HitInfo), bvh.cpp:878-879
        mat = R.tri >= 0 ? f2i(__ldg(S.triV1 + R.tri).w) : -1;
    } else {
        const int i = R.tri;
        const float4 v0 = __ldg(S.triV0 + i), v1 = __ldg(S.triV1 + i), v2 = __ldg(S.triV2 + i);
        const float4 n0 = __ldg(S.triN0 + i), n1 = __ldg(S.triN1 + i), n2 = __ldg(S.triN2 + i);
        const float4 pl = __ldg(S.triPl + i);
        float al, be, ga;
        hitEpilogue(mk3(v0), mk3(v1), mk3(v2), mk3(n0), mk3(n1), mk3(n2), mk3(pl), o, d, R.t, al, be, ga, nn);
        mat = f2i(v1.w);
    }
    const V3 P = o + d * R.t; // pointOn, src/main.cpp:164
    float4* rec = B.hitQ + 3 * (size_t)slot;
    rec[0] = make_float4(P.x, P.y, P.z, i2f(mat));
    rec[1] = make_float4(nn.x, nn.y, nn.z, i2f(outIdx));
    rec[2] = make_float4(d.x, d.y, d.z, i2f(pathId));
}

// warp-reduce the per-ray test counts, one 64-bit atomic per warp and counter
RT_DEV void accumulateTests(unsigned long long* tests, int cls, uint32_t nBox, uint32_t nTri)
{
    const uint32_t sb = __reduce_add_sync(0xffffffffu, nBox), stt = __reduce_add_sync(0xffffffffu, nTri);
    if ((threadIdx.x & 31) == 0) {
        if (sb) atomicAdd(tests + 2 * cls, (unsigned long long)sb);
        if (stt) atomicAdd(tests + 2 * cls + 1, (unsigned long long)stt);
    }
}

// ---- level 0: ray generation + closest hit ------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_primary(DevScene S, const FrameParams* __restrict__ Pp, CountBuffers B,
                                                 const int* __restrict__ tileList, float* __restrict__ fb)
{
    const FrameParams P = *Pp;
    const int n = P.nSlots;
    for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const int slot = base + threadIdx.x;
        int x = 0, y = 0, outIdx = 0;
        const bool valid = slot < n && slotToPixel(P, tileList, slot, x, y, outIdx);
        bool hit = false;
        TraceResult R;
        V3 o = mk3(P.camX, P.camY, P.camZ), d = mk3(0.0f, 0.0f, 0.0f);
        uint32_t nb = 0, nt = 0;
        if (valid) {
            d = primaryDirection(P, x, y);
            hit = traverseStrict<false, true>(S, o, d, FLT_MAX, 0.0f, 0.0f, R, nb, nt);
            if (!hit) storeRGB(fb, outIdx, mk3(0.0f, 0.0f, 0.0f)); // trace(): miss -> black, src/main.cpp:288-294
        } else if (slot < n && P.world > 1) {
            storeRGB(fb, slot, mk3(0.0f, 0.0f, 0.0f)); // padding pixels of edge tiles in the tile-major buffer
        }
        accumulateTests(B.tests, 0, nb, nt);
        pushHitRecord(S, B, 0, hit, R, o, d, outIdx, -1);
    }
}

// ---- level >= 1: closest hit over the compacted bounce queue --------------------------------------------------------------
__global__ void __launch_bounds__(128) k_bounce_closest(DevScene S, CountBuffers B, int level, float* __restrict__ fb)
{
    const int n = B.counts[CGRT_CNT_BOUNCE + level];
    for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const int i = base + threadIdx.x;
        const bool valid = i < n;
        bool hit = false;
        TraceResult R;
        V3 o = mk3(0.0f, 0.0f, 0.0f), d = o;
        int pathId = -1, outIdx = 0;
        uint32_t nb = 0, nt = 0;
        if (valid) {
            const float4 r0 = B.bounceQ[2 * (size_t)i], r1 = B.bounceQ[2 * (size_t)i + 1];
            o = mk3(r0);
            d = mk3(r1);
            pathId = f2i(r1.w);
            outIdx = B.pathPix[pathId];
            hit = traverseStrict<false, true>(S, o, d, r0.w, 0.0f, 0.0f, R, nb, nt);
            if (!hit) // reflected colour is black; unwind the levels above (src/main.cpp:288-294 then :263)
                storeRGB(fb, outIdx, foldPath(B.pathState, B.cap, level, pathId, mk3(0.0f, 0.0f, 0.0f)));
        }
        accumulateTests(B.tests, 1, nb, nt);
        pushHitRecord(S, B, level, hit, R, o, d, outIdx, pathId);
    }
}

// ---- any-hit shadow rays: one thread per (hit, light).  pointInShadow, src/main.cpp:104-135 -------------------------------
// Runs the reference's full closest-hit query (that is what src/main.cpp:115 does and what the roofline arithmetic charges a
// shadow ray with) and applies the predicate to its result: same answer as an any-hit query, no early exit.
__global__ void __launch_bounds__(128) k_shadow(DevScene S, const FrameParams* __restrict__ Pp,
                                                const float4* __restrict__ lights, CountBuffers B, int level)
{
    const int nL = Pp->nLights;
    const int n = B.counts[CGRT_CNT_HIT + level] * nL;
    for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const int i = base + threadIdx.x;
        uint32_t nb = 0, nt = 0;
        if (i < n) {
            const int h = i / nL, l = i - h * nL;
            const float4 a = B.hitQ[3 * (size_t)h];
            const V3 pointOn = mk3(a);
            const V3 lightPos = mk3(__ldg(lights + 2 * l));
            const V3 fromPosToLight = lightPos - pointOn;
            const V3 dir = normalize3(fromPosToLight);
            const float epsilon = 0.001f;
            const V3 org = pointOn + epsilon * dir;
            const float dist = length3(fromPosToLight);
            TraceResult R;
            const bool hit = traverseStrict<false, true>(S, org, dir, FLT_MAX, 0.0f, 0.0f, R, nb, nt);
            const bool shadowed = hit && !(R.t + epsilon >= dist);
            B.lit[i] = shadowed ? 0 : 1;
        }
        accumulateTests(B.tests, 2, nb, nt);
    }
}

// =================================================================================================================
// Persistent warps over the exact traversal: the path pipeline's closest-hit and shadow kernels.
// Every lane owns a resumable traversal (Trav). Between bursts of steps, lanes whose ray is finished hand in their result
// (collectively, so that queue pushes stay warp-aggregated) and are given the next ray from a global work counter, so a warp
// keeps its lanes busy instead of idling until its slowest ray is done; rays that miss the root box (most primary rays)
// cost one converged refill round. A Policy supplies the rays and consumes the results:
//     bool load(int idx, V3& o, V3& d, float& tIn, float& eps, float& maxDist)   false = nothing to trace for this index
//     bool retire(bool fin, int idx, bool traced, bool result, const TraceResult& R, const V3& ro, const V3& rd, V3& o, V3& d, float& tIn)
//          called by ALL lanes; returns true when the lane continues with a follow-up ray (o, d, tIn) of the same item
// =================================================================================================================
#ifndef CGRT_STEPS_PER_ROUND
#define CGRT_STEPS_PER_ROUND 24
#endif
#ifndef CGRT_MINBLOCKS
#define CGRT_MINBLOCKS 8 // 8 CTAs x 4 warps per SM: caps the traversal kernels at 64 registers
#endif
#define CGRT_REFILL_MIN_IDLE 6
// Launch-time knobs (environment CGRT_TUNE="blocks=8,chains=4,coop=30000,waveblocks=4" overrides the defaults at library load;
// unknown keys are ignored; they change speed only, never results)
struct Tuning {
    int blocks = 8;  // persistent CTAs (128 threads) per SM of the path pipeline's, the round pipeline's and the batch queries' searches
    int chains = 0;    // round pipeline: independent pixel subsets rendered on separate streams so that the tail of one
                       // subset's launch is filled by the other subsets' work; 0 = by frame size (4 for a 1080p frame on one GPU)
    int coop = 0;      // round pipeline: rounds with fewer rays than this are searched by k_trace8 (8 lanes per ray: low
                       // latency), larger ones by k_trace (1 lane per ray: higher throughput)
    int waveBlocks = 0; // persistent wavefront: CTAs per SM (0 = as many as fit)
};
static Tuning g_tune;
static bool g_tuneLoaded = false;
static const Tuning& tuning()
{
    if (!g_tuneLoaded) {
        g_tuneLoaded = true;
        const char* e = getenv("CGRT_TUNE");
        if (e) {
            std::string s(e);
            size_t pos = 0;
            while (pos < s.size()) {
                size_t c = s.find(',', pos);
                if (c == std::string::npos) c = s.size();
                const std::string kv = s.substr(pos, c - pos);
                const size_t eq = kv.find('=');
                if (eq != std::string::npos) {
                    const std::string key = kv.substr(0, eq);
                    const int v = atoi(kv.c_str() + eq + 1);
                    if (key == "blocks") g_tune.blocks = v;
                    else if (key == "coop") g_tune.coop = v;
                    else if (key == "chains") g_tune.chains = v;
                    else if (key == "waveblocks") g_tune.waveBlocks = v;
                }
                pos = c + 1;
            }
        }
    }
    return g_tune;
}

#ifdef CGRT_INSTRUMENT
// [0] iterations, [1] lanes running summed over iterations, [2..4] iterations that chose class k, [5..7] lanes stepped in
// class k, [8] refill rounds, [9] lanes refilled, [10] retire rounds, [11] lanes retired, [12] cycles in steps,
// [13] cycles in refill, [14] cycles in retire, [15] warps
__device__ unsigned long long g_instr[16];
// timeline: per kernel kind (0 closest, 1 any) and 25 us bucket since the first burst of the launch: [warps bursting, lanes running]
__device__ unsigned long long g_t0[2];
__device__ unsigned int g_tl[2][128][2];
__device__ unsigned int g_stepHist[64]; // k_trace: rays by number of steps (bucket = steps / 8, last bucket open)
// the value is evaluated by ALL lanes (it may contain warp collectives); lane 0 adds it
#define INSTR_ADD(i, v) do { const unsigned long long v_ = (unsigned long long)(v); if ((threadIdx.x & 31) == 0) atomicAdd(&g_instr[i], v_); } while (0)
#else
#define INSTR_ADD(i, v) do { } while (0)
#endif

template <bool ANY, class Policy>
RT_DEV void persistentTraverse(const DevScene& S, Policy& P, int n, int* workCounter)
{
    Trav T;
    TravStack K;
    int idx = -1;               // work item owned by this lane, -1 = idle
    int state = TRAV_DONE;
    bool traced = false;        // the item produced a ray (load() returned true)
    float tIn = 0.0f, eps = 0.0f, maxDist = 0.0f;
    bool exhausted = false;     // warp-uniform: the work counter has run past n
    const int lane = threadIdx.x & 31;
    const unsigned ltMask = (1u << lane) - 1u;
    INSTR_ADD(15, 1);
    while (true) {
        // ---- refill
        const unsigned idle = __ballot_sync(0xffffffffu, idx < 0);
        const int nIdle = __popc(idle);
        if (!exhausted && (nIdle >= CGRT_REFILL_MIN_IDLE || idle == 0xffffffffu)) {
#ifdef CGRT_INSTRUMENT
            const long long c0 = clock64();
#endif
            const int leader = __ffs(idle) - 1;
            int base = 0;
            if (lane == leader) base = atomicAdd(workCounter, nIdle);
            base = __shfl_sync(0xffffffffu, base, leader);
            if (base + nIdle >= n) exhausted = true;
            if (idx < 0) {
                const int mine = base + __popc(idle & ltMask);
                if (mine < n) {
                    idx = mine;
                    V3 o, d;
                    traced = P.load(idx, o, d, tIn, eps, maxDist);
                    state = TRAV_DONE;
                    if (traced) {
                        if (travBegin(S, T, o, d, tIn)) state = TRAV_CONTINUE;
                    }
                }
            }
#ifdef CGRT_INSTRUMENT
            INSTR_ADD(8, 1); INSTR_ADD(9, nIdle); INSTR_ADD(13, clock64() - c0);
#endif
        }
        // ---- retire finished lanes (collective) BEFORE stepping: fresh rays that miss the root box (most primary rays) are
        // retired and replaced right away, in converged refill rounds, until the warp holds enough live rays
        {
            const bool fin = idx >= 0 && state != TRAV_CONTINUE;
            if (__ballot_sync(0xffffffffu, fin) != 0u) {
#ifdef CGRT_INSTRUMENT
                const long long c0 = clock64();
                INSTR_ADD(10, 1); INSTR_ADD(11, __popc(__ballot_sync(0xffffffffu, fin)));
#endif
                TraceResult R;
                R.sphere = -1; R.tri = -1; R.t = tIn;
                bool result = false;
                if (fin && traced) result = travFinish<ANY>(S, T, state, eps, maxDist, R);
                V3 no, nd;
                const bool again = P.retire(fin, idx, traced, result, R, T.o, T.d, no, nd, tIn);
                if (fin) {
                    if (again) {
                        state = travBegin(S, T, no, nd, tIn) ? TRAV_CONTINUE : TRAV_DONE;
                    } else {
                        idx = -1;
                    }
                }
#ifdef CGRT_INSTRUMENT
                INSTR_ADD(14, clock64() - c0);
#endif
                continue;
            }
        }
        if (__ballot_sync(0xffffffffu, idx >= 0) == 0u) {
            if (exhausted) break;
            continue;
        }
        // ---- a burst of steps
        // Each iteration executes ONE node class, chosen by a warp vote that maximises lanes-advanced per instruction
        // (a lane waiting at a sub-tree leaf counts twice, the node classes once); lanes waiting in another class keep their
        // state. This trades a little latency for not paying all three code paths on every iteration.
#ifdef CGRT_INSTRUMENT
        const long long cs0 = clock64();
        {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            const int nRun = __popc(__ballot_sync(0xffffffffu, idx >= 0 && state == TRAV_CONTINUE));
            if (lane == 0) {
                const unsigned long long old = atomicMin(&g_t0[ANY ? 1 : 0], now);
                const unsigned long long t0 = old < now ? old : now;
                int b = (int)((now - t0) / 25000ull);
                if (b > 127) b = 127;
                atomicAdd(&g_tl[ANY ? 1 : 0][b][0], 1u);
                atomicAdd(&g_tl[ANY ? 1 : 0][b][1], (unsigned)nRun);
            }
        }
#endif
#pragma unroll 1
        for (int it = 0; it < CGRT_STEPS_PER_ROUND; it++) {
            const bool run = idx >= 0 && state == TRAV_CONTINUE;
#ifdef CGRT_INSTRUMENT
            INSTR_ADD(0, 1); INSTR_ADD(1, __popc(__ballot_sync(0xffffffffu, run)));
#endif
            const int cls = run ? travClass(T.node) : CLS_NONE;
            const int s0 = __popc(__ballot_sync(0xffffffffu, cls == CLS_REF));
            const int s1 = __popc(__ballot_sync(0xffffffffu, cls == CLS_WIDE));
            const int s2 = __popc(__ballot_sync(0xffffffffu, cls == CLS_LEAF)) * 2;
            if ((s0 | s1 | s2) == 0) break;
            if (s0 >= s1 && s0 >= s2) {
                INSTR_ADD(2, 1); INSTR_ADD(5, s0);
                if (cls == CLS_REF) state = travStepRef(S, T, K);
            } else if (s1 >= s2) {
                INSTR_ADD(3, 1); INSTR_ADD(6, s1);
                if (cls == CLS_WIDE) state = travStepWide(S, T, K);
            } else {
                INSTR_ADD(4, 1); INSTR_ADD(7, s2 / 2);
                if (cls == CLS_LEAF) state = travStepLeaf<ANY>(S, T, K, eps, maxDist);
            }
        }
#ifdef CGRT_INSTRUMENT
        INSTR_ADD(12, clock64() - cs0);
#endif
    }
}

// =================================================================================================================
// Path pipeline: k_paths -> k_shadow_all -> k_shade_paths
// Renders the frames of scenes without a fast tree, and frames with too many lit flags for the round pipeline's ray records.
// =================================================================================================================
// getFinalColor/trace/shade (src/main.cpp:241-310) for one pixel is a chain: primary ray, then one reflection ray per
// mirror hit while level + 1 < trace limit. A lane of k_paths follows that chain itself (the follow-up ray of shade(),
// main.cpp:252-256, is handed straight back to the traversal), so the chain costs no kernel boundary; the shadow rays
// (pointInShadow) do not influence the chain and are traced afterwards for all levels at once.
// FROMQ = false: work items are pixel slots (primary rays); FROMQ = true: work items are records of the replay queue, i.e.
// rays of any level that the speculative kernel could not certify (the chain continues from there in the same lane).
// VIEWS = false: frames of one camera, whose primary rays come from FrameParams (k_paths / k_paths_fast are instantiated for
// both, so that a single frame's persistent loop carries nothing of the view decode).
template <bool FROMQ, bool VIEWS = false>
struct PathsPolicy {
    const DevScene& S;
    const FrameParams& P;
    const PathBuffers& B;
    const int2* tileSeq;
    const float4* lights; // parameter block after the header (the views' cameras follow the lights)
    float* fb;
    int outIdx, level, path; // per lane
    RT_DEV bool load(int slot, V3& o, V3& d, float& tIn, float& eps, float& maxDist)
    {
        eps = 0.0f;
        maxDist = 0.0f;
        if (FROMQ) {
            const float4 a = B.replayQ[3 * (size_t)slot], b = B.replayQ[3 * (size_t)slot + 1], c = B.replayQ[3 * (size_t)slot + 2];
            o = mk3(a);
            tIn = a.w;
            d = mk3(b);
            level = f2i(b.w);
            path = f2i(c.x);
            outIdx = f2i(c.y);
            return true;
        }
        int x, y, local, v;
        level = 0;
        path = -1;
        if (!seqToPixel<VIEWS>(P, tileSeq, slot, x, y, outIdx, local, v)) {
            outIdx = -1 - local; // padding pixel of an edge tile
            return false;
        }
        if (VIEWS) {
            const ViewCamera C = viewCamera(P, lights, v);
            o = C.o;
            d = primaryDirection(P, C, x, y);
        } else {
            o = mk3(P.camX, P.camY, P.camZ);
            d = primaryDirection(P, x, y);
        }
        tIn = FLT_MAX;
        return true;
    }
    // the speculative kernel hands a ray it cannot certify to the exact kernel (rare: one atomic per ray is fine)
    RT_DEV void defer(const V3& o, const V3& d, float tIn)
    {
        const int q = atomicAdd(B.counts + CGRT_CNT_REPLAY_PATHS, 1);
        float4* r = B.replayQ + 3 * (size_t)q;
        r[0] = make_float4(o.x, o.y, o.z, tIn);
        r[1] = make_float4(d.x, d.y, d.z, i2f(level));
        r[2] = make_float4(i2f(path), i2f(outIdx), 0.0f, 0.0f);
    }
    RT_DEV bool retire(bool fin, int slot, bool traced, bool hit, const TraceResult& R, const V3& ro, const V3& rd, V3& no, V3& nd, float& nt)
    {
        const bool isHit = fin && traced && hit;
        const int newPath = warpPush(B.counts + CGRT_CNT_PATHS, isHit && level == 0);
        const int listPos = warpPush(B.counts + CGRT_CNT_HITS, isHit);
        bool again = false;
        if (fin) {
            if (!traced) {
                if (!P.screenLayout) storeRGB(fb, -1 - outIdx, mk3(0.0f, 0.0f, 0.0f)); // padding pixels (tile-major buffer)
            } else if (!hit) {
                if (level == 0) storeRGB(fb, outIdx, mk3(0.0f, 0.0f, 0.0f)); // trace(): miss -> black, main.cpp:288-294
            } else {
                if (level == 0) {
                    path = newPath;
                    B.pathPix[path] = outIdx;
                }
                V3 nn;
                int mat;
                if (R.sphere >= 0) {
                    nn = R.sphereN;
                    mat = R.tri >= 0 ? f2i(__ldg(S.triV1 + R.tri).w) : -1;
                } else {
                    const int i = R.tri;
                    const float4 v0 = __ldg(S.triV0 + i), v1 = __ldg(S.triV1 + i), v2 = __ldg(S.triV2 + i);
                    const float4 n0 = __ldg(S.triN0 + i), n1 = __ldg(S.triN1 + i), n2 = __ldg(S.triN2 + i);
                    const float4 pl = __ldg(S.triPl + i);
                    float al, be, ga;
                    hitEpilogue(mk3(v0), mk3(v1), mk3(v2), mk3(n0), mk3(n1), mk3(n2), mk3(pl), ro, rd, R.t, al, be, ga, nn);
                    mat = f2i(v1.w);
                }
                const V3 pointOn = ro + rd * R.t; // main.cpp:164
                const int rec = path * B.levels + level;
                float4* r = B.hitRec + 3 * (size_t)rec;
                r[0] = make_float4(pointOn.x, pointOn.y, pointOn.z, i2f(mat));
                r[1] = make_float4(nn.x, nn.y, nn.z, 0.0f);
                r[2] = make_float4(rd.x, rd.y, rd.z, 0.0f);
                B.hitList[listPos] = rec;
                B.pathDepth[path] = level + 1;
                const float ksz = mat >= 0 ? __ldg(S.mats + 2 * mat + 1).z : 0.0f;
                if (!(ksz <= 0.01f) && level + 1 < P.traceLimit) { // shade(): mirror test main.cpp:246, trace limit :267
                    const V3 reflected = normalize3(reflect3(rd, nn)); // ComputeReflectedRay, main.cpp:252-256
                    nt = length3(rd);
                    const float epsilon = 0.001f;
                    no = pointOn + epsilon * reflected;
                    nd = reflected;
                    level++;
                    again = true;
                }
            }
        }
        const unsigned am = __ballot_sync(0xffffffffu, again);
        if (am && (threadIdx.x & 31) == __ffs(am) - 1) atomicAdd(B.counts + CGRT_CNT_BOUNCES, __popc(am));
        return again;
    }
};

// =================================================================================================================
// Persistent warps over the SPECULATIVE traversal (cgrt_device.cuh): same refill / retire skeleton as persistentTraverse,
// two node classes (8-wide conservative node, triangle leaf), and a third way for a ray to end - "defer": the lane hands
// the ray to the Policy's replay queue, which the exact kernel drains afterwards.
// =================================================================================================================
#ifndef CGRT_FAST_STEPS
#define CGRT_FAST_STEPS 8
#endif
#ifndef CGRT_FAST_MINBLOCKS
#define CGRT_FAST_MINBLOCKS 8
#endif
template <bool ANY, class Policy>
RT_DEV void persistentFast(const DevScene& S, Policy& P, int n, int* workCounter)
{
    FastTrav T;
    FastStack K;
    int idx = -1;
    int state = TRAV_DONE;
    bool traced = false;
    float tIn = 0.0f, eps = 0.0f, maxDist = 0.0f;
    bool exhausted = false;
    const int lane = threadIdx.x & 31;
    const unsigned ltMask = (1u << lane) - 1u;
    INSTR_ADD(15, 1);
    while (true) {
        // ---- refill
        const unsigned idle = __ballot_sync(0xffffffffu, idx < 0);
        const int nIdle = __popc(idle);
        if (!exhausted && (nIdle >= CGRT_REFILL_MIN_IDLE || idle == 0xffffffffu)) {
            const int leader = __ffs(idle) - 1;
            int base = 0;
            if (lane == leader) base = atomicAdd(workCounter, nIdle);
            base = __shfl_sync(0xffffffffu, base, leader);
            if (base + nIdle >= n) exhausted = true;
            if (idx < 0) {
                const int mine = base + __popc(idle & ltMask);
                if (mine < n) {
                    idx = mine;
                    V3 o, d;
                    traced = P.load(idx, o, d, tIn, eps, maxDist);
                    state = traced ? fastStart<ANY>(S, T, K, o, d, tIn, eps, maxDist) : TRAV_DONE;
                }
            }
            INSTR_ADD(8, 1); INSTR_ADD(9, nIdle);
        }
        // ---- retire finished lanes (collective)
        {
            const bool fin = idx >= 0 && state != TRAV_CONTINUE;
            if (__ballot_sync(0xffffffffu, fin) != 0u) {
                INSTR_ADD(10, 1); INSTR_ADD(11, __popc(__ballot_sync(0xffffffffu, fin)));
                TraceResult R;
                R.sphere = -1; R.tri = -1; R.t = tIn;
                bool result = false, defer = false;
                if (fin && traced) result = fastFinish<ANY>(S, T, K.t2, state, tIn, eps, maxDist, R, defer);
                if (fin && defer) P.defer(T.o, T.d, tIn);
                V3 no, nd;
                const bool again = P.retire(fin && !defer, idx, traced, result, R, T.o, T.d, no, nd, tIn);
                if (fin) {
                    if (again) state = fastStart<ANY>(S, T, K, no, nd, tIn, eps, maxDist);
                    else idx = -1;
                }
                continue;
            }
        }
        if (__ballot_sync(0xffffffffu, idx >= 0) == 0u) {
            if (exhausted) break;
            continue;
        }
        // ---- a burst of steps: each iteration runs the node class most running lanes wait in
#ifdef CGRT_INSTRUMENT
        {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            const int nRun = __popc(__ballot_sync(0xffffffffu, idx >= 0 && state == TRAV_CONTINUE));
            if (lane == 0) {
                const unsigned long long old = atomicMin(&g_t0[ANY ? 1 : 0], now);
                const unsigned long long t0 = old < now ? old : now;
                int b = (int)((now - t0) / 25000ull);
                if (b > 127) b = 127;
                atomicAdd(&g_tl[ANY ? 1 : 0][b][0], 1u);
                atomicAdd(&g_tl[ANY ? 1 : 0][b][1], (unsigned)nRun);
            }
        }
#endif
#pragma unroll 1
        for (int it = 0; it < CGRT_FAST_STEPS; it++) {
            const bool run = idx >= 0 && state == TRAV_CONTINUE;
            const bool leaf = run && travIsLeaf(T.node);
            const int sAll = __popc(__ballot_sync(0xffffffffu, run));
            const int sLeaf = __popc(__ballot_sync(0xffffffffu, leaf));
            INSTR_ADD(0, 1); INSTR_ADD(1, sAll);
            if (sAll == 0) break;
            if (sAll - sLeaf >= sLeaf) {
                INSTR_ADD(2, 1); INSTR_ADD(5, sAll - sLeaf);
                if (run && !leaf) state = fastStepWide<ANY>(S, T, K, maxDist);
            } else {
                INSTR_ADD(4, 1); INSTR_ADD(7, sLeaf);
                if (leaf) state = fastStepLeaf<ANY>(S, T, K, eps, maxDist);
            }
        }
    }
}

template <bool VIEWS>
__global__ void __launch_bounds__(128, CGRT_FAST_MINBLOCKS) k_paths_fast(DevScene S, const FrameParams* __restrict__ Pp, PathBuffers B,
                                                    const int2* __restrict__ tileSeq, const float4* __restrict__ lights,
                                                    float* __restrict__ fb, int* work)
{
    const FrameParams P = *Pp;
    PathsPolicy<false, VIEWS> pol{S, P, B, tileSeq, lights, fb, -1, 0, -1};
    persistentFast<false>(S, pol, P.nSlots, work);
}

// exact traversal: all pixels (scenes without a fast tree) ...
template <bool VIEWS>
__global__ void __launch_bounds__(128, CGRT_MINBLOCKS) k_paths(DevScene S, const FrameParams* __restrict__ Pp, PathBuffers B,
                                               const int2* __restrict__ tileSeq, const float4* __restrict__ lights,
                                               float* __restrict__ fb, int* work)
{
    const FrameParams P = *Pp;
    PathsPolicy<false, VIEWS> pol{S, P, B, tileSeq, lights, fb, -1, 0, -1};
    persistentTraverse<false>(S, pol, P.nSlots, work);
}

// ... or the rays k_paths_fast deferred
__global__ void __launch_bounds__(128, CGRT_MINBLOCKS) k_paths_replay(DevScene S, const FrameParams* __restrict__ Pp, PathBuffers B,
                                                      float* __restrict__ fb, int* work)
{
    const int n = B.counts[CGRT_CNT_REPLAY_PATHS];
    if (n == 0) return;
    const FrameParams P = *Pp;
    PathsPolicy<true> pol{S, P, B, nullptr, nullptr, fb, -1, 0, -1};
    persistentTraverse<false>(S, pol, n, work);
}

// trace limit 0 with direct writes into a shared frame: black for this rank's pixels only
__global__ void k_clear_tiles(const FrameParams* __restrict__ Pp, const int2* __restrict__ tileSeq, float* __restrict__ fb)
{
    const FrameParams P = *Pp;
    for (int slot = blockIdx.x * blockDim.x + threadIdx.x; slot < P.nSlots; slot += gridDim.x * blockDim.x) {
        int x, y, outIdx, local;
        if (seqToPixel(P, tileSeq, slot, x, y, outIdx, local)) storeRGB(fb, outIdx, mk3(0.0f, 0.0f, 0.0f));
    }
}

template <bool FROMQ>
struct ShadowAllPolicy {
    const PathBuffers& B;
    const float4* lights;
    int nL;
    int item; // per lane: (hit record, light) work item = index of the lit flag
    RT_DEV bool load(int i, V3& o, V3& d, float& tIn, float& eps, float& maxDist)
    { // pointInShadow, src/main.cpp:104-135
        int rec, l;
        if (FROMQ) {
            item = B.replayShadow[i];
            rec = item / nL;
            l = item - rec * nL;
        } else {
            const int h = i / nL;
            l = i - h * nL;
            rec = B.hitList[h];
            item = rec * nL + l;
        }
        const V3 pointOn = mk3(B.hitRec[3 * (size_t)rec]);
        const V3 lightPos = mk3(__ldg(lights + 2 * l));
        const V3 fromPosToLight = lightPos - pointOn;
        d = normalize3(fromPosToLight);
        eps = 0.001f;
        o = pointOn + eps * d;
        tIn = FLT_MAX;
        maxDist = length3(fromPosToLight);
        return true;
    }
    RT_DEV void defer(const V3&, const V3&, float) { B.replayShadow[atomicAdd(B.counts + CGRT_CNT_REPLAY_SHADOW, 1)] = item; }
    RT_DEV bool retire(bool fin, int, bool, bool shadowed, const TraceResult&, const V3&, const V3&, V3&, V3&, float&)
    {
        if (fin) B.lit[item] = shadowed ? 0 : 1;
        return false;
    }
};

__global__ void __launch_bounds__(128, CGRT_FAST_MINBLOCKS) k_shadow_fast(DevScene S, const FrameParams* __restrict__ Pp,
                                                     const float4* __restrict__ lights, PathBuffers B, int* work)
{
    const int nL = Pp->nLights;
    ShadowAllPolicy<false> pol{B, lights, nL, 0};
    persistentFast<true>(S, pol, B.counts[CGRT_CNT_HITS] * nL, work);
}

__global__ void __launch_bounds__(128, CGRT_MINBLOCKS) k_shadow_all(DevScene S, const FrameParams* __restrict__ Pp,
                                                    const float4* __restrict__ lights, PathBuffers B, int* work)
{
    const int nL = Pp->nLights;
    ShadowAllPolicy<false> pol{B, lights, nL, 0};
    persistentTraverse<true>(S, pol, B.counts[CGRT_CNT_HITS] * nL, work);
}

__global__ void __launch_bounds__(128, CGRT_MINBLOCKS) k_shadow_replay(DevScene S, const FrameParams* __restrict__ Pp,
                                                       const float4* __restrict__ lights, PathBuffers B, int* work)
{
    const int n = B.counts[CGRT_CNT_REPLAY_SHADOW];
    if (n == 0) return;
    ShadowAllPolicy<true> pol{B, lights, Pp->nLights, 0};
    persistentTraverse<true>(S, pol, n, work);
}

// direct colour of one hit record: shading(), src/main.cpp:160-235 (point-light loop :220-232)
// CG: the lit flags were written by other SMs during this kernel (persistent wavefront): read them through L2
// nSph / soft: spherical lights (main.cpp:168-218) come first in the sum: (diffuse + specular of a point light at the centre)
// times the fraction of the light's 200 sample rays that arrive (k_soft_shadows)
template <bool CG = false>
RT_DEV V3 directColour(const DevScene& S, const float4* __restrict__ lights, int nL, const float4& a, const float4& b,
                       const float4& c, const uint8_t* __restrict__ lit, V3& ks, int nSph = 0, const float* __restrict__ soft = nullptr)
{
    const V3 P = mk3(a), N = mk3(b), D = mk3(c);
    const int mat = f2i(a.w);
    float4 m0 = make_float4(0.0f, 0.0f, 0.0f, 1.0f), m1 = make_float4(0.0f, 0.0f, 0.0f, 1.0f); // default HitInfo material
    if (mat >= 0) { m0 = __ldg(S.mats + 2 * mat); m1 = __ldg(S.mats + 2 * mat + 1); }
    const V3 kd = mk3(m0);
    ks = mk3(m1);
    const float shininess = m0.w;
    V3 result = mk3(0.0f, 0.0f, 0.0f);
    for (int l = 0; l < nSph; l++) {
        const V3 lightPos = mk3(__ldg(lights + 2 * (nL + l))), lightCol = mk3(__ldg(lights + 2 * (nL + l) + 1));
        const V3 fromPosToLight = normalize3(lightPos - P);
        V3 diffuse = mk3(0.0f, 0.0f, 0.0f), specular = diffuse;
        const float diffuseCos = dot3(fromPosToLight, N);
        if (!(diffuseCos <= 0)) diffuse = (lightCol * kd) * diffuseCos;
        const V3 reflected = normalize3(reflect3(D, N));
        const float specularCos = dot3(reflected, fromPosToLight);
        if (!(specularCos <= 0)) specular = (lightCol * ks) * (float)pow((double)specularCos, (double)shininess);
        const float softShadowCounter = soft[l];
        result = result + diffuse * softShadowCounter;
        result = result + specular * softShadowCounter;
    }
    for (int l = 0; l < nL; l++) {
        const V3 lightPos = mk3(__ldg(lights + 2 * l)), lightCol = mk3(__ldg(lights + 2 * l + 1));
        const V3 fromPosToLight = normalize3(lightPos - P);
        if (!(CG ? __ldcg(lit + l) : lit[l])) continue;
        V3 diffuse = mk3(0.0f, 0.0f, 0.0f), specular = diffuse;
        const float diffuseCos = dot3(fromPosToLight, N); // diffuseOneLight, main.cpp:84-98
        if (!(diffuseCos <= 0)) diffuse = (lightCol * kd) * diffuseCos;
        const V3 reflected = normalize3(reflect3(D, N)); // specularOneLight, main.cpp:61-82
        const float specularCos = dot3(reflected, fromPosToLight);
        if (!(specularCos <= 0)) {
            const float pw = (float)pow((double)specularCos, (double)shininess);
            specular = (lightCol * ks) * pw;
        }
        result = result + diffuse;
        result = result + specular;
    }
    return result;
}

// one thread per path: direct colour of every level, then the recursion unwound innermost first (main.cpp:241-264)
__global__ void __launch_bounds__(128) k_shade_paths(DevScene S, const FrameParams* __restrict__ Pp,
                                                     const float4* __restrict__ lights, PathBuffers B, float* __restrict__ fb)
{
    const int nL = Pp->nLights;
    const int n = B.counts[CGRT_CNT_PATHS];
    for (int path = blockIdx.x * blockDim.x + threadIdx.x; path < n; path += gridDim.x * blockDim.x) {
        const int depth = B.pathDepth[path];
        V3 direct[CGRT_MAX_LEVELS], ksv[CGRT_MAX_LEVELS];
        for (int k = 0; k < depth; k++) {
            const int rec = path * B.levels + k;
            const float4* r = B.hitRec + 3 * (size_t)rec;
            direct[k] = directColour(S, lights, nL, r[0], r[1], r[2], B.lit + (size_t)rec * nL, ksv[k]);
        }
        // deepest level: its reflection (if the surface is a mirror) is black - either the reflected ray missed or
        // trace(level + 1) hit the recursion limit (main.cpp:267-272)
        int k = depth - 1;
        V3 colour = (ksv[k].z <= 0.01f) ? direct[k] : direct[k] + mk3(0.0f, 0.0f, 0.0f) * ksv[k];
        for (k = depth - 2; k >= 0; k--) colour = direct[k] + colour * ksv[k];
        storeRGB(fb, B.pathPix[path], colour);
    }
}

// =================================================================================================================
// Round pipeline: k_gen -> { k_trace -> k_finish } per level -> k_shade_slots
// Renders the large shallow frames of scenes with a fast tree (k_wave renders the others; DESIGN 4.4).
// =================================================================================================================
// Measurements of the path pipeline above (profiles/r01_tuning.md) showed that its traversal kernels spent two thirds of their
// issued instructions outside traversal steps: ray set-up, certificate, fp64 hit epilogue and record keeping executed inside
// the persistent loop with a dozen of 32 lanes active. Here the persistent kernel does nothing but search steps; everything
// per-ray runs in flat, converged kernels before and after it, and rays of one warp are neighbours on the screen.
#ifndef CGRT_TRACE_STEPS
#define CGRT_TRACE_STEPS 8
#endif
#ifndef CGRT_TRACE_MINBLOCKS
#define CGRT_TRACE_MINBLOCKS 8
#endif
#ifndef CGRT_TRACE_REFILL
#define CGRT_TRACE_REFILL 4
#endif
#define CGRT_RAY_ANY 0x40000000 // ray record c.y: any-hit ray (value & 0x3fffffff = index of its lit flag); else the level

RT_DEV void writeRay(float4* q, const V3& o, float tIn, const V3& d, float maxDist, int slot, int meta, float eps)
{
    q[0] = make_float4(o.x, o.y, o.z, tIn);
    q[1] = make_float4(d.x, d.y, d.z, maxDist);
    q[2] = make_float4(i2f(slot), i2f(meta), eps, 0.0f);
}

// ---- level 0: ray generation + intersectDataStructure's root test; rays that enter are compacted in slot order ------------
// Chains: the tiles of the frame's sequence are dealt round-robin to `nChains` independent sub-frames (own ray lists, own
// counters, own stream); this launch generates the rays of sub-frame `chain`.
__global__ void __launch_bounds__(128) k_gen(DevScene S, const FrameParams* __restrict__ Pp, const float4* __restrict__ lights,
                                             RoundBuffers B, const int2* __restrict__ tileSeq, float* __restrict__ fb, int chain,
                                             int nChains)
{
    const FrameParams P = *Pp;
    const int tpx = P.tileW * P.tileH;
    const int nTiles = P.nSlots / tpx; // (tiles of all views)
    const int myTiles = nTiles > chain ? (nTiles - chain + nChains - 1) / nChains : 0;
    const int n = myTiles * tpx;
    for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const int i = base + threadIdx.x;
        const int slot = i < n ? ((i / tpx) * nChains + chain) * tpx + i % tpx : 0;
        bool push = false;
        V3 o = mk3(0.0f, 0.0f, 0.0f), d = mk3(0.0f, 0.0f, 0.0f);
        if (i < n) {
            int x, y, outIdx, local, v;
            B.pathDepth[slot] = 0;
            if (seqToPixel(P, tileSeq, slot, x, y, outIdx, local, v)) {
                const ViewCamera C = viewCamera(P, lights, v);
                o = C.o;
                d = primaryDirection(P, C, x, y);
                // a ray that does not enter the tree (bvh.cpp:831-844) can only hit spheres
                bool enter = S.nSpheres > 0;
                if (!enter && S.nNodes > 0) {
                    const float4 q0 = __ldg(S.nodes + 0), q1 = __ldg(S.nodes + 1);
                    enter = startsInBox(o, mk3(q0), mk3(q1));
                    if (!enter) {
                        float tmp;
                        enter = slabTest(mk3(q0), mk3(q1), o, d, FLT_MAX, tmp);
                    }
                }
                push = enter;
                if (!enter) storeRGB(fb, outIdx, mk3(0.0f, 0.0f, 0.0f)); // trace(): miss -> black, src/main.cpp:288-294
            } else if (!P.screenLayout) {
                storeRGB(fb, local, mk3(0.0f, 0.0f, 0.0f)); // padding pixels of edge tiles in the tile-major buffer
            }
        }
        const int q = warpPush(B.counts + CGRT_CNT_BOUNCE + 0, push);
        if (push) writeRay(B.cRay[0] + 3 * (size_t)q, o, FLT_MAX, d, __int_as_float(0x7f800000), slot, 0, 0.0f);
    }
}

// ---- the search: persistent warps, nothing but steps ------------------------------------------------------------------------
// Work items [0, nA) are the shadow rays of list A, [nA, nA + nB) the closest-hit rays of list B. A finished lane stores
// (state, t, tri) and takes the next ray as soon as CGRT_TRACE_REFILL lanes of its warp are idle.
RT_DEV int fastStepAny(const DevScene& S, FastTrav& T, FastStack& K, bool any, float eps, float maxDist)
{
    if (travIsLeaf(T.node)) return any ? fastStepLeaf<true>(S, T, K, eps, maxDist) : fastStepLeaf<false>(S, T, K, eps, maxDist);
    return any ? fastStepWide<true>(S, T, K, maxDist) : fastStepWide<false>(S, T, K, maxDist);
}

__global__ void __launch_bounds__(128, CGRT_TRACE_MINBLOCKS) k_trace(DevScene S, const float4* __restrict__ raysA, float4* __restrict__ resA,
                                                const int* __restrict__ nAp, int mulA, const float4* __restrict__ raysB,
                                                float4* __restrict__ resB, const int* __restrict__ nBp, int* work, int coopMax)
{
    const int nA = nAp ? *nAp * mulA : 0, nB = nBp ? *nBp : 0; // list A holds mulA (= lights) rays per counted hit
    const int n = nA + nB;
    if (n < coopMax) return; // small round: k_trace8 searches it
    // a block whose first wave would find the list already handed out has nothing to do (small late rounds)
    if ((long long)blockIdx.x * blockDim.x >= (long long)n) return;
    FastTrav T;
    FastStack K;
    int idx = -1;
    int state = TRAV_DONE;
    float eps = 0.0f, maxDist = 0.0f;
    bool exhausted = false;
    const int lane = threadIdx.x & 31;
    const unsigned ltMask = (1u << lane) - 1u;
#ifdef CGRT_INSTRUMENT
    int nSteps = 0;
#define TRACE_DONE_INSTR() do { int b_ = nSteps / 8; if (b_ > 63) b_ = 63; atomicAdd(&g_stepHist[b_], 1u); nSteps = 0; } while (0)
#define TRACE_STEP_INSTR() nSteps++
#else
#define TRACE_DONE_INSTR() do { } while (0)
#define TRACE_STEP_INSTR() do { } while (0)
#endif
    INSTR_ADD(15, 1);
    while (true) {
        const unsigned idle = __ballot_sync(0xffffffffu, idx < 0);
        const int nIdle = __popc(idle);
        if (!exhausted && nIdle >= CGRT_TRACE_REFILL) {
            const int leader = __ffs(idle) - 1;
            int base = 0;
            if (lane == leader) base = atomicAdd(work, nIdle);
            base = __shfl_sync(0xffffffffu, base, leader);
            if (base + nIdle >= n) exhausted = true;
            if (idx < 0) {
                const int mine = base + __popc(idle & ltMask);
                if (mine < n) {
                    idx = mine;
                    const float4* r = mine < nA ? raysA + 3 * (size_t)mine : raysB + 3 * (size_t)(mine - nA);
                    const float4 a = __ldg(r), b = __ldg(r + 1), c = __ldg(r + 2);
                    maxDist = b.w;
                    eps = c.z;
                    K.t2 = __int_as_float(0x7f800000);
                    state = fastBegin(S, T, mk3(a), mk3(b), a.w); // (the always-list is applied by k_finish)
                }
            }
            INSTR_ADD(8, 1); INSTR_ADD(9, nIdle);
        } else if (idle == 0xffffffffu) {
            break; // exhausted and every lane is done
        }
#pragma unroll 1
        for (int it = 0; it < CGRT_TRACE_STEPS; it++) {
            if (idx >= 0 && state != TRAV_CONTINUE) { // finished (possibly right at fastBegin): hand in the result
                float4* out = idx < nA ? resA + idx : resB + (idx - nA);
                *out = make_float4(i2f(state), T.t, i2f(T.hitTri), K.t2);
                idx = -1;
                TRACE_DONE_INSTR();
            }
            const bool run = idx >= 0;
            const bool leaf = run && travIsLeaf(T.node);
            const int sAll = __popc(__ballot_sync(0xffffffffu, run));
            const int sLeaf = __popc(__ballot_sync(0xffffffffu, leaf));
            INSTR_ADD(0, 1); INSTR_ADD(1, sAll);
            if (sAll == 0 || (!exhausted && 32 - sAll >= CGRT_TRACE_REFILL && it > 0)) break;
            const bool any = idx >= 0 && idx < nA;
            if (sAll - sLeaf >= sLeaf) {
                INSTR_ADD(2, 1); INSTR_ADD(5, sAll - sLeaf);
                if (run && !leaf) { state = any ? fastStepWide<true>(S, T, K, maxDist) : fastStepWide<false>(S, T, K, maxDist); TRACE_STEP_INSTR(); }
            } else {
                INSTR_ADD(4, 1); INSTR_ADD(7, sLeaf);
                if (leaf) { state = any ? fastStepLeaf<true>(S, T, K, eps, maxDist) : fastStepLeaf<false>(S, T, K, eps, maxDist); TRACE_STEP_INSTR(); }
            }
        }
        if (idx >= 0 && state != TRAV_CONTINUE) {
            float4* out = idx < nA ? resA + idx : resB + (idx - nA);
            *out = make_float4(i2f(state), T.t, i2f(T.hitTri), K.t2);
            idx = -1;
            TRACE_DONE_INSTR();
        }
    }
}

// ---- the search, cooperative form: EIGHT lanes per ray ----------------------------------------------------------------------
// Profiling k_trace showed that every launch ends with a long tail: the warp that holds the longest rays runs ~140 dependent
// iterations of ~350 instructions each with nothing to hide their latency (1.5 us per iteration, ~200 us per launch, six
// launches per frame). Here a ray belongs to a group of 8 lanes: in an 8-wide node every lane tests ONE child box, in a leaf
// every lane tests ONE triangle, and ballot / redux combine the group's answers. A step is ~60 instructions deep instead of
// ~350, four rays of a warp diverge instead of thirty-two, and the node / triangle fetches of a group are single contiguous
// 256 / 512-byte reads. The traversal stack of a group lives in shared memory. Same search (conservative boxes, the
// reference's triangle arithmetic, smallest acceptable distance, defer on ties / in-plane shortcuts), so k_finish's
// certificate applies unchanged.
#ifndef CGRT_TRACE8
#define CGRT_TRACE8 1
#endif
#ifndef CGRT_TRACE8_MINBLOCKS
#define CGRT_TRACE8_MINBLOCKS 10
#endif
#define CGRT_STACK8 48

__global__ void __launch_bounds__(128, CGRT_TRACE8_MINBLOCKS) k_trace8(DevScene S, const float4* __restrict__ raysA, float4* __restrict__ resA,
                                                  const int* __restrict__ nAp, int mulA, const float4* __restrict__ raysB,
                                                  float4* __restrict__ resB, const int* __restrict__ nBp, int* work, int coopMax)
{
    __shared__ uint2 stk[16][CGRT_STACK8]; // per group: (node id, entry distance bits)
    const int nA = nAp ? *nAp * mulA : 0, nB = nBp ? *nBp : 0;
    const int n = nA + nB;
    if (n >= coopMax) return; // large round: k_trace searches it
    // rays per global fetch of a warp: small rounds are spread over all warps, down to one ray per warp (latency: the four
    // groups of a warp serialise when they sit in different node classes), large ones fetch 16 at a time
    const int totalWarps = gridDim.x * 4;
    int chunk = (n + totalWarps - 1) / totalWarps;
    chunk = chunk < 1 ? 1 : (chunk > 16 ? 16 : chunk);
    if ((long long)blockIdx.x * 4 * chunk >= (long long)n) return;
    const int lane = threadIdx.x & 31, g = lane >> 3, j = lane & 7;
    const unsigned gmask = 0xFFu << (8 * g);
    uint2* K = stk[threadIdx.x >> 3];
    const float slack = 1.000001f;
    // group-uniform ray state (every lane of the group holds the same values)
    V3 o = mk3(0.0f, 0.0f, 0.0f), d = o, inv = o;
    float t = 0.0f, t2 = 0.0f, eps = 0.0f, maxDist = 0.0f;
    int hitTri = -1, idx = -1, state = TRAV_DONE, sp = 0;
    uint32_t node = 0u;
    bool any = false;
    int cur = 0, end = 0; // warp-uniform: the warp's current chunk of the work list
    bool exhausted = false;
    while (true) {
        // ---- finished groups hand in their result, then the warp hands out rays (converged)
        if (idx >= 0 && state != TRAV_CONTINUE) {
            if (j == 0) {
                float4* out = idx < nA ? resA + idx : resB + (idx - nA);
                *out = make_float4(i2f(state), t, i2f(hitTri), t2);
            }
            idx = -1;
        }
        const unsigned needy = __ballot_sync(0xffffffffu, idx < 0 && j == 0);
        if (needy != 0u && !exhausted) {
#pragma unroll
            for (int gg = 0; gg < 4; gg++) {
                if (!((needy >> (8 * gg)) & 1u) || exhausted) continue;
                if (cur == end) {
                    int base = 0;
                    if (lane == 0) base = atomicAdd(work, chunk);
                    base = __shfl_sync(0xffffffffu, base, 0);
                    cur = base;
                    end = base + chunk < n ? base + chunk : n;
                    if (cur >= n) {
                        exhausted = true;
                        continue;
                    }
                }
                const int mine = cur++;
                if (g == gg) {
                    idx = mine;
                    any = mine < nA;
                    const float4* r = any ? raysA + 3 * (size_t)mine : raysB + 3 * (size_t)(mine - nA);
                    const float4 a = __ldg(r), b = __ldg(r + 1), c = __ldg(r + 2);
                    o = mk3(a);
                    d = mk3(b);
                    maxDist = b.w;
                    eps = c.z;
                    FastTrav T0; // (every lane of the group evaluates the same start; the always-list is applied by k_finish)
                    state = fastBegin(S, T0, o, d, a.w);
                    inv = T0.inv;
                    t = T0.t;
                    t2 = __int_as_float(0x7f800000);
                    hitTri = T0.hitTri;
                    sp = 0;
                    node = T0.node;
                }
            }
        }
        if (__ballot_sync(0xffffffffu, idx >= 0) == 0u) {
            if (exhausted) break;
            continue;
        }
        // ---- one step of every active group. The per-lane tests run in divergent code WITHOUT collectives; the group results
        // are then combined with full-warp ballots / shuffles that all 32 lanes execute together (per-group masks would split
        // the warp into four separately scheduled quarters - measured 4x slower).
        const bool active = idx >= 0 && state == TRAV_CONTINUE;
        const bool isLeaf = (node & CGRT_TRI) != 0u;
        const float bound = (any ? fminf(t, maxDist) : t) * slack;
        int pos = -1;                            // leaf: position of this lane's triangle
        float near = __int_as_float(0x7f800000); // leaf: distance of an acceptable triangle that does not beat the best
        bool p = false, amb = false;     // p: this lane's child box is hit / this lane's triangle is an acceptable candidate
        unsigned key = 0xffffffffu;      // ordering key of the lane's result (entry distance | child, or candidate distance)
        uint32_t id = 0u;
        float ti = 0.0f;
        if (active) {
            if (isLeaf) {
                // leaf: lane j tests triangle j with the reference's accept arithmetic (cgrt_device.cuh fastStepLeaf)
                const int first = (int)(node & CGRT_IDX_MASK), count = (int)((node >> CGRT_TRICNT_SHIFT) & 7u) + 1;
                if (j < count) {
                    const float4* tr = S.tri4f + 4 * (size_t)(first + j);
                    const float4 pl = __ldg(tr), v0 = __ldg(tr + 1), v1 = __ldg(tr + 2), v2 = __ldg(tr + 3);
                    pos = f2i(v2.w); // position of the triangle in the reference-ordered arrays
                    const V3 nrm = mk3(pl);
                    const float on = dot3(o, nrm);
                    const bool shortcut = (on == pl.w);
                    bool cand = true;
                    float tt = 0.0f;
                    if (!shortcut) {
                        const float denominator = dot3(d, nrm);
                        if (denominator == 0) cand = false;
                        else {
                            tt = (pl.w - on) / denominator;
                            if (tt < 0) cand = false;
                            else if (hitTri < 0 ? !(tt < t) : !(tt <= t * CGRT_NEAR)) cand = false; // `t >= ray.t` / clearly farther
                        }
                    }
                    if (cand) {
                        const V3 pt = o + d * tt;
                        if (pointInTriangleDev(mk3(v0), mk3(v1), mk3(v2), nrm, pt)) {
                            if (shortcut || (hitTri >= 0 && tt == t)) amb = true; // depends on the reference's visiting order
                            else if (hitTri >= 0 && tt > t) near = tt;            // acceptable runner-up just behind the best
                            else { p = true; key = __float_as_uint(tt + 0.0f); }
                        }
                    }
                }
            } else {
                // 8-wide node: lane j tests child j against its pre-expanded box
                const float4* c = S.wide8 + 16 * (size_t)(node & CGRT_IDX_MASK) + 2 * j;
                const float4 lo = __ldg(c), hi = __ldg(c + 1);
                id = (uint32_t)f2i(lo.w);
                const float q0x = (lo.x - o.x) * inv.x, q1x = (hi.x - o.x) * inv.x;
                const float q0y = (lo.y - o.y) * inv.y, q1y = (hi.y - o.y) * inv.y;
                const float q0z = (lo.z - o.z) * inv.z, q1z = (hi.z - o.z) * inv.z;
                ti = fmaxf(fmaxf(fminf(q0x, q1x), fminf(q0y, q1y)), fminf(q0z, q1z));
                const float to = fminf(fminf(fmaxf(q0x, q1x), fmaxf(q0y, q1y)), fmaxf(q0z, q1z));
                p = id != 0u && !(to < 0.0f || ti > to * slack || ti > bound);
                if (p) key = (__float_as_uint(fmaxf(ti, 0.0f)) & ~7u) | (unsigned)j; // nearest first, ties by child index
            }
        }
        // ---- combine within each group of 8 (full-warp collectives, converged)
        const unsigned pm = (__ballot_sync(0xffffffffu, p) >> (8 * g)) & 0xFFu;
        const unsigned ambm = (__ballot_sync(0xffffffffu, amb) >> (8 * g)) & 0xFFu;
        unsigned mn = key;
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, 1));
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, 2));
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, 4));
        const unsigned winm = (__ballot_sync(0xffffffffu, p && key == mn) >> (8 * g)) & 0xFFu;
        const uint32_t nextId = __shfl_sync(0xffffffffu, id, 8 * g + (int)(mn & 7u));
        const int winPos = __shfl_sync(0xffffffffu, pos, 8 * g + (winm ? __ffs(winm) - 1 : 0)); // leaf: position of the new best
        // leaf: smallest distance among the group's acceptable triangles that are not the new best (runner-up for the certificate)
        float ru = (isLeaf && p && key != mn) ? __uint_as_float(key) : near;
        ru = fminf(ru, __shfl_xor_sync(0xffffffffu, ru, 1));
        ru = fminf(ru, __shfl_xor_sync(0xffffffffu, ru, 2));
        ru = fminf(ru, __shfl_xor_sync(0xffffffffu, ru, 4));
        if (active) {
            bool pop = false;
            if (isLeaf) {
                if (ambm != 0u || __popc(winm) > 1) {
                    state = TRAV_DEFER; // ties at the smallest distance / in-plane shortcut
                } else {
                    t2 = fminf(t2, ru);
                    if (pm != 0u) {
                        if (hitTri >= 0) t2 = fminf(t2, t); // the old best becomes the runner-up
                        t = __uint_as_float(mn);
                        hitTri = winPos;
                    }
                    if (any && pm != 0u && !(t + eps >= maxDist)) state = TRAV_FIRED;
                    else pop = true;
                }
            } else if (pm == 0u) {
                pop = true;
            } else if (sp + 7 > CGRT_STACK8) {
                state = TRAV_DEFER; // pathological depth: the exact traversal handles the ray
            } else {
                // nearest hit child next; the others go on the group's stack with their entry distance
                const int best = (int)(mn & 7u);
                if (p && j != best) {
                    const unsigned before = pm & ((1u << j) - 1u) & ~(1u << best);
                    K[sp + __popc(before)] = make_uint2(id, __float_as_uint(ti));
                }
                sp += __popc(pm) - 1;
                node = nextId;
            }
            if (pop) {
                const float b2 = (any ? fminf(t, maxDist) : t) * slack;
                state = TRAV_DONE;
                while (sp > 0) {
                    sp--;
                    const uint2 e = K[sp];
                    if (__uint_as_float(e.y) > b2) continue;
                    node = e.x;
                    state = TRAV_CONTINUE;
                    break;
                }
            }
        }
        __syncwarp();
    }
}

// ---- after the search: per-ray completion shared by k_finish (round pipeline) and k_wave (persistent wavefront) ----------------
// exact replays (<= 3e-5 of the rays): inline in the flat kernel, out of line in the persistent one (its register budget is
// set by the search loop)
__device__ __noinline__ bool replayAnyNI(const DevScene& S, const V3& o, const V3& d, float tIn, float eps, float maxDist)
{
    TraceResult R;
    return traverseFast<true>(S, o, d, tIn, eps, maxDist, R);
}
__device__ __noinline__ bool replayClosestNI(const DevScene& S, const V3& o, const V3& d, float tIn, TraceResult& R)
{
    return traverseFast<false>(S, o, d, tIn, 0.0f, 0.0f, R);
}

// shadow ray (record a, b, c; search result res = state, t, tri, t2): certificate or exact replay, sphere loop.
// Returns true iff the point is shadowed for this light (pointInShadow, main.cpp:104-135).
template <bool NI>
RT_DEV bool finishShadowRay(const DevScene& S, const float4& a, const float4& b, const float4& c, const float4& res, bool& replayS)
{
    const V3 o = mk3(a), d = mk3(b);
    int state = f2i(res.x), tri = f2i(res.z);
    const float eps = c.z, maxDist = b.w;
    float tBest = res.y;
    bool shadowed = false, settled = false;
    if (state == TRAV_DONE && S.nAlways > 0) { // the triangles outside the tree, if the ray enters the reference tree
        const float4 rq0 = __ldg(S.nodes + 0), rq1 = __ldg(S.nodes + 1);
        float tmp;
        if (startsInBox(o, mk3(rq0), mk3(rq1)) || slabTest(mk3(rq0), mk3(rq1), o, d, a.w, tmp)) {
            FastTrav T;
            float t2s = res.w;
            T.o = o; T.d = d; T.t = tBest; T.hitTri = tri; T.sp = 0; T.node = 0u;
            state = fastAlways<true>(S, T, t2s, eps, maxDist);
            if (state == TRAV_CONTINUE) state = TRAV_DONE;
            tBest = T.t;
            tri = T.hitTri;
        }
    }
    if (state == TRAV_FIRED) {
        if (certifyAny(S, o, d, tri, tBest, eps, maxDist)) { shadowed = true; settled = true; }
    } else if (state == TRAV_DONE) { // the tree does not shadow; spheres may (bvh.cpp:878-879)
        settled = true;
        float t = tBest;
        for (int sp = 0; sp < S.nSpheres; sp++) {
            const float4 sc = __ldg(S.spheres + 3 * sp);
            float ts;
            V3 sn;
            if (sphereTest(mk3(sc), sc.w, o, d, t, ts, sn)) {
                t = ts;
                if (!(ts + eps >= maxDist)) { shadowed = true; break; }
            }
        }
    }
    if (!settled) { // not certifiable: the exact reference-order traversal decides
        if (NI) shadowed = replayAnyNI(S, o, d, a.w, eps, maxDist);
        else {
            TraceResult R;
            shadowed = traverseFast<true>(S, o, d, a.w, eps, maxDist, R);
        }
        replayS = true;
    }
    return shadowed;
}

// closest-hit ray: certificate or exact replay, sphere loop (bvh.cpp:878-879). Returns hit; R = the reference's result.
template <bool NI>
RT_DEV bool finishClosestRay(const DevScene& S, const float4& a, const float4& b, const float4& res, TraceResult& R, bool& replayC)
{
    const V3 o = mk3(a), d = mk3(b);
    int state = f2i(res.x);
    R.sphere = -1;
    R.tri = f2i(res.z);
    R.t = res.y;
    float t2 = res.w;
    if (state == TRAV_DONE && S.nAlways > 0) { // the triangles outside the tree, if the ray enters the reference tree
        const float4 rq0 = __ldg(S.nodes + 0), rq1 = __ldg(S.nodes + 1);
        float tmp;
        if (startsInBox(o, mk3(rq0), mk3(rq1)) || slabTest(mk3(rq0), mk3(rq1), o, d, a.w, tmp)) {
            FastTrav T;
            T.o = o; T.d = d; T.t = R.t; T.hitTri = R.tri; T.sp = 0; T.node = 0u;
            state = fastAlways<false>(S, T, t2, 0.0f, 0.0f);
            if (state == TRAV_CONTINUE) state = TRAV_DONE;
            R.t = T.t;
            R.tri = T.hitTri;
        }
    }
    const bool settled = state == TRAV_DONE && (R.tri < 0 || certifyClosest(S, o, d, R.tri, R.t, t2, a.w));
    if (settled) {
        float t = R.t;
        for (int sp = 0; sp < S.nSpheres; sp++) {
            const float4 sc = __ldg(S.spheres + 3 * sp);
            float ts;
            V3 sn;
            if (sphereTest(mk3(sc), sc.w, o, d, t, ts, sn)) {
                t = ts;
                R.sphere = sp;
                R.sphereN = sn;
            }
        }
        R.t = t;
        return R.tri >= 0 || R.sphere >= 0;
    }
    replayC = true;
    if (NI) return replayClosestNI(S, o, d, a.w, R);
    return traverseFast<false>(S, o, d, a.w, 0.0f, 0.0f, R);
}

// shading normal + material of a hit (intersectRayWithTriangle's epilogue, ray_tracing.cpp:92-107; spheres: bvh.cpp:878-879
// leave the material of the last accepted triangle in place)
RT_DEV void hitNormalAndMaterial(const DevScene& S, const TraceResult& R, const V3& o, const V3& d, V3& nn, int& mat)
{
    if (R.sphere >= 0) {
        nn = R.sphereN;
        mat = R.tri >= 0 ? f2i(__ldg(S.triV1 + R.tri).w) : -1;
    } else {
        const int k = R.tri;
        const float4 v0 = __ldg(S.triV0 + k), v1 = __ldg(S.triV1 + k), v2 = __ldg(S.triV2 + k);
        const float4 n0 = __ldg(S.triN0 + k), n1 = __ldg(S.triN1 + k), n2 = __ldg(S.triN2 + k);
        const float4 pl = __ldg(S.triPl + k);
        float al, be, ga;
        hitEpilogue(mk3(v0), mk3(v1), mk3(v2), mk3(n0), mk3(n1), mk3(n2), mk3(pl), o, d, R.t, al, be, ga, nn);
        mat = f2i(v1.w);
    }
}

// the shadow ray of a hit towards light l (pointInShadow, src/main.cpp:104-135) and its reflection ray (ComputeReflectedRay,
// main.cpp:252-256: t = |incoming direction|, origin offset along the reflection)
RT_DEV void shadowRayOf(const float4* __restrict__ lights, int l, const V3& pointOn, V3& org, V3& dir, float& dist)
{
    const V3 lightPos = mk3(__ldg(lights + 2 * l));
    const V3 fromPosToLight = lightPos - pointOn;
    dir = normalize3(fromPosToLight);
    org = pointOn + 0.001f * dir;
    dist = length3(fromPosToLight);
}
RT_DEV void reflectionRayOf(const V3& pointOn, const V3& rd, const V3& nn, V3& org, V3& dir, float& tIn)
{
    dir = normalize3(reflect3(rd, nn));
    org = pointOn + 0.001f * dir;
    tIn = length3(rd);
}

// ---- after the search: one thread per ray ------------------------------------------------------------------------------------
// Shadow rays (list A, produced by the hits of level `level - 1`): certificate or exact replay, sphere loop, lit flag.
// Closest-hit rays (list B, level `level`): certificate or exact replay, sphere loop, hit epilogue, hit record; emits the
// shadow rays of the hit (pointInShadow, main.cpp:104-135) and its reflection ray (shade(), main.cpp:246-256).
__global__ void __launch_bounds__(128) k_finish(DevScene S, const FrameParams* __restrict__ Pp, const float4* __restrict__ lights,
                                                RoundBuffers B, int level, const float4* __restrict__ raysA,
                                                const float4* __restrict__ resA, const int* __restrict__ nAp,
                                                const float4* __restrict__ raysB, const float4* __restrict__ resB,
                                                const int* __restrict__ nBp, float4* __restrict__ nextC, float4* __restrict__ nextS,
                                                float* __restrict__ fb, const int2* __restrict__ tileSeq)
{
    const FrameParams P = *Pp;
    const int nL = P.nLights;
    const int nA = nAp ? *nAp * nL : 0, nB = nBp ? *nBp : 0;
    const int n = nA + nB;
    for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const int i = base + threadIdx.x;
        bool hit = false, bounce = false, replayC = false, replayS = false;
        V3 pointOn = mk3(0.0f, 0.0f, 0.0f), nn = pointOn, rd = pointOn;
        int slot = 0, rec = 0;
        if (i < nA) { // ---- shadow ray
            const float4* r = raysA + 3 * (size_t)i;
            const float4 a = r[0], b = r[1], c = r[2], res = resA[i];
            const bool shadowed = finishShadowRay<false>(S, a, b, c, res, replayS);
            B.lit[f2i(c.y) & 0x3fffffff] = shadowed ? 0 : 1;
        } else if (i < n) { // ---- closest-hit ray of `level`
            const float4* r = raysB + 3 * (size_t)(i - nA);
            const float4 a = r[0], b = r[1], c = r[2], res = resB[i - nA];
            const V3 o = mk3(a), d = mk3(b);
            slot = f2i(c.x);
            TraceResult R;
            hit = finishClosestRay<false>(S, a, b, res, R, replayC);
            if (!hit) {
                if (level == 0) { // trace(): miss -> black, src/main.cpp:288-294
                    int x, y, outIdx, local;
                    if (seqToPixel(P, tileSeq, slot, x, y, outIdx, local)) storeRGB(fb, outIdx, mk3(0.0f, 0.0f, 0.0f));
                }
            } else {
                int mat;
                hitNormalAndMaterial(S, R, o, d, nn, mat);
                pointOn = o + d * R.t; // main.cpp:164
                rd = d;
                rec = slot * B.levels + level;
                float4* h = B.hitRec + 3 * (size_t)rec;
                h[0] = make_float4(pointOn.x, pointOn.y, pointOn.z, i2f(mat));
                h[1] = make_float4(nn.x, nn.y, nn.z, 0.0f);
                h[2] = make_float4(d.x, d.y, d.z, 0.0f);
                B.pathDepth[slot] = level + 1;
                const float ksz = mat >= 0 ? __ldg(S.mats + 2 * mat + 1).z : 0.0f;
                bounce = !(ksz <= 0.01f) && level + 1 < P.traceLimit; // shade(): mirror test main.cpp:246, trace limit :267
            }
        }
        // ---- emission (warp-aggregated, slots stay in screen order within the warp)
        if (level == 0) warpPush(B.counts + CGRT_CNT_PATHS, hit);
        const int sBase = warpPush(B.counts + CGRT_CNT_HIT + level, hit && nL > 0);
        const int cPos = warpPush(B.counts + CGRT_CNT_BOUNCE + level + 1, bounce);
        const unsigned rc = __ballot_sync(0xffffffffu, replayC), rs = __ballot_sync(0xffffffffu, replayS);
        if ((threadIdx.x & 31) == 0) {
            if (rc) atomicAdd(B.counts + CGRT_CNT_REPLAY_PATHS, __popc(rc));
            if (rs) atomicAdd(B.counts + CGRT_CNT_REPLAY_SHADOW, __popc(rs));
        }
        if (hit && nL > 0) {
            for (int l = 0; l < nL; l++) {
                V3 org, dir;
                float dist;
                shadowRayOf(lights, l, pointOn, org, dir, dist);
                writeRay(nextS + 3 * ((size_t)sBase * nL + l), org, FLT_MAX, dir, dist, slot, CGRT_RAY_ANY | (rec * nL + l), 0.001f);
            }
        }
        if (bounce) {
            V3 org, dir;
            float tIn;
            reflectionRayOf(pointOn, rd, nn, org, dir, tIn);
            writeRay(nextC + 3 * (size_t)cPos, org, tIn, dir, __int_as_float(0x7f800000), slot, level + 1, 0.0f);
        }
    }
}

// ---- batch queries (cgrt_intersect_closest / _any) through the same split: search-only persistent kernel, flat finish ------------
// The one-kernel form (k_closest_batch / k_any_batch: a thread follows its ray through search, certificate and replay) keeps
// the certificate's twelve exact slab tests and the fp64 epilogue inside the divergent per-ray loop; on 16 M incoherent rays
// of the 1 M-triangle soup it ran at 152 / 196 Mrays/s and slower than the exact traversal (profiles/r01_configs.md). Here the
// rays are turned into the round pipeline's records, k_trace searches them, and a flat kernel certifies / replays and writes
// the hit records.
__global__ void __launch_bounds__(256) k_batch_prep(const float4* __restrict__ rays, const float* __restrict__ maxDist, float eps,
                                                    int n, int any, float4* __restrict__ rec, int* __restrict__ ctl)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 r0 = __ldg(rays + 2 * (size_t)i), r1 = __ldg(rays + 2 * (size_t)i + 1);
        rec[3 * (size_t)i] = r0;
        rec[3 * (size_t)i + 1] = make_float4(r1.x, r1.y, r1.z, any ? __ldg(maxDist + i) : __int_as_float(0x7f800000));
        rec[3 * (size_t)i + 2] = make_float4(i2f(i), i2f(any ? CGRT_RAY_ANY : 0), eps, 0.0f);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        ctl[0] = n; // list length read by k_trace
        ctl[1] = 0; // its work counter
    }
}
__global__ void __launch_bounds__(128) k_batch_finish_closest(DevScene S, const float4* __restrict__ rec, const float4* __restrict__ res,
                                                              int n, float4* __restrict__ hits)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 a = rec[3 * (size_t)i], b = rec[3 * (size_t)i + 1];
        TraceResult R;
        bool replay = false;
        const bool hit = finishClosestRay<false>(S, a, b, res[i], R, replay);
        writeHit(S, mk3(a), mk3(b), a.w, hit, R, hits + 2 * (size_t)i);
    }
}
__global__ void __launch_bounds__(128) k_batch_finish_any(DevScene S, const float4* __restrict__ rec, const float4* __restrict__ res,
                                                          int n, uint8_t* __restrict__ occluded)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        bool replay = false;
        occluded[i] = finishShadowRay<false>(S, rec[3 * (size_t)i], rec[3 * (size_t)i + 1], rec[3 * (size_t)i + 2], res[i], replay) ? 1 : 0;
    }
}

// one thread per pixel slot: direct colour of every level, then the recursion unwound innermost first (main.cpp:241-264)
__global__ void __launch_bounds__(128) k_shade_slots(DevScene S, const FrameParams* __restrict__ Pp, const float4* __restrict__ lights,
                                                     RoundBuffers B, const int2* __restrict__ tileSeq, float* __restrict__ fb)
{
    const FrameParams P = *Pp;
    const int nL = P.nLights;
    for (int base = blockIdx.x * blockDim.x; base < P.nSlots; base += gridDim.x * blockDim.x) {
        const int slot = base + threadIdx.x;
        const int depth = slot < P.nSlots ? B.pathDepth[slot] : 0;
        bool wrote = false;
        int x = 0, y = 0;
        if (depth > 0) { // (else the pixel is already final: black)
            V3 direct[CGRT_MAX_LEVELS], ksv[CGRT_MAX_LEVELS];
            for (int k = 0; k < depth; k++) {
                const int rec = slot * B.levels + k;
                const float4* r = B.hitRec + 3 * (size_t)rec;
                direct[k] = directColour(S, lights, nL, r[0], r[1], r[2], B.lit + (size_t)rec * nL, ksv[k], P.nSph,
                                         P.nSph ? B.soft + (size_t)rec * P.nSph : nullptr);
            }
            int k = depth - 1;
            V3 colour = (ksv[k].z <= 0.01f) ? direct[k] : direct[k] + mk3(0.0f, 0.0f, 0.0f) * ksv[k];
            for (k = depth - 2; k >= 0; k--) colour = direct[k] + colour * ksv[k];
            int outIdx, local;
            wrote = seqToPixel(P, tileSeq, slot, x, y, outIdx, local);
            if (wrote) storeRGB(fb, outIdx, colour);
        }
        noteColoured(B.counts + CGRT_CNT_BBOX, wrote, x, P.height - 1 - y, P.width, P.height);
    }
}

// ---- spherical-light soft shadows (src/main.cpp:168-218): 200 sample rays per hit and spherical light -------------------------
// The reference draws the sample points with std::random_device (non-deterministic); here a counter-based generator keyed by
// (hit record, light, sample, frame seed): three N(0,1) values by Box-Muller from hashed uniforms, normalised (randomUnitVector,
// :46-59) - the same distribution, reproducible frames. Each sample is a bounded any-hit query: ray.t = distance to the sample
// point, lit iff intersect() finds nothing closer (:181-199; the reference's `newRay.t > lightT` branch cannot fire).
// k_soft_list compacts the frame's hit records; k_soft_shadows: one 256-thread block per (hit record, light), one thread per sample.
__global__ void k_soft_list(const FrameParams* __restrict__ Pp, RoundBuffers B, int cap)
{
    const int n = Pp->nSlots;
    for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const int slot = base + threadIdx.x;
        const int depth = slot < n ? B.pathDepth[slot] : 0;
        for (int k = 0; k < B.levels; k++) {
            const int q = warpPush(B.softList + cap, k < depth);
            if (k < depth) B.softList[q] = slot * B.levels + k;
        }
    }
}
RT_DEV unsigned hash32(unsigned x)
{
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
RT_DEV float uniform01(unsigned h) { return ((h >> 8) + 0.5f) * (1.0f / 16777216.0f); } // (0, 1)
__global__ void __launch_bounds__(256) k_soft_shadows(DevScene S, const FrameParams* __restrict__ Pp, const float4* __restrict__ lights,
                                                      RoundBuffers B, int cap)
{
    __shared__ int litCount;
    const FrameParams& P = *Pp;
    const int nSph = P.nSph, nL = P.nLights;
    const int nHits = B.softList[cap];
    for (int item = blockIdx.x; item < nHits * nSph; item += gridDim.x) {
        const int rec = B.softList[item / nSph], l = item % nSph;
        if (threadIdx.x == 0) litCount = 0;
        __syncthreads();
        if (threadIdx.x < 200) {
            const float4 hp = B.hitRec[3 * (size_t)rec];
            const V3 pointOn = mk3(hp);
            const float4 lp = __ldg(lights + 2 * (nL + l));
            // samples are keyed by the record's index in a frame of its view alone, so that a view of several renders the
            // samples of its single frame
            const int slot = rec / B.levels;
            int v, q, single;
            decodeSlot(P, slot, v, q, single);
            const int key1 = single * B.levels + (rec - slot * B.levels);
            // randomUnitVector: y, x, s ~ N(0,1)
            const unsigned key = hash32((unsigned)key1 * 0x9e3779b9u + (unsigned)l * 0x85ebca6bu + threadIdx.x * 0xc2b2ae35u + B.softSeed);
            const float u1 = uniform01(hash32(key ^ 0x68bc21ebu)), u2 = uniform01(hash32(key ^ 0x02e5be93u));
            const float u3 = uniform01(hash32(key ^ 0x967a889bu)), u4 = uniform01(hash32(key ^ 0x368cc8b7u));
            const float r1 = sqrtf(-2.0f * logf(u1)), r2 = sqrtf(-2.0f * logf(u3));
            const V3 g = mk3(r1 * cosf(6.2831853f * u2), r1 * sinf(6.2831853f * u2), r2 * cosf(6.2831853f * u4));
            const V3 randomPointOnSphere = mk3(lp) + lp.w * normalize3(g);
            const V3 dir = normalize3(randomPointOnSphere - pointOn);
            const V3 org = pointOn + 0.001f * dir;
            const float lightT = length3(org - randomPointOnSphere);
            TraceResult R;
            // intersect(newRay) with ray.t = lightT: true iff an acceptable triangle (or a sphere) lies closer
            const bool blocked = traverseSpec<true>(S, org, dir, lightT, 0.0f, __int_as_float(0x7f800000), R);
            if (!blocked) atomicAdd(&litCount, 1);
        }
        __syncthreads();
        if (threadIdx.x == 0) B.soft[(size_t)rec * nSph + l] = (float)litCount / 200.0f;
        __syncthreads();
    }
}

#include "cgrt_wave.cuh"

// ---- counting wavefront: shading + bounce emission, one thread per hit.  shading/shade, src/main.cpp:61-98, 220-264 ---------
__global__ void __launch_bounds__(128) k_shade(DevScene S, const FrameParams* __restrict__ Pp,
                                               const float4* __restrict__ lights, CountBuffers B, int level,
                                               float* __restrict__ fb)
{
    const int nL = Pp->nLights;
    const int traceLimit = Pp->traceLimit;
    const int n = B.counts[CGRT_CNT_HIT + level];
    for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const int h = base + threadIdx.x;
        const bool valid = h < n;
        bool bounce = false;
        V3 P = mk3(0.0f, 0.0f, 0.0f), N = P, D = P, result = P, ks = P;
        int outIdx = 0, pathId = -1;
        if (valid) {
            const float4 a = B.hitQ[3 * (size_t)h], b = B.hitQ[3 * (size_t)h + 1], c = B.hitQ[3 * (size_t)h + 2];
            P = mk3(a); N = mk3(b); D = mk3(c);
            const int mat = f2i(a.w);
            outIdx = f2i(b.w);
            pathId = f2i(c.w);
            // default-constructed HitInfo material when only a sphere was hit: kd unspecified in the reference (we use 0),
            // ks 0, shininess 1 (src/mesh.h:17-23)
            float4 m0 = make_float4(0.0f, 0.0f, 0.0f, 1.0f), m1 = make_float4(0.0f, 0.0f, 0.0f, 1.0f);
            if (mat >= 0) { m0 = __ldg(S.mats + 2 * mat); m1 = __ldg(S.mats + 2 * mat + 1); }
            const V3 kd = mk3(m0);
            ks = mk3(m1);
            const float shininess = m0.w;
            for (int l = 0; l < nL; l++) { // point-light loop, src/main.cpp:220-232
                const V3 lightPos = mk3(__ldg(lights + 2 * l)), lightCol = mk3(__ldg(lights + 2 * l + 1));
                const V3 fromPosToLight = normalize3(lightPos - P);
                if (!B.lit[(size_t)h * nL + l]) continue;
                V3 diffuse = mk3(0.0f, 0.0f, 0.0f), specular = diffuse;
                const float diffuseCos = dot3(fromPosToLight, N); // diffuseOneLight, src/main.cpp:84-98
                if (!(diffuseCos <= 0)) diffuse = (lightCol * kd) * diffuseCos;
                const V3 reflected = normalize3(reflect3(D, N)); // specularOneLight, src/main.cpp:61-82
                const float specularCos = dot3(reflected, fromPosToLight);
                if (!(specularCos <= 0)) {
                    // pow(float,float): evaluated in double and narrowed, which reproduces a correctly rounded powf
                    const float pw = (float)pow((double)specularCos, (double)shininess);
                    specular = (lightCol * ks) * pw;
                }
                result = result + diffuse;
                result = result + specular;
            }
            V3 colour;
            bool terminal = true;
            if (ks.z <= 0.01f) { // comma operator: only ks.z decides, src/main.cpp:246
                colour = result;
            } else if (level + 1 >= traceLimit) { // trace(level+1) returns black without a ray, src/main.cpp:267-272
                colour = result + mk3(0.0f, 0.0f, 0.0f) * ks;
            } else {
                terminal = false;
                bounce = true;
            }
            if (terminal) storeRGB(fb, outIdx, foldPath(B.pathState, B.cap, level, pathId, colour));
        }
        const int slot = warpPush(B.counts + CGRT_CNT_BOUNCE + level + 1, bounce);
        if (bounce) {
            // ComputeReflectedRay, src/main.cpp:252-256: t = |incoming direction|, origin offset by 0.001 along the reflection
            const V3 reflected = normalize3(reflect3(D, N));
            const float tmax = length3(D);
            const float epsilon = 0.001f;
            const V3 org = P + epsilon * reflected;
            if (level == 0) {
                pathId = slot; // a path is born at its first bounce; its id indexes pathState / pathPix
                B.pathPix[pathId] = outIdx;
            }
            B.bounceQ[2 * (size_t)slot] = make_float4(org.x, org.y, org.z, tmax);
            B.bounceQ[2 * (size_t)slot + 1] = make_float4(reflected.x, reflected.y, reflected.z, i2f(pathId));
            float4* st = B.pathState + ((size_t)level * B.cap + pathId) * 2;
            st[0] = make_float4(result.x, result.y, result.z, 0.0f);
            st[1] = make_float4(ks.x, ks.y, ks.z, 0.0f);
        }
    }
}

// ---- primary rays only (cgrt_generate_rays) --------------------------------------------------------------------------------
__global__ void k_generate_rays(const FrameParams* __restrict__ Pp, float4* __restrict__ rays)
{
    const FrameParams P = *Pp;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.width * P.height) return;
    const int y = i / P.width, x = i - y * P.width;
    const V3 d = primaryDirection(P, x, y);
    rays[2 * (size_t)i] = make_float4(P.camX, P.camY, P.camZ, FLT_MAX);
    rays[2 * (size_t)i + 1] = make_float4(d.x, d.y, d.z, 0.0f);
}

// ---- synchronous host render, overlapped delivery: the bounding box of the pixels the shading pass coloured (counts[CGRT_CNT_BBOX],
// kept by the shading pass), copied from the device frame straight into the caller's page-locked frame in full 128-byte runs;
// every other pixel of that frame was blanked by a copy-engine transfer while the frame rendered
__global__ void __launch_bounds__(256) k_deliver_box(const int* __restrict__ bbox, int W, int H, const float* __restrict__ frame,
                                                     float* __restrict__ hostFrame)
{
    const int x1 = bbox[0] - 1, r1 = bbox[1] - 1, x0 = W - bbox[2], r0 = H - bbox[3];
    if (bbox[0] <= 0 || x1 < x0 || r1 < r0) return; // nothing was coloured
    const int f0 = (3 * x0) & ~31, f1 = 3 * x1 + 3; // floats of a row, start rounded down to a 128-byte run
    const int perRow = f1 - f0;
    const long long total = (long long)perRow * (r1 - r0 + 1);
    // (the destination is blank already: a warp whose 32 floats are all +0.0 has nothing to send over PCIe - inside the box
    // most of a frame still is background)
    for (long long base = (blockIdx.x * (long long)blockDim.x + threadIdx.x) & ~31ll; base < total; base += (long long)gridDim.x * blockDim.x) {
        const long long i = base + (threadIdx.x & 31);
        const bool in = i < total;
        size_t o = 0;
        float v = 0.0f;
        if (in) {
            const int row = r0 + (int)(i / perRow), f = f0 + (int)(i % perRow);
            o = (size_t)row * W * 3 + f;
            v = frame[o];
        }
        if (__ballot_sync(0xffffffffu, in && __float_as_uint(v) != 0u) != 0u && in) hostFrame[o] = v;
    }
}
void launchDeliverBox(const int* bbox, int W, int H, const float* frame, float* hostFrame, int numSMs, cudaStream_t st)
{
    k_deliver_box<<<numSMs * 8, 256, 0, st>>>(bbox, W, H, frame, hostFrame);
}

// ---- rank 0: de-interleave gathered tile buffers into the Screen layout -----------------------------------------------------
__global__ void k_assemble(const float* __restrict__ gathered, size_t perRankFloats, const int* __restrict__ tileLists,
                           const int* __restrict__ tileCounts, int maxTiles, int world, int tileW, int tileH, int tilesX,
                           int width, int height, float* __restrict__ frame)
{
    const int tpx = tileW * tileH;
    const size_t total = (size_t)world * maxTiles * tpx;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / ((size_t)maxTiles * tpx));
        const int rem = (int)(i - (size_t)r * maxTiles * tpx);
        const int lt = rem / tpx, q = rem - lt * tpx;
        if (lt >= tileCounts[r]) continue;
        const int g = tileLists[(size_t)r * maxTiles + lt];
        const int ty = g / tilesX, tx = g - ty * tilesX;
        const int x = tx * tileW + q % tileW, y = ty * tileH + q / tileW;
        if (x >= width || y >= height) continue;
        const float* src = gathered + (size_t)r * perRankFloats + 3 * (size_t)rem;
        float* dst = frame + 3 * ((size_t)(height - 1 - y) * width + x);
        dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2];
    }
}

// Screen::writeBitmapToFile quantisation, src/screen.cpp:38-49: clamp(c,0,1) = min(max(c,0),1), *255.0f, truncate
__global__ void k_quantize(const float* __restrict__ frame, size_t nPixels, uint8_t* __restrict__ rgba)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nPixels) return;
    uchar4 o;
    float c[3];
    for (int k = 0; k < 3; k++) {
        float v = frame[3 * i + k];
        v = v < 0.0f ? 0.0f : v; // glm::max(x, 0): (x < 0) ? 0 : x
        v = 1.0f < v ? 1.0f : v; // glm::min(x, 1): (1 < x) ? 1 : x
        c[k] = v * 255.0f;
    }
    o.x = (unsigned char)c[0]; o.y = (unsigned char)c[1]; o.z = (unsigned char)c[2]; o.w = 255;
    reinterpret_cast<uchar4*>(rgba)[i] = o;
}

// =================================================================================================================
// Post passes of renderRayTracing (src/main.cpp:663-687 anti-aliasing, :318-584 motion blur): image kernels around the renderer
// =================================================================================================================
// Anti-aliasing (main.cpp:663-687): four rays per pixel at NDC (float(2x+i)/W * (2/level) - 1, float(2y+j)/H * (2/level) - 1),
// level = 2, i.e. exactly the pixel-corner rays of a (2W x 2H) frame (float(k)/(2W)*2 == float(k)/W*1 bit for bit), summed in
// the order (j outer, i inner) into `color` and divided by level * 2.5 = 5 (sic). `color` is never initialised in the reference;
// this implementation starts it at zero (documented assumption).
__global__ void k_aa_downsample(const float* __restrict__ big, int W, int H, float* __restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W * H) return;
    const int row = i / W, x = i - row * W; // Screen layout: row = H-1-y
    const int y = H - 1 - row;
    const int W2 = 2 * W, H2 = 2 * H;
    float c[3] = {0.0f, 0.0f, 0.0f};
    for (int j = 0; j < 2; j++)
        for (int k = 0; k < 2; k++) {
            const int xc = 2 * x + k, yc = 2 * y + j;
            const float* src = big + 3 * ((size_t)(H2 - 1 - yc) * W2 + xc);
            c[0] = c[0] + src[0]; c[1] = c[1] + src[1]; c[2] = c[2] + src[2];
        }
    const float level = 2.0f;
    const float div = level * 2.5f;
    out[3 * (size_t)i + 0] = c[0] / div;
    out[3 * (size_t)i + 1] = c[1] / div;
    out[3 * (size_t)i + 2] = c[2] / div;
}

// Motion blur (blurEffect, main.cpp:318-584): matrixPixels += frame for the 15 shifted look-at points, then / 16
__global__ void k_accumulate(float* __restrict__ acc, const float* __restrict__ frame, size_t n, int first)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    acc[i] = first ? (0.0f + frame[i]) : (acc[i] + frame[i]);
}
__global__ void k_divide(const float* __restrict__ acc, size_t n, float div, float* __restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = acc[i] / div;
}

// ---- bloom (bloomEffect, src/main.cpp:586-628; bookkeeping :698-705) --------------------------------------------------------------
// The reference keeps the pixels whose colour sums to more than 1 (matrixColorsScreen, else black) and then replaces every entry,
// IN PLACE and in scan order (y outer, x inner, y = 0 at the bottom), by the average of its 21 x 21 neighbourhood (clipped at the
// borders; the entry itself first, then rows i = -10..10, columns j = -10..10 in that order) - so an entry sees the NEW values of
// the rows below it in the image (y + i < y) and of its left neighbours, and the OLD values of everything else. The pixel becomes
// that average plus the ray-traced colour.
// That is a recurrence, but one with a wavefront: entry (x, y) needs row y - 1 finished up to column x + 10 only. One warp per
// row, rows chasing each other 11 columns apart (~W / 11 rows in flight), each warp keeping its 21 x 21 window in shared memory
// (one new column per step) and adding the up to 440 terms of an entry in the reference's order - the additions of one entry
// are a dependent chain by definition (float addition is not associative), the three channels are three lanes.
// k_bloom_init: M[y * W + x] = thresholded colour in the reference's index order (ray space: image row H - 1 - y), progress = 0.
__global__ void k_bloom_init(const float* __restrict__ frame, int W, int H, float* __restrict__ M, int* __restrict__ progress)
{
    const size_t n = (size_t)W * H;
    for (size_t p = blockIdx.x * (size_t)blockDim.x + threadIdx.x; p < n; p += (size_t)gridDim.x * blockDim.x) {
        const int y = (int)(p / W), x = (int)(p - (size_t)y * W);
        const float* c = frame + 3 * ((size_t)(H - 1 - y) * W + x);
        const bool keep = c[0] + c[1] + c[2] > 1; // color.x + color.y + color.z > 1, main.cpp:700
        M[3 * p + 0] = keep ? c[0] : 0.0f;
        M[3 * p + 1] = keep ? c[1] : 0.0f;
        M[3 * p + 2] = keep ? c[2] : 0.0f;
        if (x == 0) progress[y] = 0;
    }
}
#define BLOOM_R 10
#define BLOOM_D (2 * BLOOM_R + 1)
__global__ void __launch_bounds__(128) k_bloom(float* M, const float* __restrict__ frame, int W, int H, float* __restrict__ out,
                                               int* progress)
{
    __shared__ float win[4][3][BLOOM_D][BLOOM_D]; // [warp][channel][window row i + 10][column mod 21]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int y = blockIdx.x * 4 + warp;
    if (y >= H) return;
    float(*w)[BLOOM_D][BLOOM_D] = win[warp];
    const int i0 = y - BLOOM_R < 0 ? -y : -BLOOM_R, i1 = y + BLOOM_R > H - 1 ? H - 1 - y : BLOOM_R; // valid rows of the window
    int seen = y == 0 ? W : 0; // columns of row y - 1 known to be finished
    // lane r < 21 loads window row r - 10 of one column (three channels), through L2: other warps write M while this one reads
    auto loadColumn = [&](int xx) {
        const int i = lane - BLOOM_R;
        if (lane < BLOOM_D && i >= i0 && i <= i1) {
            const float* src = M + 3 * ((size_t)(y + i) * W + xx);
            w[0][lane][xx % BLOOM_D] = __ldcg(src);
            w[1][lane][xx % BLOOM_D] = __ldcg(src + 1);
            w[2][lane][xx % BLOOM_D] = __ldcg(src + 2);
        }
    };
    auto waitFor = [&](int need) { // row y - 1 finished up to column `need` (exclusive)
        if (seen >= need) return;
        int v = seen;
        if (lane == 0) {
            while ((v = *(volatile int*)(progress + y - 1)) < need) __nanosleep(64);
        }
        seen = __shfl_sync(0xffffffffu, v, 0);
        __threadfence(); // (the loads of row y - 1's entries come after the progress value that announced them)
    };
    waitFor(BLOOM_R < W ? BLOOM_R : W);
    for (int xx = 0; xx < BLOOM_R && xx < W; xx++) loadColumn(xx);
    for (int x = 0; x < W; x++) {
        if (x + BLOOM_R < W) {
            waitFor(x + BLOOM_R + 1);
            loadColumn(x + BLOOM_R);
        }
        __syncwarp();
        if (lane < 3) {
            const int j0 = x - BLOOM_R < 0 ? -x : -BLOOM_R, j1 = x + BLOOM_R > W - 1 ? W - 1 - x : BLOOM_R;
            float acc = w[lane][BLOOM_R][x % BLOOM_D];
            const int s0 = (x + j0) % BLOOM_D;
            for (int i = i0; i <= i1; i++) {
                const float* row = w[lane][i + BLOOM_R];
                int s = s0;
                for (int j = j0; j <= j1; j++) {
                    if (i != 0 || j != 0) acc += row[s];
                    s = s + 1 == BLOOM_D ? 0 : s + 1;
                }
            }
            const int counter = (i1 - i0 + 1) * (j1 - j0 + 1); // 1 + the number of terms added
            const float m = acc / counter;
            w[lane][BLOOM_R][x % BLOOM_D] = m; // the entries to the right see the new value
            M[3 * ((size_t)y * W + x) + lane] = m;
            const size_t o = 3 * ((size_t)(H - 1 - y) * W + x) + lane;
            out[o] = m + frame[o]; // screen.setPixel(x, y, matrixColorsScreen + color), main.cpp:621
        }
        if ((x & 7) == 7 || x == W - 1) { // announce progress every 8 columns: the writes above first, then the counter
            __threadfence();
            __syncwarp();
            if (lane == 0) *(volatile int*)(progress + y) = x + 1;
        }
        __syncwarp();
    }
}
void launchBloom(const float* frame, int W, int H, float* M, int* progress, float* out, int numSMs, cudaStream_t st)
{
    const size_t n = (size_t)W * H;
    int blocks = (int)((n + 255) / 256);
    blocks = blocks > numSMs * 16 ? numSMs * 16 : blocks;
    k_bloom_init<<<blocks, 256, 0, st>>>(frame, W, H, M, progress);
    k_bloom<<<(H + 3) / 4, 128, 0, st>>>(M, frame, W, H, out, progress);
}

void launchAADownsample(const float* big, int W, int H, float* out, cudaStream_t st)
{
    k_aa_downsample<<<(W * H + 255) / 256, 256, 0, st>>>(big, W, H, out);
}
void launchAccumulate(float* acc, const float* frame, size_t n, bool first, cudaStream_t st)
{
    if (n) k_accumulate<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(acc, frame, n, first ? 1 : 0);
}
void launchDivide(const float* acc, size_t n, float div, float* out, cudaStream_t st)
{
    if (n) k_divide<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(acc, n, div, out);
}

// =================================================================================================================
// Launch wrappers
// =================================================================================================================
static inline int gridFor(size_t n, int block, int maxBlocks)
{
    size_t g = (n + block - 1) / block;
    if (g < 1) g = 1;
    if (g > (size_t)maxBlocks) g = maxBlocks;
    return (int)g;
}

void launchPermuteTri4(const float4* tri4, const int* fastOrder, float4* tri4f, int n, cudaStream_t st)
{
    if (n > 0) k_permute_tri4<<<(n + 255) / 256, 256, 0, st>>>(tri4, fastOrder, tri4f, n);
}

void launchSetupPlanes(const float4* v0, const float4* v1, const float4* v2, float4* pl, float4* tri4, int n, cudaStream_t st)
{
    if (n > 0) k_setup_planes<<<(n + 255) / 256, 256, 0, st>>>(v0, v1, v2, pl, tri4, n);
}

#define CGRT_BATCH_CHUNK (4 << 20) // rays per pass of the split batch path: 256 MB of stream-ordered scratch
#define CGRT_BATCH_SPLIT_MIN 8192  // smaller batches (the scalar intersect(Ray&, HitInfo&) is a batch of one) take the one-kernel form
// the split path for one kind of query; returns false when the stream-ordered scratch is not available (the caller falls back)
static bool launchSplitBatch(const DevScene& S, const float4* rays, const float* maxDist, float eps, size_t n, bool any,
                             float4* hits, uint8_t* occluded, int numSMs, cudaStream_t st)
{
    const size_t chunk = n < CGRT_BATCH_CHUNK ? n : (size_t)CGRT_BATCH_CHUNK;
    { // keep the stream-ordered pool's memory between calls (by default it goes back to the driver at every synchronisation,
      // and the next call pays for mapping 256 MB again)
        static bool kept[64] = {false};
        int dev = 0;
        cudaGetDevice(&dev);
        if (!kept[dev & 63]) {
            cudaMemPool_t pool;
            if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
                unsigned long long keep = ~0ull;
                cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
            }
            cudaGetLastError();
            kept[dev & 63] = true;
        }
    }
    float4* rec = nullptr;
    float4* res = nullptr;
    int* ctl = nullptr;
    if (cudaMallocAsync((void**)&rec, chunk * 3 * sizeof(float4), st) != cudaSuccess ||
        cudaMallocAsync((void**)&res, chunk * sizeof(float4), st) != cudaSuccess ||
        cudaMallocAsync((void**)&ctl, 2 * sizeof(int), st) != cudaSuccess) {
        cudaGetLastError();
        if (rec) cudaFreeAsync(rec, st);
        if (res) cudaFreeAsync(res, st);
        return false;
    }
    const int persistent = numSMs * tuning().blocks;
    for (size_t done = 0; done < n; done += chunk) {
        const int m = (int)(n - done < chunk ? n - done : chunk);
        const int flat = gridFor((size_t)m, 128, numSMs * 16);
        k_batch_prep<<<gridFor((size_t)m, 256, numSMs * 8), 256, 0, st>>>(rays + 2 * done, any ? maxDist + done : nullptr, eps, m, any ? 1 : 0, rec, ctl);
        if (any) {
            k_trace<<<persistent, 128, 0, st>>>(S, rec, res, ctl, 1, nullptr, nullptr, nullptr, ctl + 1, 0);
            k_batch_finish_any<<<flat, 128, 0, st>>>(S, rec, res, m, occluded + done);
        } else {
            k_trace<<<persistent, 128, 0, st>>>(S, nullptr, nullptr, nullptr, 1, rec, res, ctl, ctl + 1, 0);
            k_batch_finish_closest<<<flat, 128, 0, st>>>(S, rec, res, m, hits + 2 * done);
        }
    }
    cudaFreeAsync(rec, st);
    cudaFreeAsync(res, st);
    cudaFreeAsync(ctl, st);
    return true;
}

void launchClosestBatch(const DevScene& S, const float4* rays, size_t n, float4* hits, uint32_t* counts, int numSMs,
                        cudaStream_t st)
{
    if (n == 0) return;
    if (!counts && S.fastRoot != 0u && n >= CGRT_BATCH_SPLIT_MIN && !getenv("CGRT_BATCH_ONE_KERNEL") &&
        launchSplitBatch(S, rays, nullptr, 0.0f, n, false, hits, nullptr, numSMs, st))
        return;
    const int grid = gridFor(n, 128, numSMs * 16);
    if (counts) k_closest_batch<true><<<grid, 128, 0, st>>>(S, rays, n, hits, counts);
    else k_closest_batch<false><<<grid, 128, 0, st>>>(S, rays, n, hits, nullptr);
}

void launchAnyBatch(const DevScene& S, const float4* rays, const float* maxDist, float eps, size_t n, uint8_t* occluded,
                    int numSMs, cudaStream_t st)
{
    if (n == 0) return;
    if (S.fastRoot != 0u && n >= CGRT_BATCH_SPLIT_MIN && !getenv("CGRT_BATCH_ONE_KERNEL") &&
        launchSplitBatch(S, rays, maxDist, eps, n, true, nullptr, occluded, numSMs, st))
        return;
    k_any_batch<<<gridFor(n, 128, numSMs * 16), 128, 0, st>>>(S, rays, maxDist, eps, n, occluded);
}

void launchBruteBatch(const DevScene& S, const float4* rays, size_t n, float4* hits, int numSMs, cudaStream_t st)
{
    if (n == 0) return;
    k_brute_batch<<<gridFor(n, 128, numSMs * 16), 128, 0, st>>>(S, rays, n, hits);
}

void launchUnitAabb(const float* boxes, const float4* rays, size_t n, uint8_t* hit, float* t, cudaStream_t st)
{
    if (n) k_unit_aabb<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(boxes, rays, n, hit, t);
}
void launchUnitTriangle(const float* tris, const float4* rays, size_t n, float4* out, cudaStream_t st)
{
    if (n) k_unit_triangle<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(tris, rays, n, out);
}
void launchUnitPlane(const float4* planes, const float4* rays, size_t n, uint8_t* hit, float* t, cudaStream_t st)
{
    if (n) k_unit_plane<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(planes, rays, n, hit, t);
}
void launchUnitTrianglePlane(const float* tris, size_t n, float4* planes, cudaStream_t st)
{
    if (n) k_unit_triangle_plane<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(tris, n, planes);
}
void launchUnitPointInTriangle(const float* in, size_t n, uint8_t* inside, cudaStream_t st)
{
    if (n) k_unit_point_in_triangle<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(in, n, inside);
}
void launchUnitSphere(const float4* spheres, const float4* rays, size_t n, float* out, cudaStream_t st)
{
    if (n) k_unit_sphere<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(spheres, rays, n, out);
}

void launchGenerateRays(const FrameParams* dP, int nPixels, float4* rays, cudaStream_t st)
{
    if (nPixels) k_generate_rays<<<(nPixels + 127) / 128, 128, 0, st>>>(dP, rays);
}

// `tr` (optional) records CUDA events around the kernels whose class is selected, for per-kernel device times.
static inline void traceBegin(WaveTrace* tr, int cls, cudaStream_t st)
{
    if (tr && (tr->classMask >> cls & 1) && tr->n < tr->maxKernels) cudaEventRecord(tr->ev[2 * tr->n], st);
}
static inline void traceEnd(WaveTrace* tr, int cls, cudaStream_t st)
{
    if (tr) tr->launches[cls]++;
    if (tr && (tr->classMask >> cls & 1) && tr->n < tr->maxKernels) {
        cudaEventRecord(tr->ev[2 * tr->n + 1], st);
        tr->cls[tr->n++] = cls;
    }
}

// Frame of trace limit 0: trace(0, ...) returns black for every pixel without casting a ray, src/main.cpp:267-272.
// Returns the kernels it launched: 1 when only this rank's pixels of a shared Screen-layout frame are cleared, else 0 (memset).
static int launchBlackFrame(const FrameParams& hP, const FrameParams* dP, const int2* dTileSeq, float* fb, int numSMs,
                            cudaStream_t st)
{
    if (hP.world > 1 && hP.screenLayout) {
        k_clear_tiles<<<gridFor((size_t)hP.nSlots, 128, numSMs * 16), 128, 0, st>>>(dP, dTileSeq, fb);
        return 1;
    }
    const size_t px = hP.world == 1 ? (size_t)hP.width * hP.height * hP.nViews : (size_t)hP.nSlots; // (every view's frame)
    cudaMemsetAsync(fb, 0, px * 3 * sizeof(float), st);
    return 0;
}

// One frame of the level-by-level counting wavefront (CGRT_RENDER_COUNT: sequential leaf scans that count the reference's
// box / triangle tests). Every queue length lives in device memory (B.counts), so the sequence needs no host round trip:
// the grids are sized for the worst case the host knows (nSlots) and the kernels loop over the device-side count.
int launchCountingFrame(const DevScene& S, const FrameParams* dP, const FrameParams& hP, const float4* dLights,
                        const CountBuffers& B, const int* dTileList, float* fb, int numSMs, WaveTrace* tr, cudaStream_t st)
{
    int launches = 0;
    cudaMemsetAsync(B.counts, 0, sizeof(int) * CGRT_CNT_TOTAL, st);
    cudaMemsetAsync(B.tests, 0, sizeof(unsigned long long) * 6, st);
    // (no tile sequence: the counting frame is never rendered into a shared Screen-layout frame, cgrt_render_device refuses it)
    if (hP.traceLimit <= 0) return launchBlackFrame(hP, dP, nullptr, fb, numSMs, st);
    const int persistent = numSMs * 8; // persistent warps: 8 CTAs x 4 warps per SM (register-limited residency is 5-8 CTAs)
    const int gPrimary = gridFor((size_t)hP.nSlots, 128, 1 << 30);
    traceBegin(tr, 0, st);
    k_primary<<<gPrimary, 128, 0, st>>>(S, dP, B, dTileList, fb);
    traceEnd(tr, 0, st);
    launches++;
    const int gHit = gridFor((size_t)hP.nSlots, 128, persistent);
    const int gShadow = gridFor((size_t)hP.nSlots * (hP.nLights > 0 ? hP.nLights : 1), 128, persistent);
    for (int level = 0; level < hP.traceLimit; level++) {
        if (level > 0) {
            traceBegin(tr, 1, st);
            k_bounce_closest<<<gHit, 128, 0, st>>>(S, B, level, fb);
            traceEnd(tr, 1, st);
            launches++;
        }
        if (hP.nLights > 0) {
            traceBegin(tr, 2, st);
            k_shadow<<<gShadow, 128, 0, st>>>(S, dP, dLights, B, level);
            traceEnd(tr, 2, st);
            launches++;
        }
        traceBegin(tr, 3, st);
        k_shade<<<gHit, 128, 0, st>>>(S, dP, dLights, B, level, fb);
        traceEnd(tr, 3, st);
        launches++;
    }
    return launches;
}

int launchPathPipeline(const DevScene& S, const FrameParams* dP, const FrameParams& hP, const float4* dLights,
                       const PathBuffers& B, const int2* dTileSeq, float* fb, int numSMs, WaveTrace* tr, cudaStream_t st)
{
    cudaMemsetAsync(B.counts, 0, sizeof(int) * CGRT_CNT_TOTAL, st);
    if (hP.traceLimit <= 0) return launchBlackFrame(hP, dP, dTileSeq, fb, numSMs, st);
    int launches = 0;
    const int persistent = numSMs * tuning().blocks;
    const int gPaths = min(gridFor((size_t)hP.nSlots, 128, 1 << 30), persistent);
    int* work = B.counts + CGRT_CNT_WORK;
    traceBegin(tr, 0, st);
    if (S.fastRoot != 0u) { // speculative search + certificate; what cannot be certified is replayed exactly
        if (hP.nViews > 1) k_paths_fast<true><<<gPaths, 128, 0, st>>>(S, dP, B, dTileSeq, dLights, fb, work + 0);
        else k_paths_fast<false><<<gPaths, 128, 0, st>>>(S, dP, B, dTileSeq, dLights, fb, work + 0);
        k_paths_replay<<<gPaths, 128, 0, st>>>(S, dP, B, fb, work + 2);
        launches += 2;
        if (tr) tr->launches[0]++;
    } else {
        if (hP.nViews > 1) k_paths<true><<<gPaths, 128, 0, st>>>(S, dP, B, dTileSeq, dLights, fb, work + 0);
        else k_paths<false><<<gPaths, 128, 0, st>>>(S, dP, B, dTileSeq, dLights, fb, work + 0);
        launches++;
    }
    traceEnd(tr, 0, st);
    if (hP.nLights > 0) {
        traceBegin(tr, 2, st);
        if (S.fastRoot != 0u) {
            k_shadow_fast<<<persistent, 128, 0, st>>>(S, dP, dLights, B, work + 1);
            k_shadow_replay<<<persistent, 128, 0, st>>>(S, dP, dLights, B, work + 3);
            launches += 2;
            if (tr) tr->launches[2]++;
        } else {
            k_shadow_all<<<persistent, 128, 0, st>>>(S, dP, dLights, B, work + 1);
            launches++;
        }
        traceEnd(tr, 2, st);
    }
    traceBegin(tr, 3, st);
    k_shade_paths<<<gridFor((size_t)hP.nSlots, 128, numSMs * 16), 128, 0, st>>>(S, dP, dLights, B, fb);
    traceEnd(tr, 3, st);
    launches++;
    return launches;
}

// chains by the size of this rank's share of the frame (measured on the 1080p C3 frame: 4 chains best on one GPU; a chain
// needs enough rays per round to be worth its 18 launches)
int roundPipelineChains(int nSlots)
{
    int c = tuning().chains;
    if (c <= 0) c = nSlots >= 1500000 ? 4 : (nSlots >= 700000 ? 2 : 1);
    return c > CGRT_MAX_CHAINS ? CGRT_MAX_CHAINS : c;
}
// rays per chain-round below which the cooperative search is used (measured: 120 K for one chain, 15 K for four)
static int coopThreshold(int nChains)
{
    const int c = tuning().coop; // > 0: explicit threshold, < 0: never (k_trace only), 0: by chain count
    if (c != 0) return c < 0 ? 0 : c;
    return nChains <= 1 ? 120000 : 60000 / nChains;
}

int launchRoundPipeline(const DevScene& S, const FrameParams* dP, const FrameParams& hP, const float4* dLights,
                        const RoundBuffers* chains, int nChains, const ChainSync& sync, const int2* dTileSeq, float* fb,
                        int numSMs, WaveTrace* tr, cudaStream_t st)
{
    cudaMemsetAsync(chains[0].counts, 0, sizeof(int) * CGRT_CNT_TOTAL * nChains, st); // the chains' counters are contiguous
    if (hP.traceLimit <= 0) return launchBlackFrame(hP, dP, dTileSeq, fb, numSMs, st);
    int launches = 0;
    const int persistent = numSMs * tuning().blocks;
    const int flat = gridFor((size_t)hP.nSlots, 128, numSMs * 16);
    const int flatChain = gridFor((size_t)hP.nSlots / nChains + 1, 128, numSMs * 16);
    const bool shadows = hP.nLights > 0;
    const int rounds = hP.traceLimit + (shadows ? 1 : 0);
    const int coopMax = coopThreshold(nChains);
    // fork: every chain's stream starts after the frame's parameter upload / counter reset on `st`
    if (nChains > 1) {
        cudaEventRecord(sync.fork, st);
        for (int c = 1; c < nChains; c++) cudaStreamWaitEvent(sync.streams[c], sync.fork, 0);
    }
    for (int c = 0; c < nChains; c++) {
        cudaStream_t sc = c == 0 ? st : sync.streams[c];
        traceBegin(tr, 0, sc);
        k_gen<<<flatChain, 128, 0, sc>>>(S, dP, dLights, chains[c], dTileSeq, fb, c, nChains);
        traceEnd(tr, 0, sc);
        launches++;
    }
    for (int r = 0; r < rounds; r++) {
        for (int c = 0; c < nChains; c++) {
            const RoundBuffers& B = chains[c];
            cudaStream_t sc = c == 0 ? st : sync.streams[c];
            int* counts = B.counts;
            // closest-hit rays of level r (list B) + shadow rays of the hits of level r-1 (list A)
            const bool haveC = r < hP.traceLimit, haveS = shadows && r >= 1;
            const float4* raysB = haveC ? B.cRay[r & 1] : nullptr;
            float4* resB = haveC ? B.cRes[r & 1] : nullptr;
            const int* nB = haveC ? counts + CGRT_CNT_BOUNCE + r : nullptr;
            const float4* raysA = haveS ? B.sRay[(r - 1) & 1] : nullptr;
            float4* resA = haveS ? B.sRes[(r - 1) & 1] : nullptr;
            const int* nA = haveS ? counts + CGRT_CNT_HIT + (r - 1) : nullptr;
            traceBegin(tr, 2, sc);
            // the ray count of the round lives on the device: both searches are launched, the one that does not apply returns at once
            if (coopMax < (1 << 30))
                k_trace<<<persistent, 128, 0, sc>>>(S, raysA, resA, nA, hP.nLights, raysB, resB, nB, counts + CGRT_CNT_WORK + r, coopMax);
            if (coopMax > 0)
                k_trace8<<<numSMs * CGRT_TRACE8_MINBLOCKS, 128, 0, sc>>>(S, raysA, resA, nA, hP.nLights, raysB, resB, nB,
                                                                         counts + CGRT_CNT_WORK + r, coopMax);
            launches += (coopMax < (1 << 30) ? 1 : 0) + (coopMax > 0 ? 1 : 0); // both are launches, one returns at once
            traceEnd(tr, 2, sc);
            traceBegin(tr, 1, sc);
            k_finish<<<flatChain, 128, 0, sc>>>(S, dP, dLights, B, r, raysA, resA, nA, raysB, resB, nB, B.cRay[(r + 1) & 1],
                                               B.sRay[r & 1], fb, dTileSeq);
            traceEnd(tr, 1, sc);
            launches++;
        }
    }
    // join
    for (int c = 1; c < nChains; c++) {
        cudaEventRecord(sync.join[c], sync.streams[c]);
        cudaStreamWaitEvent(st, sync.join[c], 0);
    }
    if (hP.nSph > 0) { // spherical-light soft shadows of every hit record of the frame, before the shading pass reads them
        const int capSoft = hP.nSlots * chains[0].levels;
        cudaMemsetAsync(chains[0].softList + capSoft, 0, sizeof(int), st);
        k_soft_list<<<flat, 128, 0, st>>>(dP, chains[0], capSoft);
        k_soft_shadows<<<numSMs * 8, 256, 0, st>>>(S, dP, dLights, chains[0], capSoft);
        launches += 2;
    }
    traceBegin(tr, 3, st);
    k_shade_slots<<<flat, 128, 0, st>>>(S, dP, dLights, chains[0], dTileSeq, fb);
    traceEnd(tr, 3, st);
    launches++;
    return launches;
}

int waveGridBlocks(int numSMs)
{
    static int perSM[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    if (perSM[dev] == 0) {
        const char* cv = getenv("CGRT_WAVE_CARVEOUT"); // % of the SM's 228 KB configured as shared memory (the rest is L1)
        cudaFuncSetAttribute(k_wave, cudaFuncAttributePreferredSharedMemoryCarveout, cv ? atoi(cv) : 25);
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_wave, 128, 0) != cudaSuccess || nb < 1) nb = 1;
        perSM[dev] = nb;
    }
    int b = perSM[dev];
    const int cap = tuning().waveBlocks;
    if (cap > 0 && cap < b) b = cap;
    return numSMs * b;
}

int launchWavePipeline(const DevScene& S, const FrameParams* dP, const FrameParams& hP, const float4* dLights,
                       const RoundBuffers& B, const WaveQ& Q, const int2* dTileSeq, float* fb, int numSMs, WaveTrace* tr,
                       cudaStream_t st)
{
    cudaMemsetAsync(B.counts, 0, sizeof(int) * CGRT_CNT_TOTAL, st);
    cudaMemsetAsync(Q.ctl, 0, sizeof(int) * WCTL_INTS, st);
    if (hP.traceLimit <= 0) return launchBlackFrame(hP, dP, dTileSeq, fb, numSMs, st);
    if (hP.nSlots <= 0) return 0; // this rank owns no pixel of the frame
    // every CTA must be resident at once: warps wait for rays that other CTAs produce
    const int grid = waveGridBlocks(numSMs);
    traceBegin(tr, 2, st);
    k_wave<<<grid, 128, 0, st>>>(S, hP, dLights, Q, B, dTileSeq, fb);
    traceEnd(tr, 2, st);
    return 1;
}

void launchAssemble(const float* gathered, size_t perRankFloats, const int* tileLists, const int* tileCounts, int maxTiles,
                    int world, int tileW, int tileH, int tilesX, int width, int height, float* frame, int numSMs,
                    cudaStream_t st)
{
    const size_t total = (size_t)world * maxTiles * tileW * tileH;
    if (total == 0) return;
    k_assemble<<<gridFor(total, 256, numSMs * 8), 256, 0, st>>>(gathered, perRankFloats, tileLists, tileCounts, maxTiles,
                                                               world, tileW, tileH, tilesX, width, height, frame);
}

// =================================================================================================================
// Frame hand-off between the GPUs of one box (one process per GPU). With CGRT_RENDER_SCREEN_LAYOUT every rank stores its
// pixels straight into the frame of rank 0 through NVLink peer memory, so the only exchange step left is "my pixels of frame
// `seq` have landed" (rank r -> rank 0) and "frame `seq` has been consumed, you may overwrite it" (rank 0 -> rank r):
// 32-bit sequence numbers in device memory, written with system-scope release and polled with system-scope acquire.
// =================================================================================================================
struct FlagPtrs {
    uint32_t* p[CGRT_MAX_PEERS];
};

// runs after everything enqueued before it on the stream (kernel boundary), so the stores of the shading kernels are complete
__global__ void k_flag_signal(FlagPtrs f, int n, uint32_t seq)
{
    const int i = threadIdx.x;
    if (i >= n || f.p[i] == nullptr) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f.p[i]), "r"(seq) : "memory");
}

// one thread per flag; the kernel (and with it the stream) proceeds when every flag has reached `seq`. A peer that never
// arrives must not hang the GPU: after `timeoutNs` the thread gives up and bumps *status.
__global__ void k_flag_wait(const uint32_t* flags, int n, uint32_t seq, unsigned long long timeoutNs, uint32_t* status)
{
    const int i = threadIdx.x;
    if (i >= n) return;
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (true) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + i) : "memory");
        if ((int32_t)(v - seq) >= 0) break;
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > timeoutNs) {
            if (status) atomicAdd(status, 1u);
            break;
        }
        __nanosleep(200);
    }
    __threadfence_system();
}

void launchFlagSignal(uint32_t* const* flags, int n, uint32_t seq, cudaStream_t st)
{
    FlagPtrs f;
    for (int i = 0; i < CGRT_MAX_PEERS; i++) f.p[i] = i < n ? flags[i] : nullptr;
    if (n > 0) k_flag_signal<<<1, CGRT_MAX_PEERS, 0, st>>>(f, n, seq);
}

void launchFlagWait(const uint32_t* flags, int n, uint32_t seq, unsigned long long timeoutNs, uint32_t* status, cudaStream_t st)
{
    if (n > 0) k_flag_wait<<<1, 32 * ((n + 31) / 32), 0, st>>>(flags, n, seq, timeoutNs, status);
}

#ifdef CGRT_INSTRUMENT
void readInstrumentation(unsigned long long* out, bool reset)
{
    cudaMemcpyFromSymbol(out, g_instr, sizeof(unsigned long long) * 16);
    if (reset) {
        unsigned long long z[16] = {0};
        cudaMemcpyToSymbol(g_instr, z, sizeof z);
    }
}
void readStepHist(unsigned int* out, bool reset)
{
    cudaMemcpyFromSymbol(out, g_stepHist, sizeof(unsigned int) * 64);
    if (reset) {
        static unsigned int z[64];
        cudaMemcpyToSymbol(g_stepHist, z, sizeof z);
    }
}
void readTimeline(unsigned int* out, bool reset)
{
    cudaMemcpyFromSymbol(out, g_tl, sizeof(unsigned int) * 2 * 128 * 2);
    if (reset) {
        static unsigned int z[2 * 128 * 2];
        cudaMemcpyToSymbol(g_tl, z, sizeof z);
        unsigned long long m[2] = {~0ull, ~0ull};
        cudaMemcpyToSymbol(g_t0, m, sizeof m);
    }
}
#endif

void launchQuantize(const float* frame, size_t nPixels, uint8_t* rgba, cudaStream_t st)
{
    if (nPixels) k_quantize<<<(unsigned)((nPixels + 255) / 256), 256, 0, st>>>(frame, nPixels, rgba);
}

} // namespace cgrt
