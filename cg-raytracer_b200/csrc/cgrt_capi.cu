// extern "C" boundary of libcgrt_b200.so (include/cgrt_b200.h). Host logic only: scene flattening, BVH build (bvh_build.cpp),
// uploads, per-frame constants, queue allocation, kernel sequencing. No CPU implementation of the path lives here: every
// query is answered by the kernels in cgrt_kernels.cu, and every entry fails loudly when no CUDA device is usable.
#include "../../include/cgrt_b200.h"
#include "bvh_build.h"
#include "cgrt_kernels.h"

#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

using namespace cgrt;
#ifdef CGRT_INSTRUMENT
namespace cgrt { void readInstrumentation(unsigned long long* out, bool reset); void readTimeline(unsigned int* out, bool reset); void readStepHist(unsigned int* out, bool reset); }
#endif

static thread_local std::string g_err;
static int fail(int code, const std::string& msg)
{
    g_err = msg;
    return code;
}
#define CK(call)                                                                                                      \
    do {                                                                                                              \
        cudaError_t e_ = (call);                                                                                      \
        if (e_ != cudaSuccess) {                                                                                      \
            char buf_[512];                                                                                           \
            snprintf(buf_, sizeof buf_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return fail((e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver) ? CGRT_ERR_NO_DEVICE           \
                                                                                        : CGRT_ERR_CUDA,               \
                        buf_);                                                                                        \
        }                                                                                                             \
    } while (0)

static int useDevice(int device);
static int useSceneDevice(const cgrt_scene* s);

static int useDevice(int device)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(CGRT_ERR_NO_DEVICE, std::string("no usable CUDA device (the product has no CPU path): ") +
                                            (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    if (device < 0 || device >= n) return fail(CGRT_ERR_INVALID, "device ordinal out of range");
    CK(cudaSetDevice(device));
    return CGRT_OK;
}

struct DeviceInfo {
    int numSMs = 0;
};
static int deviceInfo(int device, DeviceInfo& di)
{
    static std::mutex mu;
    static std::map<int, DeviceInfo> cache;
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(device);
    if (it == cache.end()) {
        DeviceInfo d;
        CK(cudaDeviceGetAttribute(&d.numSMs, cudaDevAttrMultiProcessorCount, device));
        it = cache.emplace(device, d).first;
    }
    di = it->second;
    return CGRT_OK;
}

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    int ensure(size_t count)
    {
        if (count <= n && p) return CGRT_OK;
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        if (count == 0) count = 1;
        cudaError_t e = cudaMalloc((void**)&p, count * sizeof(T));
        if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? CGRT_ERR_OOM : CGRT_ERR_CUDA,
                                          std::string("cudaMalloc failed: ") + cudaGetErrorString(e));
        n = count;
        return CGRT_OK;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
};

// ---- tile partition --------------------------------------------------------------------------------------------------
// Interleaved screen tiles: tile (tx,ty) belongs to rank (tx + ty*skew) mod world, skew coprime to world so that the
// compact lit region of a frame spreads evenly over the GPUs (SURVEY.md §8(e)).
struct TileLayout {
    int tileW, tileH, tilesX, tilesY, world, skew, maxTiles;
    std::vector<std::vector<int>> lists; // per rank: owned global tile ids, increasing
};
static int gcdInt(int a, int b) { return b == 0 ? a : gcdInt(b, a % b); }
static void makeTileLayout(const cgrt_render_params& p, TileLayout& L)
{
    L.tileW = p.tile_w > 0 ? p.tile_w : 8;
    L.tileH = p.tile_h > 0 ? p.tile_h : 8;
    L.tilesX = (p.width + L.tileW - 1) / L.tileW;
    L.tilesY = (p.height + L.tileH - 1) / L.tileH;
    L.world = p.world > 0 ? p.world : 1;
    L.skew = 1;
    if (L.world > 1) {
        L.skew = 3;
        while (gcdInt(L.skew, L.world) != 1) L.skew++;
    }
    L.lists.assign(L.world, std::vector<int>());
    for (int ty = 0; ty < L.tilesY; ty++)
        for (int tx = 0; tx < L.tilesX; tx++) L.lists[(tx + ty * L.skew) % L.world].push_back(ty * L.tilesX + tx);
    L.maxTiles = 0;
    for (auto& l : L.lists) L.maxTiles = std::max(L.maxTiles, (int)l.size());
}

static int checkRenderParams(const cgrt_render_params* p)
{
    if (!p) return fail(CGRT_ERR_INVALID, "null render params");
    if (p->width <= 0 || p->height <= 0) return fail(CGRT_ERR_INVALID, "width/height must be positive");
    if ((int64_t)p->width * p->height > (int64_t)1 << 28) return fail(CGRT_ERR_INVALID, "frame too large");
    if (p->trace_limit < 0 || p->trace_limit > CGRT_MAX_LEVELS) return fail(CGRT_ERR_INVALID, "trace_limit out of range");
    if (p->world < 1 || p->rank < 0 || p->rank >= p->world) return fail(CGRT_ERR_INVALID, "rank/world invalid");
    if (p->tile_w < 0 || p->tile_h < 0 || p->tile_w > 64 || p->tile_h > 64) return fail(CGRT_ERR_INVALID, "tile size invalid");
    return CGRT_OK;
}

// ---- camera constants (host, libm): Trackball::position / generateRay, glm::quat(euler), quat * vec3 ---------------------
static void crossH(const float a[3], const float b[3], float r[3])
{
    r[0] = a[1] * b[2] - b[1] * a[2];
    r[1] = a[2] * b[0] - b[2] * a[0];
    r[2] = a[0] * b[1] - b[0] * a[1];
}
static void cameraConstants(const cgrt_camera& c, FrameParams& P)
{
    // glm::quat(eulerAngles): c = cos(e*0.5), s = sin(e*0.5)
    const float hx = c.euler[0] * 0.5f, hy = c.euler[1] * 0.5f, hz = c.euler[2] * 0.5f;
    const float cx = std::cos(hx), cy = std::cos(hy), cz = std::cos(hz);
    const float sx = std::sin(hx), sy = std::sin(hy), sz = std::sin(hz);
    P.qw = cx * cy * cz + sx * sy * sz;
    P.qx = sx * cy * cz - cx * sy * sz;
    P.qy = cx * sy * cz + sx * cy * sz;
    P.qz = cx * cy * sz - sx * sy * cz;
    // position = lookAt + q * (0, 0, -dist)   (framework/src/trackball.cpp:70-73)
    const float q[3] = {P.qx, P.qy, P.qz};
    const float v[3] = {0.0f, 0.0f, -c.dist};
    float uv[3], uuv[3];
    crossH(q, v, uv);
    crossH(q, uv, uuv);
    P.camX = c.look_at[0] + (v[0] + ((uv[0] * P.qw) + uuv[0]) * 2.0f);
    P.camY = c.look_at[1] + (v[1] + ((uv[1] * P.qw) + uuv[1]) * 2.0f);
    P.camZ = c.look_at[2] + (v[2] + ((uv[2] * P.qw) + uuv[2]) * 2.0f);
    P.halfH = std::tan(c.fovy / 2.0f);   // framework/src/trackball.cpp:94
    P.halfW = c.aspect * P.halfH;        // :95
}

// ---- structural self-check of the fast tree (host, at build time; exported through cgrt_bvh_fast_tree_stats) ------------
// out: [0] 8-wide nodes reachable from the root, [1] triangles reachable, [2] triangles reached more than once or never,
//      [3] vertices outside the box of the child slot they hang under (boxes must CONTAIN their geometry), [4] depth in 8-wide
//      levels, [5] parent-chain errors (a triangle's leaf must reach node 0 through `parent`), [6] 1 = tree present
static void fastTreeSelfCheck(const std::vector<MeshView>& views, const BuiltBVH& bvh, int64_t out[8])
{
    for (int k = 0; k < 8; k++) out[k] = 0;
    if (bvh.fastRoot == 0u) return;
    out[6] = 1;
    const uint32_t ID_MASK = 0x03ffffffu, ID_TRI = 0x20000000u;
    std::vector<int> seen(bvh.leafTris.size(), 0);
    std::vector<char> always(bvh.leafTris.size(), 0);
    for (int32_t a : bvh.alwaysTest) always[a] = 1;
    out[7] = (int64_t)bvh.alwaysTest.size();
    struct Item { uint32_t id; int depth; float lo[3], hi[3]; };
    std::vector<Item> stack;
    Item root{bvh.fastRoot, 1, {-FLT_MAX, -FLT_MAX, -FLT_MAX}, {FLT_MAX, FLT_MAX, FLT_MAX}};
    stack.push_back(root);
    while (!stack.empty()) {
        const Item it = stack.back();
        stack.pop_back();
        if (it.id & ID_TRI) {
            const int first = (int)(it.id & ID_MASK), count = (int)((it.id >> 26) & 7u) + 1;
            for (int ft = first; ft < first + count; ft++) {
                // leaves hold positions of the fast tree's own order (identity unless the SAH tree is used)
                const int t = bvh.fastOrder.empty() ? ft : (ft >= 0 && (size_t)ft < bvh.fastOrder.size() ? bvh.fastOrder[ft] : -1);
                if (t < 0 || (size_t)t >= seen.size()) { out[2]++; continue; }
                seen[t]++;
                out[1]++;
                const LeafTri lt = bvh.leafTris[t];
                const MeshView& mv = views[lt.mesh];
                for (int k = 0; k < 3 && !always[t]; k++) { // (always-list triangles are not covered by the boxes by design)
                    const float* v = mv.vertices + 6 * (size_t)mv.triangles[3 * (size_t)lt.tri + k];
                    for (int a = 0; a < 3; a++)
                        if (std::isfinite(v[a]) && (v[a] < it.lo[a] || v[a] > it.hi[a])) out[3]++;
                }
                // the certificate's chain: leaf -> ... -> root
                int node = bvh.triLeafNode[t], guard = 0;
                while (node > 0 && guard++ < 64) node = bvh.parent[node];
                if (node != 0 || !bvh.nodes[bvh.triLeafNode[t]].isLeaf || t < bvh.nodes[bvh.triLeafNode[t]].firstTri ||
                    t >= bvh.nodes[bvh.triLeafNode[t]].firstTri + bvh.nodes[bvh.triLeafNode[t]].triCount)
                    out[5]++;
            }
            continue;
        }
        const WideNode& w = bvh.wide[it.id & ID_MASK];
        out[0]++;
        out[4] = std::max<int64_t>(out[4], it.depth);
        for (int c = 0; c < 8; c++) {
            if (w.id[c] == 0u) continue;
            Item ch{w.id[c], it.depth + 1, {w.lo[c][0], w.lo[c][1], w.lo[c][2]}, {w.hi[c][0], w.hi[c][1], w.hi[c][2]}};
            stack.push_back(ch);
        }
    }
    if (!bvh.fastOrder.empty()) // SAH tree: the always-list triangles are outside the tree by construction
        for (int32_t a : bvh.alwaysTest) { seen[a]++; out[1]++; }
    for (int v : seen)
        if (v != 1) out[2]++;
}

// ---- the scene object --------------------------------------------------------------------------------------------------
// Share of the SMs that finish (WaveQ::finEvery), found by measurement: how much finishing a frame needs per search step
// depends on the scene (hit rate, lights, how long the searches are), and a wrong split leaves one of the two stages waiting.
// Frames of one shape rendered repeatedly (the UI re-renders every frame, main.cpp:907-914) are timed on the device (an event
// pair per frame, read back when complete - the renderer never waits for it); the neighbours of the current setting are tried
// NOTE on synchronous copies: cudaMemcpy from PAGEABLE host memory returns when the data has been staged, not when the DMA
// has landed, and cudaMemset is asynchronous as well; both run on the legacy default stream, which the scene's NON-BLOCKING
// streams (and the callers' own) are not ordered with. Every upload a later kernel depends on is therefore followed by
// uploadsDone() before anything is launched (found by tools/wave_soak.py: a frame of another shape rendered with the previous
// shape's tile list once in ~3000 shape changes).
static cudaError_t uploadsDone() { return cudaDeviceSynchronize(); }

// once each and the fastest is kept. Scheduling only: every setting renders the same pixels.
struct WaveTuner {
    static const int RING = 8, LO = 2, HI = 14;
    int key[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int cur = 0;                 // current setting (0 = not started)
    float ms[HI + 2] = {0};      // best device time seen per setting, 0 = unknown
    int pendingOf[HI + 2] = {0}; // frames in flight per setting
    int frames = 0;
    struct Slot { cudaEvent_t a = nullptr, b = nullptr; int setting = 0; bool busy = false; } ring[RING];
    int next = 0, recording = -1;
};

// The kernel set that renders a frame (cgrt_kernels.h). The values are ABI: cgrt_render_stats::pipeline reports them and
// capi.class_names and bench.py index by them.
enum FramePipeline : uint32_t { PIPE_COUNT = 0, PIPE_PATHS = 1, PIPE_ROUNDS = 2, PIPE_WAVE = 3 };

struct cgrt_scene {
    int device = 0;
    DeviceInfo di;
    std::mutex mu;    // renders: the per-scene queues and the parameter ring are shared by the frames of one scene
    std::mutex hostMu; // the host-pointer render forms (cgrt_render, _effects, _submit): one frame of a scene at a time through its
                       // internal frame buffer and stream
    std::mutex devMu; // the pointer table `dev` (queries take a snapshot; set_spheres replaces the sphere entries)
    cudaStream_t stream = nullptr;

    BuiltBVH bvh;
    std::vector<int32_t> leafGlobalId; // leaf order -> global triangle id
    bool hostOnly = false;             // built with CGRT_SCENE_HOST_ONLY: no device state, queries are refused
    int64_t nTris = 0;
    int nMeshes = 0;

    DevBuf<float4> wide8, tri4, tri4f, nodes, triPl, triV0, triV1, triV2, triN0, triN1, triN2, mats, spheres, pairs, wide;
    DevBuf<int> origToLeaf, refParent, alwaysTri, fastOrder;
    DevScene dev{};

    std::vector<cgrt_point_light> lights;
    std::vector<float> sphLights; // [n][7] position, radius, colour (src/scene.h:47-51)
    unsigned softSeed = 1u;
    DevBuf<int> softList;
    DevBuf<float> soft;

    // per-frame parameter block: pinned ring -> device block
    static const int RING = 64;
    unsigned char* hParamRing = nullptr; // RING x paramBlockBytes, pinned
    size_t paramBlockBytes = 0;
    int ringPos = 0;
    DevBuf<unsigned char> dParamBlock;

    // wavefront queues
    DevBuf<float4> hitQ, bounceQ, pathState;
    DevBuf<uint8_t> lit;
    DevBuf<int> pathPix, counts, tileList;
    DevBuf<unsigned long long> tests;
    DevBuf<float4> hitRec;
    DevBuf<int> hitList, pathDepth, replayShadow;
    DevBuf<float4> replayQ;
    DevBuf<float4> cRay[2], cRes[2], sRay[2], sRes[2];
    DevBuf<float4> waveRays, waveFin; // persistent wavefront: ticket-indexed ray records / finished-search records
    DevBuf<int> waveCtl, waveTrace;
    DevBuf<float4> waveResume;
    DevBuf<unsigned> waveLat;
    uint32_t waveSeq = 0;
    FramePipeline lastPipeline = PIPE_COUNT; // kernel set of the last frame (choosePipeline)
    int lastChains = 1;                      // PIPE_ROUNDS: chains of the last frame (their counters are summed)
    // streaming form (cgrt_render_submit / cgrt_render_wait)
    cudaStream_t copyStream = nullptr;
    cudaEvent_t renderDone[2] = {nullptr, nullptr}, copyDone[2] = {nullptr, nullptr};
    DevBuf<float> streamFrame[2];
    DevBuf<float> fxA, fxB, fxC, fxM; // cgrt_render_effects: supersampled / shifted frame, accumulator, bloom output, bloom matrix
    DevBuf<int> fxProg;               // bloom: finished columns per image row
    bool slotUsed[2] = {false, false};
    uint64_t submitSeq = 0;
    int64_t fastStats[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    ChainSync chainSync{};
    std::vector<cudaEvent_t> traceEvents;
    WaveTrace trace{};
    // tile partition of the current frame geometry (rebuilt only when width/height/tile/world/rank change)
    TileLayout layout;
    DevBuf<int2> tileSeq; // production order: (global tile id, local tile index), centre-out
    uint64_t primaryPixels = 0; // pixels of this rank inside the image
    int tileKey[6] = {0, 0, 0, 0, 0, 0};
    DevBuf<float> frame; // internal framebuffer for the host-pointer render
    DevBuf<float> zeroFrame; // all zeros: source of the copy-engine transfer that blanks a page-locked destination while it renders
    float* hFramePinned = nullptr;
    size_t hFramePinnedFloats = 0;

    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    WaveTuner tuner;
    cudaStream_t lastStream = nullptr;
    uint64_t lastLaunches = 0;
    FrameParams lastParams{};
    bool haveLast = false;
    int* hStats = nullptr;       // page-locked: the frame's counters + the wavefront's watchdog word, copied behind a synchronous
    bool statsOnHost = false;    // frame on its own stream so that collecting the statistics costs no further round trips
};

static int useSceneDevice(const cgrt_scene* s)
{
    if (s->hostOnly)
        return fail(CGRT_ERR_NO_DEVICE, "scene was created with CGRT_SCENE_HOST_ONLY (BVH introspection only): "
                                        "queries need a device-resident scene; there is no CPU path");
    return useDevice(s->device);
}

static void destroyScene(cgrt_scene* s)
{
    if (!s) return;
    if (s->hostOnly) {
        delete s;
        return;
    }
    cudaSetDevice(s->device);
    s->wide8.release(); s->tri4.release(); s->tri4f.release(); s->fastOrder.release(); s->nodes.release(); s->triPl.release(); s->triV0.release(); s->triV1.release(); s->triV2.release();
    s->triN0.release(); s->triN1.release(); s->triN2.release(); s->mats.release(); s->spheres.release();
    s->origToLeaf.release(); s->refParent.release(); s->alwaysTri.release(); s->pairs.release(); s->wide.release(); s->dParamBlock.release(); s->hitQ.release(); s->bounceQ.release(); s->pathState.release();
    s->lit.release(); s->pathPix.release(); s->counts.release(); s->tileList.release(); s->tileSeq.release(); s->frame.release();
    s->tests.release(); s->hitRec.release(); s->hitList.release(); s->pathDepth.release(); s->replayShadow.release(); s->replayQ.release();
    for (int k = 0; k < 2; k++) { s->cRay[k].release(); s->cRes[k].release(); s->sRay[k].release(); s->sRes[k].release(); }
    s->softList.release(); s->soft.release();
    s->waveRays.release(); s->waveFin.release(); s->waveCtl.release(); s->waveTrace.release(); s->waveResume.release();
    for (cudaEvent_t e : s->traceEvents) cudaEventDestroy(e);
    if (s->hParamRing) cudaFreeHost(s->hParamRing);
    if (s->hFramePinned) cudaFreeHost(s->hFramePinned);
    if (s->hStats) cudaFreeHost(s->hStats);
    if (s->chainSync.fork) {
        cudaEventDestroy(s->chainSync.fork);
        for (int c = 1; c < CGRT_MAX_CHAINS; c++) {
            if (s->chainSync.streams[c]) cudaStreamDestroy(s->chainSync.streams[c]);
            if (s->chainSync.join[c]) cudaEventDestroy(s->chainSync.join[c]);
        }
    }
    if (s->copyStream) {
        cudaStreamDestroy(s->copyStream);
        for (int k = 0; k < 2; k++) { cudaEventDestroy(s->renderDone[k]); cudaEventDestroy(s->copyDone[k]); }
    }
    s->streamFrame[0].release(); s->streamFrame[1].release();
    s->zeroFrame.release();
    s->fxA.release(); s->fxB.release(); s->fxC.release(); s->fxM.release(); s->fxProg.release();
    for (WaveTuner::Slot& sl : s->tuner.ring) { if (sl.a) cudaEventDestroy(sl.a); if (sl.b) cudaEventDestroy(sl.b); }
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

static int uploadSpheres(cgrt_scene* s, const float* spheres, int n)
{
    std::vector<float4> h((size_t)std::max(n, 0) * 3);
    for (int i = 0; i < n; i++) {
        const float* p = spheres + 12 * (size_t)i;
        h[3 * i + 0] = make_float4(p[0], p[1], p[2], p[3]);
        h[3 * i + 1] = make_float4(p[4], p[5], p[6], p[10]);
        h[3 * i + 2] = make_float4(p[7], p[8], p[9], p[11]);
    }
    int rc = s->spheres.ensure(h.size());
    if (rc) return rc;
    if (n > 0) CK(cudaMemcpy(s->spheres.p, h.data(), h.size() * sizeof(float4), cudaMemcpyHostToDevice));
    CK(uploadsDone());
    s->dev.spheres = s->spheres.p;
    s->dev.nSpheres = n;
    return CGRT_OK;
}

extern "C" {

int cgrt_version(void) { return CGRT_VERSION; }
const char* cgrt_last_error(void) { return g_err.c_str(); }

int cgrt_device_count(int* count)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (count) *count = (e == cudaSuccess) ? n : 0;
    if (e != cudaSuccess || n == 0)
        return fail(CGRT_ERR_NO_DEVICE, std::string("no usable CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count 0"));
    return CGRT_OK;
}

int cgrt_scene_create(const cgrt_scene_desc* d, const cgrt_scene_options* opt, cgrt_scene** out)
{
    if (!d || !out) return fail(CGRT_ERR_INVALID, "null argument");
    *out = nullptr;
    if (d->n_meshes < 0 || d->n_spheres < 0) return fail(CGRT_ERR_INVALID, "negative counts");
    const int device = opt ? opt->device : 0;
    int maxDepth = (opt && opt->bvh_max_depth > 0) ? opt->bvh_max_depth : 12; // src/bounding_volume_hierarchy.cpp:48
    if (maxDepth > CGRT_MAX_BVH_DEPTH) return fail(CGRT_ERR_INVALID, "bvh_max_depth exceeds the traversal stack");
    const bool hostOnly = opt && (opt->flags & CGRT_SCENE_HOST_ONLY);
    int rc = hostOnly ? CGRT_OK : useDevice(device);
    if (rc) return rc;

    // ---- validate + view the meshes
    std::vector<MeshView> views;
    size_t vo = 0, to = 0;
    int32_t gid = 0;
    for (int m = 0; m < d->n_meshes; m++) {
        const int nv = d->mesh_vertex_count[m], nt = d->mesh_triangle_count[m];
        if (nv <= 0 || nt <= 0)
            return fail(CGRT_ERR_INVALID, "mesh without vertices/triangles (the reference dereferences triangles[0], bvh.cpp:237)");
        MeshView v;
        v.vertices = d->vertices + 6 * vo;
        v.triangles = d->triangles + 3 * to;
        v.nv = nv;
        v.nt = nt;
        v.triOffset = gid;
        for (size_t i = 0; i < (size_t)nt * 3; i++)
            if (v.triangles[i] >= (uint32_t)nv) return fail(CGRT_ERR_INVALID, "triangle index out of range");
        views.push_back(v);
        vo += nv;
        to += nt;
        gid += nt;
    }

    cgrt_scene* s = new cgrt_scene();
    s->device = device;
    s->nTris = gid;
    s->nMeshes = d->n_meshes;
    s->hostOnly = hostOnly;
    if (!hostOnly) {
        rc = deviceInfo(device, s->di);
        if (rc) { destroyScene(s); return rc; }
    }

    // ---- host build with the reference split rule
    buildReferenceBVH(views, maxDepth, s->bvh);
    const size_t T = s->bvh.leafTris.size();
    const size_t NN = s->bvh.nodes.size();
    s->leafGlobalId.resize(T); // the reference's own leaf order (introspection); device arrays may be permuted inside leaves
    for (size_t i = 0; i < T; i++) s->leafGlobalId[i] = views[s->bvh.leafTris[i].mesh].triOffset + s->bvh.leafTris[i].tri;
    const bool subTrees = !(opt && (opt->flags & CGRT_SCENE_NO_SUBTREES));
    const bool fastTree = subTrees && !(opt && (opt->flags & CGRT_SCENE_EXACT_ONLY));
    if (subTrees) {
        // sub-leaf size of the culling sub-trees (speed only; CGRT_SUBLEAF / CGRT_MINLEAF override for tuning)
        int subLeaf = 6, minLeaf = 8;
        if (const char* e = getenv("CGRT_SUBLEAF")) subLeaf = std::max(1, std::min(8, atoi(e)));
        if (const char* e = getenv("CGRT_MINLEAF")) minLeaf = std::max(2, atoi(e));
        buildLeafSubTrees(views, s->bvh, minLeaf, subLeaf);
    } else {
        s->bvh.leafRank.assign(T, 0);
        for (const HostNode& n : s->bvh.nodes)
            if (n.isLeaf)
                for (int i = 0; i < n.triCount; i++) s->bvh.leafRank[n.firstTri + i] = i;
    }
    if (fastTree) {
        // fast-tree flavour (speed only; results do not depend on it): independent binned-SAH tree unless CGRT_FAST_TREE=ref
        const char* ft = getenv("CGRT_FAST_TREE");
        buildFastTree(views, s->bvh, !(ft && std::string(ft) == "ref"));
        fastTreeSelfCheck(views, s->bvh, s->fastStats);
    }
    if (hostOnly) { // BVH introspection only (builder tests on machines without a GPU); every query entry refuses it
        *out = s;
        return CGRT_OK;
    }

    // ---- flatten: 32-byte nodes + leaf-ordered SoA triangles
    std::vector<float4> hNodes(NN * 2);
    for (size_t i = 0; i < NN; i++) {
        const HostNode& n = s->bvh.nodes[i];
        uint32_t a, b;
        if (n.isLeaf) { a = (uint32_t)n.firstTri; b = (uint32_t)n.triCount; }
        else { a = (uint32_t)n.child0; b = 0u; }
        float fa, fb;
        std::memcpy(&fa, &a, 4);
        std::memcpy(&fb, &b, 4);
        hNodes[2 * i] = make_float4(n.lo[0], n.lo[1], n.lo[2], fa);
        hNodes[2 * i + 1] = make_float4(n.hi[0], n.hi[1], n.hi[2], fb);
    }
    std::vector<float4> hv[3], hn[3];
    for (int k = 0; k < 3; k++) { hv[k].resize(T); hn[k].resize(T); }
    std::vector<int> hOrigToLeaf((size_t)gid, 0);
    for (size_t i = 0; i < T; i++) {
        const LeafTri lt = s->bvh.leafTris[i];
        const MeshView& mv = views[lt.mesh];
        const int32_t g = mv.triOffset + lt.tri;
        hOrigToLeaf[g] = (int)i;
        for (int k = 0; k < 3; k++) {
            const float* vtx = mv.vertices + 6 * (size_t)mv.triangles[3 * (size_t)lt.tri + k];
            float w = 0.0f;
            if (k == 0) std::memcpy(&w, &g, 4);
            if (k == 1) std::memcpy(&w, &lt.mesh, 4);
            if (k == 2) std::memcpy(&w, &s->bvh.leafRank[i], 4);
            hv[k][i] = make_float4(vtx[0], vtx[1], vtx[2], w);
            float nw = 0.0f; // triN0.w: reference leaf of the triangle (certification of the speculative traversal)
            if (k == 0 && i < s->bvh.triLeafNode.size()) std::memcpy(&nw, &s->bvh.triLeafNode[i], 4);
            hn[k][i] = make_float4(vtx[3], vtx[4], vtx[5], nw);
        }
    }
    std::vector<float4> hMats((size_t)d->n_meshes * 2);
    for (int m = 0; m < d->n_meshes; m++) {
        const float* p = d->materials + 8 * (size_t)m;
        hMats[2 * m] = make_float4(p[0], p[1], p[2], p[6]);
        hMats[2 * m + 1] = make_float4(p[3], p[4], p[5], p[7]);
    }

#define UP(buf, vec)                                                                                         \
    do {                                                                                                     \
        rc = s->buf.ensure((vec).size());                                                                    \
        if (rc) { destroyScene(s); return rc; }                                                              \
        if (!(vec).empty()) {                                                                                \
            cudaError_t e_ = cudaMemcpy(s->buf.p, (vec).data(), (vec).size() * sizeof((vec)[0]), cudaMemcpyHostToDevice); \
            if (e_ != cudaSuccess) { destroyScene(s); return fail(CGRT_ERR_CUDA, cudaGetErrorString(e_)); }   \
        }                                                                                                    \
    } while (0)
    UP(nodes, hNodes);
    UP(triV0, hv[0]); UP(triV1, hv[1]); UP(triV2, hv[2]);
    UP(triN0, hn[0]); UP(triN1, hn[1]); UP(triN2, hn[2]);
    UP(mats, hMats);
    UP(origToLeaf, hOrigToLeaf);
    std::vector<int> hParent(s->bvh.parent.begin(), s->bvh.parent.end());
    if (hParent.empty()) hParent.assign(std::max<size_t>(NN, 1), -1);
    UP(refParent, hParent);
    std::vector<int> hAlways(s->bvh.alwaysTest.begin(), s->bvh.alwaysTest.end());
    UP(alwaysTri, hAlways);
    // ---- the production traversal's node array: one 4 x float4 entry per inner node (reference or sub-tree) holding both
    // children with their visit ids (encoding documented in cgrt_device.cuh)
    const uint32_t ID_MASK = 0x03ffffffu, ID_REFLEAF = 0x10000000u, ID_TRI = 0x20000000u, ID_SUB = 0x40000000u,
                   ID_REFSCAN = 0x80000000u;
    if (s->bvh.wideRoot.size() != NN) s->bvh.wideRoot.assign(NN, -1);
    const int nRefPairs = NN > 0 ? (int)(NN - 1) / 2 : 0;
    if ((size_t)nRefPairs > ID_MASK || s->bvh.wide.size() > ID_MASK || T > ID_MASK || NN > ID_MASK) {
        destroyScene(s);
        return fail(CGRT_ERR_INVALID, "scene too large for the 26-bit node ids of the traversal");
    }
    auto pack = [](const float lo[3], const float hi[3], uint32_t w0, uint32_t w1, float4* out) {
        float f0, f1;
        std::memcpy(&f0, &w0, 4);
        std::memcpy(&f1, &w1, 4);
        out[0] = make_float4(lo[0], lo[1], lo[2], f0);
        out[1] = make_float4(hi[0], hi[1], hi[2], f1);
    };
    auto refId = [&](int cidx) -> uint32_t {
        const HostNode& n = s->bvh.nodes[cidx];
        if (!n.isLeaf) return (uint32_t)((n.child0 - 1) / 2);
        const int wr = s->bvh.wideRoot[cidx];
        if (wr >= 0) return ID_REFLEAF | (uint32_t)wr;
        return ID_REFSCAN | (uint32_t)cidx;
    };
    (void)ID_TRI; (void)ID_SUB;
    std::vector<float4> hPairs((size_t)nRefPairs * 4);
    for (size_t i = 0; i < NN; i++) {
        const HostNode& n = s->bvh.nodes[i];
        if (n.isLeaf) continue;
        float4* out = hPairs.data() + 4 * (size_t)((n.child0 - 1) / 2);
        const HostNode &l = s->bvh.nodes[n.child0], &r = s->bvh.nodes[n.child1];
        pack(l.lo, l.hi, refId(n.child0), (uint32_t)n.child0, out);
        pack(r.lo, r.hi, refId(n.child1), (uint32_t)n.child1, out + 2);
    }
    std::vector<float4> hWide(s->bvh.wide.size() * 16, make_float4(0.0f, 0.0f, 0.0f, 0.0f)); // 256-byte nodes (cgrt_device.cuh CGRT_WIDE_STRIDE)
    for (size_t j = 0; j < s->bvh.wide.size(); j++) {
        const WideNode& n = s->bvh.wide[j];
        float4* out = hWide.data() + 16 * j;
        for (int k = 0; k < 3; k++)
            for (int h = 0; h < 2; h++) {
                out[2 * k + h] = make_float4(n.lo[4 * h][k], n.lo[4 * h + 1][k], n.lo[4 * h + 2][k], n.lo[4 * h + 3][k]);
                out[6 + 2 * k + h] = make_float4(n.hi[4 * h][k], n.hi[4 * h + 1][k], n.hi[4 * h + 2][k], n.hi[4 * h + 3][k]);
            }
        for (int h = 0; h < 2; h++) {
            float f[4];
            std::memcpy(f, &n.id[4 * h], 16);
            out[12 + h] = make_float4(f[0], f[1], f[2], f[3]);
        }
    }
    UP(wide, hWide);
    std::vector<float4> hWide8(s->bvh.wide.size() * 16);
    for (size_t jn = 0; jn < s->bvh.wide.size(); jn++) {
        const WideNode& n = s->bvh.wide[jn];
        for (int c = 0; c < 8; c++) {
            float fid;
            std::memcpy(&fid, &n.id[c], 4);
            hWide8[16 * jn + 2 * c] = make_float4(n.lo[c][0], n.lo[c][1], n.lo[c][2], fid);
            hWide8[16 * jn + 2 * c + 1] = make_float4(n.hi[c][0], n.hi[c][1], n.hi[c][2], 0.0f);
        }
    }
    UP(wide8, hWide8);
    s->dev.rootId = NN > 0 ? (int)refId(0) : 0;
    UP(pairs, hPairs);
#undef UP
    rc = s->triPl.ensure(T);
    if (rc) { destroyScene(s); return rc; }
    rc = s->tri4.ensure(4 * T);
    if (rc) { destroyScene(s); return rc; }
    rc = s->tri4f.ensure(4 * T);
    if (rc) { destroyScene(s); return rc; }
    if (s->bvh.fastOrder.size() == T && T > 0) {
        std::vector<int> hOrder(s->bvh.fastOrder.begin(), s->bvh.fastOrder.end());
        rc = s->fastOrder.ensure(T);
        if (rc) { destroyScene(s); return rc; }
        cudaError_t e_ = cudaMemcpy(s->fastOrder.p, hOrder.data(), T * sizeof(int), cudaMemcpyHostToDevice);
        if (e_ != cudaSuccess) { destroyScene(s); return fail(CGRT_ERR_CUDA, cudaGetErrorString(e_)); }
    }

    cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev1);
    if (e != cudaSuccess) { destroyScene(s); return fail(CGRT_ERR_CUDA, cudaGetErrorString(e)); }

    e = uploadsDone(); // (see the note on synchronous copies)
    if (e != cudaSuccess) { destroyScene(s); return fail(CGRT_ERR_CUDA, cudaGetErrorString(e)); }
    launchSetupPlanes(s->triV0.p, s->triV1.p, s->triV2.p, s->triPl.p, s->tri4.p, (int)T, s->stream);
    launchPermuteTri4(s->tri4.p, s->bvh.fastOrder.size() == T ? s->fastOrder.p : nullptr, s->tri4f.p, (int)T, s->stream);
    e = cudaStreamSynchronize(s->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { destroyScene(s); return fail(CGRT_ERR_CUDA, std::string("plane set-up kernel: ") + cudaGetErrorString(e)); }

    s->dev.nodes = s->nodes.p;
    s->dev.triPl = s->triPl.p;
    s->dev.tri4 = s->tri4.p;
    s->dev.tri4f = s->tri4f.p;
    s->dev.triV0 = s->triV0.p; s->dev.triV1 = s->triV1.p; s->dev.triV2 = s->triV2.p;
    s->dev.triN0 = s->triN0.p; s->dev.triN1 = s->triN1.p; s->dev.triN2 = s->triN2.p;
    s->dev.mats = s->mats.p;
    s->dev.origToLeaf = s->origToLeaf.p;
    s->dev.pairs = s->pairs.p;
    s->dev.wide = s->wide.p;
    s->dev.wide8 = s->wide8.p;
    s->dev.refParent = s->refParent.p;
    s->dev.alwaysTri = s->alwaysTri.p;
    s->dev.nAlways = s->bvh.fastRoot != 0u ? (int)s->bvh.alwaysTest.size() : 0;
    s->dev.fastRoot = s->bvh.fastRoot;
    s->dev.nNodes = (int)NN;
    s->dev.nTris = (int)T;
    s->dev.nMeshes = d->n_meshes;
    rc = uploadSpheres(s, d->spheres, d->n_spheres);
    if (rc) { destroyScene(s); return rc; }
    *out = s;
    return CGRT_OK;
}

void cgrt_scene_destroy(cgrt_scene* s) { destroyScene(s); }

int cgrt_scene_set_lights(cgrt_scene* s, const cgrt_point_light* lights, int32_t n)
{
    if (!s || n < 0 || (n > 0 && !lights)) return fail(CGRT_ERR_INVALID, "bad lights");
    std::lock_guard<std::mutex> lk(s->mu);
    s->lights.assign(lights, lights + n);
    return CGRT_OK;
}

int cgrt_scene_set_spherical_lights(cgrt_scene* s, const float* lights, int32_t n, uint32_t seed)
{
    if (!s || n < 0 || n > 64 || (n > 0 && !lights)) return fail(CGRT_ERR_INVALID, "bad spherical lights");
    std::lock_guard<std::mutex> lk(s->mu);
    s->sphLights.assign(lights, lights + (size_t)n * 7);
    s->softSeed = seed;
    return CGRT_OK;
}

int cgrt_scene_set_spheres(cgrt_scene* s, const float* spheres, int32_t n)
{
    if (!s || n < 0 || (n > 0 && !spheres)) return fail(CGRT_ERR_INVALID, "bad spheres");
    std::lock_guard<std::mutex> lk(s->mu);
    std::lock_guard<std::mutex> lk2(s->devMu);
    int rc = useSceneDevice(s);
    if (rc) return rc;
    CK(cudaDeviceSynchronize());
    return uploadSpheres(s, spheres, n);
}

int cgrt_bvh_num_levels(const cgrt_scene* s) { return s ? s->bvh.numLevels : 0; }
int cgrt_bvh_num_nodes(const cgrt_scene* s) { return s ? (int)s->bvh.nodes.size() : 0; }
int64_t cgrt_scene_num_triangles(const cgrt_scene* s) { return s ? s->nTris : 0; }

int cgrt_bvh_export_nodes(const cgrt_scene* s, int32_t* meta, float* aabb)
{
    if (!s || !meta || !aabb) return fail(CGRT_ERR_INVALID, "null argument");
    for (size_t i = 0; i < s->bvh.nodes.size(); i++) {
        const HostNode& n = s->bvh.nodes[i];
        meta[5 * i + 0] = n.isLeaf;
        meta[5 * i + 1] = n.level;
        meta[5 * i + 2] = n.child0;
        meta[5 * i + 3] = n.child1;
        meta[5 * i + 4] = n.isLeaf ? n.triCount : 0;
        for (int k = 0; k < 3; k++) {
            aabb[6 * i + k] = n.lo[k];
            aabb[6 * i + 3 + k] = n.hi[k];
        }
    }
    return CGRT_OK;
}

int cgrt_bvh_leaf_triangles(const cgrt_scene* s, int32_t node, int32_t* out, int32_t cap)
{
    if (!s || node < 0 || node >= (int)s->bvh.nodes.size()) return -1;
    const HostNode& n = s->bvh.nodes[node];
    if (!n.isLeaf) return 0;
    for (int i = 0; i < n.triCount && i < cap; i++) out[i] = s->leafGlobalId[n.firstTri + i];
    return n.triCount;
}

// ---- batch queries -------------------------------------------------------------------------------------------------
int cgrt_intersect_closest_device(cgrt_scene* s, const cgrt_ray* d_rays, size_t n, cgrt_hit* d_hits, uint32_t* d_counts,
                                  void* stream)
{
    if (!s || (n && (!d_rays || !d_hits))) return fail(CGRT_ERR_INVALID, "null argument");
    int rc = useSceneDevice(s);
    if (rc) return rc;
    DevScene S;
    { // (the only shared state on the query path: a snapshot of the scene's pointer table, taken under the lock that
      // cgrt_scene_set_spheres holds while it replaces the sphere list; renders hold it for the enqueue of a frame)
        std::lock_guard<std::mutex> lk(s->devMu);
        S = s->dev;
    }
    launchClosestBatch(S, (const float4*)d_rays, n, (float4*)d_hits, d_counts, s->di.numSMs, (cudaStream_t)stream);
    CK(cudaGetLastError());
    return CGRT_OK;
}

int cgrt_intersect_any_device(cgrt_scene* s, const cgrt_ray* d_rays, const float* d_max_dist, float eps, size_t n,
                              uint8_t* d_occluded, void* stream)
{
    if (!s || (n && (!d_rays || !d_max_dist || !d_occluded))) return fail(CGRT_ERR_INVALID, "null argument");
    int rc = useSceneDevice(s);
    if (rc) return rc;
    DevScene S;
    {
        std::lock_guard<std::mutex> lk(s->devMu);
        S = s->dev;
    }
    launchAnyBatch(S, (const float4*)d_rays, d_max_dist, eps, n, d_occluded, s->di.numSMs, (cudaStream_t)stream);
    CK(cudaGetLastError());
    return CGRT_OK;
}

// Scratch of the host-pointer query forms: per HOST THREAD and device, kept between calls - a stream and three growable device
// buffers. The reference's intersect() is called concurrently from every OpenMP thread (src/main.cpp:653-656 -> :276, :115):
// here the threads share nothing on the query path (no scene-wide lock, no per-call cudaMalloc / cudaFree - cudaFree
// synchronises the whole device - no stream creation), so their copies and kernels overlap on the device.
struct ThreadScratch {
    int device = -1;
    cudaStream_t st = nullptr;
    void* buf[3] = {nullptr, nullptr, nullptr};
    size_t cap[3] = {0, 0, 0};
    ~ThreadScratch() { release(); }
    void release()
    {
        if (device < 0) return;
        if (cudaSetDevice(device) == cudaSuccess) { // (at thread exit the context may already be gone: errors are ignored)
            for (int k = 0; k < 3; k++)
                if (buf[k]) cudaFree(buf[k]);
            if (st) cudaStreamDestroy(st);
        }
        cudaGetLastError();
        for (int k = 0; k < 3; k++) { buf[k] = nullptr; cap[k] = 0; }
        st = nullptr;
        device = -1;
    }
    int use(int dev)
    {
        if (device == dev && st) return CGRT_OK;
        release();
        CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        device = dev;
        return CGRT_OK;
    }
    int get(int k, size_t bytes, void** out)
    {
        if (bytes > cap[k]) {
            if (buf[k]) CK(cudaFree(buf[k]));
            buf[k] = nullptr;
            cap[k] = 0;
            const size_t want = std::max(bytes + bytes / 4, (size_t)4096);
            cudaError_t e = cudaMalloc(&buf[k], want);
            if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? CGRT_ERR_OOM : CGRT_ERR_CUDA,
                                              std::string("cudaMalloc failed: ") + cudaGetErrorString(e));
            cap[k] = want;
        }
        *out = buf[k];
        return CGRT_OK;
    }
};
static thread_local ThreadScratch g_scratch;

// scratch helper for the remaining host-pointer forms (brute force, unit predicates): freed on scope exit
struct Scratch {
    std::vector<void*> ptrs;
    cudaStream_t st = nullptr;
    ~Scratch()
    {
        for (void* p : ptrs) cudaFree(p);
        if (st) cudaStreamDestroy(st);
    }
    int alloc(void** p, size_t bytes)
    {
        cudaError_t e = cudaMalloc(p, bytes ? bytes : 1);
        if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? CGRT_ERR_OOM : CGRT_ERR_CUDA,
                                          std::string("cudaMalloc failed: ") + cudaGetErrorString(e));
        ptrs.push_back(*p);
        return CGRT_OK;
    }
    int stream()
    {
        CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        return CGRT_OK;
    }
};
#define RC(x)              \
    do {                   \
        int rc_ = (x);     \
        if (rc_) return rc_; \
    } while (0)

int cgrt_intersect_closest(cgrt_scene* s, const cgrt_ray* rays, size_t n, cgrt_hit* hits, uint32_t* counts)
{
    if (!s || (n && (!rays || !hits))) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useSceneDevice(s));
    if (n == 0) return CGRT_OK;
    ThreadScratch& sc = g_scratch;
    RC(sc.use(s->device));
    void *dR, *dH, *dC = nullptr;
    RC(sc.get(0, n * sizeof(cgrt_ray), &dR));
    RC(sc.get(1, n * sizeof(cgrt_hit), &dH));
    if (counts) RC(sc.get(2, n * 2 * sizeof(uint32_t), &dC));
    CK(cudaMemcpyAsync(dR, rays, n * sizeof(cgrt_ray), cudaMemcpyHostToDevice, sc.st));
    RC(cgrt_intersect_closest_device(s, (const cgrt_ray*)dR, n, (cgrt_hit*)dH, (uint32_t*)dC, sc.st));
    CK(cudaMemcpyAsync(hits, dH, n * sizeof(cgrt_hit), cudaMemcpyDeviceToHost, sc.st));
    if (counts) CK(cudaMemcpyAsync(counts, dC, n * 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, sc.st));
    CK(cudaStreamSynchronize(sc.st));
    return CGRT_OK;
}

int cgrt_intersect_any(cgrt_scene* s, const cgrt_ray* rays, const float* max_dist, float eps, size_t n, uint8_t* occluded)
{
    if (!s || (n && (!rays || !max_dist || !occluded))) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useSceneDevice(s));
    if (n == 0) return CGRT_OK;
    ThreadScratch& sc = g_scratch;
    RC(sc.use(s->device));
    void *dR, *dM, *dO;
    RC(sc.get(0, n * sizeof(cgrt_ray), &dR));
    RC(sc.get(1, n * sizeof(float), &dM));
    RC(sc.get(2, n, &dO));
    CK(cudaMemcpyAsync(dR, rays, n * sizeof(cgrt_ray), cudaMemcpyHostToDevice, sc.st));
    CK(cudaMemcpyAsync(dM, max_dist, n * sizeof(float), cudaMemcpyHostToDevice, sc.st));
    RC(cgrt_intersect_any_device(s, (const cgrt_ray*)dR, (const float*)dM, eps, n, (uint8_t*)dO, sc.st));
    CK(cudaMemcpyAsync(occluded, dO, n, cudaMemcpyDeviceToHost, sc.st));
    CK(cudaStreamSynchronize(sc.st));
    return CGRT_OK;
}

int cgrt_intersect_brute(cgrt_scene* s, const cgrt_ray* rays, size_t n, cgrt_hit* hits)
{
    if (!s || (n && (!rays || !hits))) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useSceneDevice(s));
    if (n == 0) return CGRT_OK;
    Scratch sc;
    RC(sc.stream());
    void *dR, *dH;
    RC(sc.alloc(&dR, n * sizeof(cgrt_ray)));
    RC(sc.alloc(&dH, n * sizeof(cgrt_hit)));
    CK(cudaMemcpyAsync(dR, rays, n * sizeof(cgrt_ray), cudaMemcpyHostToDevice, sc.st));
    DevScene S;
    {
        std::lock_guard<std::mutex> lk(s->mu);
        S = s->dev;
    }
    launchBruteBatch(S, (const float4*)dR, n, (float4*)dH, s->di.numSMs, sc.st);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(hits, dH, n * sizeof(cgrt_hit), cudaMemcpyDeviceToHost, sc.st));
    CK(cudaStreamSynchronize(sc.st));
    return CGRT_OK;
}

// ---- unit predicates -------------------------------------------------------------------------------------------------
struct UnitIO {
    Scratch sc;
    int in(void** d, const void* h, size_t bytes)
    {
        RC(sc.alloc(d, bytes));
        CK(cudaMemcpyAsync(*d, h, bytes, cudaMemcpyHostToDevice, sc.st));
        return CGRT_OK;
    }
    int out(void* h, const void* d, size_t bytes)
    {
        CK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, sc.st));
        return CGRT_OK;
    }
    int finish()
    {
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(sc.st));
        return CGRT_OK;
    }
};

int cgrt_ray_aabb(int device, const float* boxes, const cgrt_ray* rays, size_t n, uint8_t* hit, float* t)
{
    if (n && (!boxes || !rays || !hit || !t)) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useDevice(device));
    if (!n) return CGRT_OK;
    UnitIO io;
    RC(io.sc.stream());
    void *dB, *dR, *dH, *dT;
    RC(io.in(&dB, boxes, n * 24));
    RC(io.in(&dR, rays, n * 32));
    RC(io.sc.alloc(&dH, n));
    RC(io.sc.alloc(&dT, n * 4));
    launchUnitAabb((const float*)dB, (const float4*)dR, n, (uint8_t*)dH, (float*)dT, io.sc.st);
    RC(io.out(hit, dH, n));
    RC(io.out(t, dT, n * 4));
    return io.finish();
}

int cgrt_ray_triangle(int device, const float* tris, const cgrt_ray* rays, size_t n, cgrt_hit* out)
{
    if (n && (!tris || !rays || !out)) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useDevice(device));
    if (!n) return CGRT_OK;
    UnitIO io;
    RC(io.sc.stream());
    void *dT, *dR, *dO;
    RC(io.in(&dT, tris, n * 72));
    RC(io.in(&dR, rays, n * 32));
    RC(io.sc.alloc(&dO, n * 32));
    launchUnitTriangle((const float*)dT, (const float4*)dR, n, (float4*)dO, io.sc.st);
    RC(io.out(out, dO, n * 32));
    return io.finish();
}

int cgrt_ray_plane(int device, const float* planes, const cgrt_ray* rays, size_t n, uint8_t* hit, float* t)
{
    if (n && (!planes || !rays || !hit || !t)) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useDevice(device));
    if (!n) return CGRT_OK;
    UnitIO io;
    RC(io.sc.stream());
    void *dP, *dR, *dH, *dT;
    RC(io.in(&dP, planes, n * 16));
    RC(io.in(&dR, rays, n * 32));
    RC(io.sc.alloc(&dH, n));
    RC(io.sc.alloc(&dT, n * 4));
    launchUnitPlane((const float4*)dP, (const float4*)dR, n, (uint8_t*)dH, (float*)dT, io.sc.st);
    RC(io.out(hit, dH, n));
    RC(io.out(t, dT, n * 4));
    return io.finish();
}

int cgrt_triangle_plane(int device, const float* tris, size_t n, float* planes)
{
    if (n && (!tris || !planes)) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useDevice(device));
    if (!n) return CGRT_OK;
    UnitIO io;
    RC(io.sc.stream());
    void *dT, *dP;
    RC(io.in(&dT, tris, n * 36));
    RC(io.sc.alloc(&dP, n * 16));
    launchUnitTrianglePlane((const float*)dT, n, (float4*)dP, io.sc.st);
    RC(io.out(planes, dP, n * 16));
    return io.finish();
}

int cgrt_point_in_triangle(int device, const float* in, size_t n, uint8_t* inside)
{
    if (n && (!in || !inside)) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useDevice(device));
    if (!n) return CGRT_OK;
    UnitIO io;
    RC(io.sc.stream());
    void *dI, *dO;
    RC(io.in(&dI, in, n * 60));
    RC(io.sc.alloc(&dO, n));
    launchUnitPointInTriangle((const float*)dI, n, (uint8_t*)dO, io.sc.st);
    RC(io.out(inside, dO, n));
    return io.finish();
}

int cgrt_ray_sphere(int device, const float* spheres, const cgrt_ray* rays, size_t n, float* out)
{
    if (n && (!spheres || !rays || !out)) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useDevice(device));
    if (!n) return CGRT_OK;
    UnitIO io;
    RC(io.sc.stream());
    void *dS, *dR, *dO;
    RC(io.in(&dS, spheres, n * 16));
    RC(io.in(&dR, rays, n * 32));
    RC(io.sc.alloc(&dO, n * 20));
    launchUnitSphere((const float4*)dS, (const float4*)dR, n, (float*)dO, io.sc.st);
    RC(io.out(out, dO, n * 20));
    return io.finish();
}

int cgrt_generate_rays(int device, const cgrt_camera* cam, int32_t width, int32_t height, cgrt_ray* rays)
{
    if (!cam || !rays || width <= 0 || height <= 0) return fail(CGRT_ERR_INVALID, "bad argument");
    RC(useDevice(device));
    FrameParams P;
    std::memset(&P, 0, sizeof P);
    cameraConstants(*cam, P);
    P.width = width;
    P.height = height;
    UnitIO io;
    RC(io.sc.stream());
    void *dP, *dR;
    RC(io.in(&dP, &P, sizeof P));
    const size_t n = (size_t)width * height;
    RC(io.sc.alloc(&dR, n * 32));
    launchGenerateRays((const FrameParams*)dP, (int)n, (float4*)dR, io.sc.st);
    RC(io.out(rays, dR, n * 32));
    return io.finish();
}

// ---- rendering -----------------------------------------------------------------------------------------------------
size_t cgrt_tile_buffer_floats(const cgrt_render_params* p)
{
    if (checkRenderParams(p)) return 0;
    if (p->world == 1) return (size_t)p->width * p->height * 3;
    TileLayout L;
    makeTileLayout(*p, L);
    return (size_t)L.maxTiles * L.tileW * L.tileH * 3;
}

int cgrt_tile_list(const cgrt_render_params* p, int32_t rank, int32_t* out, int32_t cap)
{
    if (checkRenderParams(p) || rank < 0 || rank >= p->world) return -1;
    TileLayout L;
    makeTileLayout(*p, L);
    const std::vector<int>& l = L.lists[rank];
    for (size_t i = 0; i < l.size() && (int32_t)i < cap; i++) out[i] = l[i];
    return (int)l.size();
}

// the round pipeline needs the fast tree and lit-flag indices that fit the ray record's 30 bits
static bool useRounds(const cgrt_scene* s, const FrameParams& P)
{
    if (s->dev.fastRoot == 0u) return false;
    const uint64_t flags = (uint64_t)std::max(P.nSlots, 1) * (uint64_t)std::max(P.traceLimit, 1) * (uint64_t)std::max(P.nLights, 1);
    return flags < ((uint64_t)1 << 30);
}

// Two pipelines render the same frame bit for bit; which one runs is a question of speed only (CGRT_PIPELINE=wave|rounds forces
// one for A/B runs). The persistent wavefront (k_wave, one kernel per frame, levels overlapped) wins where the frame is a chain
// of dependent levels or small: trace limit >= 3, or a share of fewer than 400 K pixel slots (C3 1080p 1.35 vs 1.40 ms, its 1/8
// share 0.50 vs 0.75 ms, C1 0.13 vs 0.17 ms). The round pipeline (one flat kernel per level) wins on large shallow frames whose
// cost is streaming pixels and finishing many cheap rays (C2 1080p limit 1: 0.31 vs 0.40 ms; C5 2160p limit 2: 0.89 vs 1.25 ms).
static bool useWave(const cgrt_scene* s, const FrameParams& P)
{
    static int pref = -1; // 0 rounds, 1 wave, 2 automatic
    if (pref < 0) {
        const char* e = getenv("CGRT_PIPELINE");
        pref = (e && std::strcmp(e, "rounds") == 0) ? 0 : ((e && std::strcmp(e, "wave") == 0) ? 1 : 2);
    }
    if (pref == 0 || !useRounds(s, P) || P.nSlots >= (1 << 26) || P.traceLimit > 16) return false; // ray record: level << 26 | slot
    if (P.nSph > 0) return false; // spherical-light soft shadows are a pass of the round pipeline (before its shading kernel)
    // (shares of a multi-GPU frame: the one-launch form also wins on shallow frames up to ~2 M slots per rank - C2 on 4 GPUs
    // 0.23 vs 0.37 ms, C5 on 4 GPUs 0.58 vs 0.64 ms - where the round pipeline's per-launch floors no longer shrink with the share)
    return pref == 1 || P.traceLimit >= 3 || P.nSlots < 400000 || (P.world > 1 && P.nSlots < 2500000);
}

// the one decision of which kernel set renders a frame: the counting wavefront when asked for, else the fastest the scene and
// the frame allow
static FramePipeline choosePipeline(const cgrt_scene* s, const FrameParams& P, int flags)
{
    if (flags & CGRT_RENDER_COUNT) return PIPE_COUNT;
    if (useWave(s, P)) return PIPE_WAVE;
    return useRounds(s, P) ? PIPE_ROUNDS : PIPE_PATHS;
}
// pipelines that keep hit records and depths per pixel slot (what the overlapped delivery of cgrt_render needs)
static bool hasSlotRecords(FramePipeline pipe) { return pipe == PIPE_ROUNDS || pipe == PIPE_WAVE; }
// independent sub-frames of the last frame, each with its own CGRT_CNT_TOTAL counters
static int chainsOf(const cgrt_scene* s) { return s->lastPipeline == PIPE_ROUNDS ? s->lastChains : 1; }
// tickets the queue must hold: every slot can cast one closest-hit ray and one shadow ray per light at every level; plus the
// tickets idle lanes hold beyond the last ray (one per resident lane at most)
static size_t waveTicketCap(const FrameParams& P)
{
    return (size_t)std::max(P.nSlots, 1) * std::max(P.traceLimit, 1) * (1 + (size_t)std::max(P.nLights, 0)) + ((size_t)1 << 19) +
           (size_t)waveGridBlocks(1) * 128 * 160; // + the second records of rays handed over at the change-over (one per lane, <= 160 SMs)
}

// harvest the frames that have completed, then choose the setting of the next frame (see WaveTuner)
static int waveTunerChoose(WaveTuner& T, const int key[8], int start)
{
    if (std::memcmp(key, T.key, sizeof T.key) != 0) { // another frame shape: start over (events are kept)
        for (WaveTuner::Slot& sl : T.ring) sl.busy = false;
        std::memcpy(T.key, key, sizeof T.key);
        std::memset(T.ms, 0, sizeof T.ms);
        std::memset(T.pendingOf, 0, sizeof T.pendingOf);
        T.cur = std::min(std::max(start, (int)WaveTuner::LO), (int)WaveTuner::HI);
        T.frames = 0;
    }
    for (int k = 0; k < WaveTuner::RING; k++) { // oldest first; frames complete in order, so the first one still running ends the look
        WaveTuner::Slot& sl = T.ring[(T.next + k) % WaveTuner::RING];
        if (!sl.busy) continue;
        if (cudaEventQuery(sl.b) != cudaSuccess) break;
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, sl.a, sl.b) == cudaSuccess && ms > 0.0f)
            T.ms[sl.setting] = T.ms[sl.setting] == 0.0f ? ms : std::min(T.ms[sl.setting], ms);
        T.pendingOf[sl.setting]--;
        sl.busy = false;
    }
    (void)cudaGetLastError(); // (cudaErrorNotReady of the queries is not an error)
    T.frames++;
    if ((T.frames & 255) == 0) { // look at the neighbours again now and then (the camera or the lights may have moved)
        for (int f = WaveTuner::LO; f <= WaveTuner::HI; f++) if (f != T.cur) T.ms[f] = 0.0f;
        T.ms[T.cur] *= 1.05f;
    }
    const int c = T.cur;
    if (T.frames <= 2 || T.ms[c] == 0.0f) return c; // (the first frame of a shape pays for allocations and cold caches)
    for (int f : {c - 1, c + 1}) {
        if (f < WaveTuner::LO || f > WaveTuner::HI) continue;
        if (T.ms[f] == 0.0f) return T.pendingOf[f] > 0 ? c : f; // try it once; while that frame is in flight, carry on
    }
    int best = c;
    for (int f : {c - 1, c + 1})
        if (f >= WaveTuner::LO && f <= WaveTuner::HI && T.ms[f] < 0.98f * T.ms[best]) best = f;
    T.cur = best;
    return best;
}
static int waveTunerBegin(WaveTuner& T, int setting, cudaStream_t st)
{
    T.recording = -1;
    for (int k = 0; k < WaveTuner::RING; k++) {
        WaveTuner::Slot& sl = T.ring[(T.next + k) % WaveTuner::RING];
        if (sl.busy) continue;
        if (!sl.a && (cudaEventCreate(&sl.a) != cudaSuccess || cudaEventCreate(&sl.b) != cudaSuccess)) return 0;
        sl.setting = setting;
        if (cudaEventRecord(sl.a, st) != cudaSuccess) return 0;
        T.recording = (T.next + k) % WaveTuner::RING;
        T.next = (T.recording + 1) % WaveTuner::RING;
        return 1;
    }
    return 0; // every slot still in flight: this frame is not timed
}
static void waveTunerEnd(WaveTuner& T, cudaStream_t st)
{
    if (T.recording < 0) return;
    WaveTuner::Slot& sl = T.ring[T.recording];
    if (cudaEventRecord(sl.b, st) == cudaSuccess) {
        sl.busy = true;
        T.pendingOf[sl.setting]++;
    }
    T.recording = -1;
}

// scheduling knobs / watchdog of the persistent wavefront (CGRT_WAVE="mode=0,group_below=400000,switch=0,fin=0,tune=1,handover=1,timeout_ms=4000"; 0 = automatic; they
// change speed only, never results). mode 0: the search form follows the size of this rank's share of the frame - one lane per
// ray for large shares (throughput), eight lanes per ray for small ones (latency)
static bool waveTuning(WaveQ& Q, int nSlots, int nLights, int world)
{
    static int mode = 0, groupBelow = 400000, fin = 0, timeoutMs = 4000, switchBelow = 0, handOver = 1, tune = 1;
    static bool loaded = false;
    if (!loaded) {
        loaded = true;
        if (const char* e = getenv("CGRT_WAVE")) {
            std::string t(e);
            size_t pos = 0;
            while (pos < t.size()) {
                size_t c = t.find(',', pos);
                if (c == std::string::npos) c = t.size();
                const std::string kv = t.substr(pos, c - pos);
                const size_t eq = kv.find('=');
                if (eq != std::string::npos) {
                    const std::string key = kv.substr(0, eq);
                    const int v = atoi(kv.c_str() + eq + 1);
                    if (key == "mode") mode = v;
                    else if (key == "group_below") groupBelow = v;
                    else if (key == "fin") fin = v;
                    else if (key == "switch") switchBelow = v;
                    else if (key == "timeout_ms") timeoutMs = v;
                    else if (key == "handover") handOver = v;
                    else if (key == "tune") tune = v;
                }
                pos = c + 1;
            }
        }
    }
    Q.mode = mode == 1 || mode == 2 ? mode : (nSlots < groupBelow ? 2 : 1);
    // share of the SMs that run the finish warps: every hit costs one hit epilogue plus one shadow ray to emit and to finish per
    // light (measured with the two-stage certificates, profiles/r02_tuning.md: C3, 1 light: 1/6 of the SMs, 1/8 for the
    // GROUP-only share of C3 - but 1/5 for the Cornell box, and too few finishers cost more than too many; 3 lights: 1/4).
    // This is the STARTING value: WaveTuner moves it by measurement
    // (shares of a multi-GPU frame are rendered back to back, where the tuner gets no samples: small C3 shares want 1/8-1/9)
    Q.finEvery = fin > 0 ? std::max(fin, 2) : (nLights >= 3 ? 4 : (nLights == 2 ? 5 : (Q.mode == 2 && world > 1 ? 8 : 6)));
    // (GROUP-only frames never change over; measured on the C3 frame and its 1/2, 1/4 shares: 100 K in flight for a whole 1080p
    // frame, 60 K for smaller shares)
    Q.switchBelow = Q.mode == 2 ? 0 : (switchBelow > 0 ? switchBelow : (nSlots >= 1500000 ? 100000 : 60000));
    Q.timeoutNs = (unsigned long long)std::max(timeoutMs, 1) * 1000000ull;
    if (!handOver) Q.resume = nullptr; // rays finish in the search form they started in
    return fin <= 0 && tune != 0;      // the finisher share may be tuned by measurement (WaveTuner)
}

// A frame of nViews cameras (cgrt_render_views) is one frame of nViews x the one-view pixel slots: the tile sequence and
// primaryPixels stay those of one view, everything sized from P.nSlots grows with the views.
static int prepareFrame(cgrt_scene* s, const cgrt_camera* cams, int nViews, const cgrt_render_params* p, FrameParams& P,
                        const int** dTileList, const int2** dTileSeq, FramePipeline* pipe)
{
    const int tw = p->tile_w > 0 ? p->tile_w : 8, th = p->tile_h > 0 ? p->tile_h : 8;
    const int key[6] = {p->width, p->height, tw, th, p->world, p->rank};
    if (std::memcmp(key, s->tileKey, sizeof key) != 0 || !s->tileSeq.p) {
        TileLayout& L = s->layout;
        makeTileLayout(*p, L);
        const std::vector<int>& mine = L.lists[p->rank];
        // processing order: tiles sorted by the distance of their centre from the image centre. Scenes are normalised around
        // the look-at point (mesh.cpp:143-166), so the object - and with it every long mirror chain - projects to the middle
        // of the frame: those paths start first, the border tiles whose rays miss the root box fill the end of the launch.
        std::vector<int2> seq(mine.size());
        std::vector<std::pair<float, int>> order(mine.size());
        s->primaryPixels = 0;
        for (size_t lt = 0; lt < mine.size(); lt++) {
            const int ty = mine[lt] / L.tilesX, tx = mine[lt] % L.tilesX;
            const float cx = (tx + 0.5f) * L.tileW - 0.5f * p->width, cy = (ty + 0.5f) * L.tileH - 0.5f * p->height;
            order[lt] = std::make_pair(cx * cx + cy * cy, (int)lt);
            const int w = std::min(L.tileW, p->width - tx * L.tileW), h = std::min(L.tileH, p->height - ty * L.tileH);
            s->primaryPixels += (uint64_t)w * h;
        }
        std::sort(order.begin(), order.end());
        for (size_t k = 0; k < order.size(); k++) seq[k] = make_int2(mine[order[k].second], order[k].second);
        RC(s->tileList.ensure(std::max<size_t>(mine.size(), 1)));
        RC(s->tileSeq.ensure(std::max<size_t>(mine.size(), 1)));
        CK(cudaDeviceSynchronize()); // a previous frame may still read the old lists
        if (!mine.empty()) {
            CK(cudaMemcpy(s->tileList.p, mine.data(), mine.size() * sizeof(int), cudaMemcpyHostToDevice));
            CK(cudaMemcpy(s->tileSeq.p, seq.data(), seq.size() * sizeof(int2), cudaMemcpyHostToDevice));
        }
        CK(uploadsDone());
        std::memcpy(s->tileKey, key, sizeof key);
    }
    const TileLayout& L = s->layout;
    std::memset(&P, 0, sizeof P);
    cameraConstants(cams[0], P);
    P.nViews = nViews;
    P.width = p->width;
    P.height = p->height;
    P.nLights = (int)s->lights.size();
    P.nSph = (int)(s->sphLights.size() / 7);
    P.traceLimit = p->trace_limit;
    P.tileW = L.tileW;
    P.tileH = L.tileH;
    P.tilesX = L.tilesX;
    P.world = L.world;
    P.rank = p->rank;
    P.screenLayout = (L.world == 1 || (p->flags & CGRT_RENDER_SCREEN_LAYOUT)) ? 1 : 0;
    // pixel slots count whole tiles: thin frames with large tiles have many more slots than pixels
    const int64_t slots = (int64_t)nViews * (int64_t)L.lists[p->rank].size() * L.tileW * L.tileH;
    if (slots > INT_MAX) return fail(CGRT_ERR_INVALID, "too many pixel slots: views x tiles x tile pixels must stay below 2^31");
    P.nSlots = (int)slots;
    *dTileList = L.world > 1 ? s->tileList.p : nullptr;
    *dTileSeq = s->tileSeq.p;
    // queues sized for the worst case (every pixel hits, every hit bounces); only the used prefix is touched
    const size_t cap = (size_t)std::max(P.nSlots, 1);
    const int nL = std::max(P.nLights, 1);
    const int levels = std::max(P.traceLimit - 1, 1);
    const int pathLevels = std::max(P.traceLimit, 1);
    if (P.nSph > 0 && !useRounds(s, P)) return fail(CGRT_ERR_INVALID, "spherical lights need a scene with a search tree (not CGRT_SCENE_EXACT_ONLY / NO_SUBTREES)");
    *pipe = choosePipeline(s, P, p->flags);
    if (*pipe != PIPE_COUNT) { // hit records indexed by (pixel slot or path, level)
        RC(s->hitRec.ensure(cap * pathLevels * 3));
        RC(s->pathDepth.ensure(cap));
        RC(s->lit.ensure(cap * pathLevels * nL));
    }
    switch (*pipe) {
    case PIPE_COUNT: // level-by-level counting wavefront
        RC(s->hitQ.ensure(cap * 3));
        RC(s->bounceQ.ensure(cap * 2));
        RC(s->lit.ensure(cap * nL));
        RC(s->pathState.ensure(cap * 2 * levels));
        break;
    case PIPE_WAVE: { // persistent wavefront: one ticket-indexed ray array
        const size_t tickets = waveTicketCap(P);
        if (tickets >= ((size_t)1 << 30)) return fail(CGRT_ERR_INVALID, "frame too large for the ray queue's 30-bit tickets");
        if (!s->waveRays.p || s->waveRays.n < tickets * 3) { // (the records' tags compare against waveSeq >= 1: start from zero)
            RC(s->waveRays.ensure(tickets * 3));
            CK(cudaMemset(s->waveRays.p, 0, tickets * 3 * sizeof(float4)));
            RC(s->waveFin.ensure(tickets * 2));
            CK(cudaMemset(s->waveFin.p, 0, tickets * 2 * sizeof(float4)));
            CK(uploadsDone());
        }
        RC(s->waveCtl.ensure(WCTL_INTS));
        RC(s->waveResume.ensure((size_t)waveGridBlocks(s->di.numSMs) * 128 * WAVE_RESUME_F4));
        break;
    }
    case PIPE_ROUNDS: { // round pipeline: two ray lists per kind
        if (P.nSph > 0) {
            RC(s->softList.ensure(cap * pathLevels + 1));
            RC(s->soft.ensure(cap * pathLevels * (size_t)P.nSph));
        }
        const size_t capR = cap + (size_t)CGRT_MAX_CHAINS * P.tileW * P.tileH; // per-chain rounding to whole tiles
        for (int k = 0; k < 2; k++) {
            RC(s->cRay[k].ensure(capR * 3));
            RC(s->cRes[k].ensure(capR));
            RC(s->sRay[k].ensure(capR * nL * 3));
            RC(s->sRes[k].ensure(capR * nL));
        }
        break;
    }
    case PIPE_PATHS: // path pipeline: compacted list of the records
        RC(s->hitList.ensure(cap * pathLevels));
        if (s->dev.fastRoot != 0u) { // replay queues of the speculative kernels
            RC(s->replayQ.ensure(cap * 3));
            RC(s->replayShadow.ensure(cap * pathLevels * nL));
        }
        break;
    }
    RC(s->pathPix.ensure(cap));
    RC(s->counts.ensure(CGRT_CNT_TOTAL * CGRT_MAX_CHAINS));
    RC(s->tests.ensure(6));
    // parameter block: FrameParams header + lights (2 x float4 each) + cameras (CGRT_VIEW_F4 x float4 each)
    const size_t need = CGRT_PARAM_BLOCK_HEADER + ((size_t)nL + (size_t)P.nSph) * 32 + (size_t)nViews * CGRT_VIEW_F4 * 16;
    if (need > s->paramBlockBytes || !s->hParamRing) {
        CK(cudaDeviceSynchronize());
        if (s->hParamRing) cudaFreeHost(s->hParamRing);
        s->hParamRing = nullptr;
        s->paramBlockBytes = std::max(need, (size_t)CGRT_PARAM_BLOCK_HEADER + 16 * 32);
        CK(cudaMallocHost((void**)&s->hParamRing, s->paramBlockBytes * cgrt_scene::RING));
        RC(s->dParamBlock.ensure(s->paramBlockBytes));
    }
    return CGRT_OK;
}

static_assert(sizeof(FrameParams) <= CGRT_PARAM_BLOCK_HEADER, "FrameParams must fit the parameter block header");

int cgrt_bvh_fast_tree_stats(const cgrt_scene* s, int64_t* out)
{
    if (!s || !out) return fail(CGRT_ERR_INVALID, "null argument");
    for (int k = 0; k < 8; k++) out[k] = s->fastStats[k];
    return CGRT_OK;
}

// ---- each pipeline's view of the scene's frame buffers (sized by prepareFrame) ---------------------------------------------------
static CountBuffers countBuffers(const cgrt_scene* s, const FrameParams& P)
{
    CountBuffers B;
    B.hitQ = s->hitQ.p;
    B.bounceQ = s->bounceQ.p;
    B.lit = s->lit.p;
    B.pathPix = s->pathPix.p;
    B.pathState = s->pathState.p;
    B.counts = s->counts.p;
    B.tests = s->tests.p;
    B.cap = (size_t)std::max(P.nSlots, 1);
    return B;
}

static PathBuffers pathBuffers(const cgrt_scene* s, const FrameParams& P)
{
    PathBuffers B;
    B.hitRec = s->hitRec.p;
    B.hitList = s->hitList.p;
    B.lit = s->lit.p;
    B.pathPix = s->pathPix.p;
    B.pathDepth = s->pathDepth.p;
    B.replayQ = s->replayQ.p;
    B.replayShadow = s->replayShadow.p;
    B.counts = s->counts.p;
    B.cap = (size_t)std::max(P.nSlots, 1);
    B.levels = std::max(P.traceLimit, 1);
    return B;
}

// chain c of nChains: its own ray lists and counters, the frame's hit records
static RoundBuffers roundBuffers(const cgrt_scene* s, const FrameParams& P, int c, int nChains)
{
    const size_t tpx = (size_t)P.tileW * P.tileH;
    const size_t capC = ((size_t)std::max(P.nSlots, 1) / tpx / nChains + 1) * tpx; // slots one chain can own
    const size_t nLc = (size_t)std::max(P.nLights, 1);
    RoundBuffers B;
    for (int k = 0; k < 2; k++) {
        B.cRay[k] = s->cRay[k].p + c * capC * 3; B.cRes[k] = s->cRes[k].p + c * capC;
        B.sRay[k] = s->sRay[k].p + c * capC * nLc * 3; B.sRes[k] = s->sRes[k].p + c * capC * nLc;
    }
    B.hitRec = s->hitRec.p;
    B.lit = s->lit.p;
    B.pathDepth = s->pathDepth.p;
    B.counts = s->counts.p + c * CGRT_CNT_TOTAL;
    B.levels = std::max(P.traceLimit, 1);
    B.softList = s->softList.p;
    B.soft = s->soft.p;
    B.softSeed = s->softSeed;
    return B;
}

// k_wave's ray / finish queues (its records and counters are those of a one-chain round frame). Clears the optional
// diagnostics buffers on `st`.
static int waveQueues(cgrt_scene* s, cudaStream_t st, WaveQ& Q)
{
    Q.rays = s->waveRays.p;
    Q.fin = s->waveFin.p;
    Q.ctl = s->waveCtl.p;
    Q.seq = ++s->waveSeq;
    if (Q.seq == 0u) Q.seq = ++s->waveSeq;
    Q.cap = (int)std::min<size_t>(s->waveRays.n / 3, (size_t)0x3fffffff);
    Q.resume = s->waveResume.p;
    Q.resumeCap = (int)std::min<size_t>(s->waveResume.n / WAVE_RESUME_F4, (size_t)0xffffff);
    Q.lat = nullptr;
#ifdef CGRT_WAVE_LAT
    if (getenv("CGRT_WAVE_LAT")) {
        RC(s->waveLat.ensure((size_t)Q.cap * 16));
        CK(cudaMemsetAsync(s->waveLat.p, 0, (size_t)Q.cap * 16 * sizeof(unsigned), st));
        Q.lat = s->waveLat.p;
    }
#endif
    Q.trace = nullptr;
    if (getenv("CGRT_WAVE_TRACE") || Q.lat != nullptr) { // timeline of the frame's counters (cgrt_debug_wave_timeline); off by default
        RC(s->waveTrace.ensure((size_t)WAVE_TRACE_SAMPLES * 8));
        CK(cudaMemsetAsync(s->waveTrace.p, 0, (size_t)WAVE_TRACE_SAMPLES * 8 * sizeof(int), st));
        Q.trace = s->waveTrace.p;
    }
    return CGRT_OK;
}

// one frame of nViews cameras into d_out (cgrt_render_device: one camera; cgrt_render_views_device: several)
static int renderDevice(cgrt_scene* s, const cgrt_camera* cams, int nViews, const cgrt_render_params* p, float* d_out, void* stream)
{
    RC(useSceneDevice(s));
    std::lock_guard<std::mutex> lk(s->mu);
    cudaStream_t st = (cudaStream_t)stream;
    FrameParams P;
    const int* dTiles = nullptr;
    const int2* dSeq = nullptr;
    FramePipeline pipe;
    RC(prepareFrame(s, cams, nViews, p, P, &dTiles, &dSeq, &pipe));
    if (P.screenLayout && P.world > 1 && pipe == PIPE_COUNT)
        return fail(CGRT_ERR_INVALID, "CGRT_RENDER_COUNT renders into the tile-major buffer; it cannot be combined with CGRT_RENDER_SCREEN_LAYOUT");
    // per-frame upload (camera constants + lights, read live from the scene like src/main.cpp:835-876 allows)
    unsigned char* slot = s->hParamRing + (size_t)s->ringPos * s->paramBlockBytes;
    s->ringPos = (s->ringPos + 1) % cgrt_scene::RING;
    std::memcpy(slot, &P, sizeof P);
    float4* hl = (float4*)(slot + CGRT_PARAM_BLOCK_HEADER);
    for (size_t i = 0; i < s->lights.size(); i++) {
        const cgrt_point_light& l = s->lights[i];
        hl[2 * i] = make_float4(l.position[0], l.position[1], l.position[2], 0.0f);
        hl[2 * i + 1] = make_float4(l.color[0], l.color[1], l.color[2], 0.0f);
    }
    for (int i = 0; i < P.nSph; i++) { // spherical lights follow the point lights: [position | radius] [colour | -]
        const float* q = s->sphLights.data() + 7 * (size_t)i;
        hl[2 * (s->lights.size() + i)] = make_float4(q[0], q[1], q[2], q[3]);
        hl[2 * (s->lights.size() + i) + 1] = make_float4(q[4], q[5], q[6], 0.0f);
    }
    float4* hc = hl + 2 * (s->lights.size() + (size_t)P.nSph); // the views' cameras follow the lights
    for (int v = 0; v < nViews; v++) {
        FrameParams C;
        cameraConstants(cams[v], C);
        hc[CGRT_VIEW_F4 * v] = make_float4(C.camX, C.camY, C.camZ, C.halfW);
        hc[CGRT_VIEW_F4 * v + 1] = make_float4(C.qx, C.qy, C.qz, C.qw);
        hc[CGRT_VIEW_F4 * v + 2] = make_float4(C.halfH, 0.0f, 0.0f, 0.0f);
    }
    const size_t bytes = CGRT_PARAM_BLOCK_HEADER + (s->lights.size() + (size_t)P.nSph) * 32 + (size_t)nViews * CGRT_VIEW_F4 * 16;
    CK(cudaMemcpyAsync(s->dParamBlock.p, slot, bytes, cudaMemcpyHostToDevice, st));
    const int maxKernels = CGRT_TRACE_MAX_KERNELS;
    if ((p->flags & CGRT_RENDER_PROFILE_ALL) && s->traceEvents.empty()) {
        s->traceEvents.resize(2 * maxKernels);
        for (cudaEvent_t& e : s->traceEvents) CK(cudaEventCreate(&e));
    }
    std::memset(&s->trace, 0, sizeof s->trace);
    s->trace.ev = s->traceEvents.data();
    s->trace.maxKernels = maxKernels;
    s->trace.classMask = p->flags & CGRT_RENDER_PROFILE_ALL;
    const FrameParams* dP = (const FrameParams*)s->dParamBlock.p;
    const float4* dLights = (const float4*)(s->dParamBlock.p + CGRT_PARAM_BLOCK_HEADER);
    const int numSMs = s->di.numSMs;
    CK(cudaEventRecord(s->ev0, st));
    int launches = 0;
    switch (pipe) {
    case PIPE_COUNT:
        launches = launchCountingFrame(s->dev, dP, P, dLights, countBuffers(s, P), dTiles, d_out, numSMs, &s->trace, st);
        break;
    case PIPE_PATHS:
        launches = launchPathPipeline(s->dev, dP, P, dLights, pathBuffers(s, P), dSeq, d_out, numSMs, &s->trace, st);
        break;
    case PIPE_ROUNDS: {
        // chains: independent sub-frames (tiles dealt round-robin) on their own streams
        const int nChains = roundPipelineChains(P.nSlots);
        if (nChains > 1 && !s->chainSync.fork) {
            CK(cudaEventCreateWithFlags(&s->chainSync.fork, cudaEventDisableTiming));
            for (int c = 1; c < CGRT_MAX_CHAINS; c++) {
                CK(cudaStreamCreateWithFlags(&s->chainSync.streams[c], cudaStreamNonBlocking));
                CK(cudaEventCreateWithFlags(&s->chainSync.join[c], cudaEventDisableTiming));
            }
        }
        RoundBuffers RB[CGRT_MAX_CHAINS];
        for (int c = 0; c < nChains; c++) RB[c] = roundBuffers(s, P, c, nChains);
        launches = launchRoundPipeline(s->dev, dP, P, dLights, RB, nChains, s->chainSync, dSeq, d_out, numSMs, &s->trace, st);
        s->lastChains = nChains;
        break;
    }
    case PIPE_WAVE: {
        WaveQ Q;
        RC(waveQueues(s, st, Q));
        const bool tuned = waveTuning(Q, P.nSlots, P.nLights, P.world) && !(p->flags & CGRT_RENDER_PROFILE_ALL);
        if (tuned) {
            const int key[8] = {P.width, P.height, P.nSlots, P.traceLimit, P.nLights, P.world, P.rank, Q.mode};
            Q.finEvery = waveTunerChoose(s->tuner, key, Q.finEvery);
            waveTunerBegin(s->tuner, Q.finEvery, st);
        }
        launches = launchWavePipeline(s->dev, dP, P, dLights, roundBuffers(s, P, 0, 1), Q, dSeq, d_out, numSMs, &s->trace, st);
        if (tuned) waveTunerEnd(s->tuner, st);
        break;
    }
    }
    s->lastPipeline = pipe;
    CK(cudaEventRecord(s->ev1, st));
    CK(cudaGetLastError());
    s->lastStream = st;
    s->statsOnHost = false;
    s->lastLaunches = (uint64_t)launches;
    s->lastParams = P;
    s->haveLast = true;
    return CGRT_OK;
}

int cgrt_render_device(cgrt_scene* s, const cgrt_camera* cam, const cgrt_render_params* p, float* d_out, void* stream)
{
    if (!s || !cam || !d_out) return fail(CGRT_ERR_INVALID, "null argument");
    RC(checkRenderParams(p));
    return renderDevice(s, cam, 1, p, d_out, stream);
}

// the arguments cgrt_render_views refuses, checked before any CUDA call
static int checkViews(const cgrt_scene* s, const cgrt_camera* cams, int32_t nViews, const cgrt_render_params* p, const float* out)
{
    if (!s || !cams || !out) return fail(CGRT_ERR_INVALID, "null argument");
    RC(checkRenderParams(p));
    if (nViews < 1 || nViews > CGRT_MAX_VIEWS) return fail(CGRT_ERR_INVALID, "n_views must be in 1..1024");
    if ((int64_t)nViews * p->width * p->height > (int64_t)1 << 28) return fail(CGRT_ERR_INVALID, "views too large: n_views x width x height > 2^28");
    if (p->world != 1) return fail(CGRT_ERR_INVALID, "cgrt_render_views renders whole frames (world == 1)");
    if (p->flags & ~CGRT_RENDER_PROFILE_ALL) return fail(CGRT_ERR_INVALID, "cgrt_render_views takes the CGRT_RENDER_PROFILE_* flags only");
    // pixel slots of whole tiles (tile size as makeTileLayout picks it; prepareFrame checks the same total for every frame)
    const int64_t tw = p->tile_w > 0 ? p->tile_w : 8, th = p->tile_h > 0 ? p->tile_h : 8;
    if (nViews * ((p->width + tw - 1) / tw) * tw * ((p->height + th - 1) / th) * th > INT_MAX)
        return fail(CGRT_ERR_INVALID, "too many pixel slots: views x tiles x tile pixels must stay below 2^31");
    return CGRT_OK;
}

int cgrt_render_views_device(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p, float* d_out,
                             void* stream)
{
    RC(checkViews(s, cams, n_views, p, d_out));
    return renderDevice(s, cams, n_views, p, d_out, stream);
}

int cgrt_render_collect_stats(cgrt_scene* s, cgrt_render_stats* stats)
{
    if (!s || !stats) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useSceneDevice(s));
    std::lock_guard<std::mutex> lk(s->mu);
    std::memset(stats, 0, sizeof *stats);
    if (!s->haveLast) return fail(CGRT_ERR_INVALID, "no frame rendered yet");
    CK(cudaStreamSynchronize(s->lastStream));
    int counts[CGRT_CNT_TOTAL];
    const bool onHost = s->statsOnHost && s->hStats != nullptr;
    {
        const int nc = chainsOf(s);
        std::vector<int> all((size_t)CGRT_CNT_TOTAL * nc);
        if (onHost) std::memcpy(all.data(), s->hStats, all.size() * sizeof(int));
        else CK(cudaMemcpy(all.data(), s->counts.p, all.size() * sizeof(int), cudaMemcpyDeviceToHost));
        for (int k = 0; k < CGRT_CNT_TOTAL; k++) {
            counts[k] = 0;
            for (int c = 0; c < nc; c++) counts[k] += all[(size_t)c * CGRT_CNT_TOTAL + k];
        }
    }
    const FrameParams& P = s->lastParams;
    // logical rays (SURVEY.md §8(d)): primary = pixels of this rank inside the image, in every view
    const uint64_t primary = s->primaryPixels * (uint64_t)P.nViews;
    stats->primary = primary;
    if (s->lastPipeline == PIPE_WAVE) { // persistent wavefront: the watchdog of k_wave (a warp waited for seconds) invalidates the frame
        int err = 0;
        if (onHost) err = s->hStats[CGRT_CNT_TOTAL * CGRT_MAX_CHAINS];
        else CK(cudaMemcpy(&err, s->waveCtl.p + WCTL_ERR, sizeof(int), cudaMemcpyDeviceToHost));
        if (err) return fail(CGRT_ERR_CUDA, "k_wave watchdog: the persistent wavefront did not complete; the frame is invalid");
    }
    stats->pipeline = s->lastPipeline;
    if (hasSlotRecords(s->lastPipeline)) {
        stats->primary_hit = (uint64_t)counts[CGRT_CNT_PATHS];
        for (int l = 0; l < P.traceLimit; l++) {
            stats->shadow += (uint64_t)counts[CGRT_CNT_HIT + l] * (uint64_t)P.nLights;
            if (l >= 1) stats->bounce += (uint64_t)counts[CGRT_CNT_BOUNCE + l];
        }
        if (P.nSph > 0) { // 200 sample rays per hit record and spherical light (main.cpp:177)
            int nHits = 0;
            CK(cudaMemcpy(&nHits, s->softList.p + (size_t)std::max(P.nSlots, 1) * std::max(P.traceLimit, 1), sizeof(int), cudaMemcpyDeviceToHost));
            stats->shadow += 200ull * (uint64_t)nHits * (uint64_t)P.nSph;
        }
        stats->replayed_closest = (uint32_t)counts[CGRT_CNT_REPLAY_PATHS];
        stats->replayed_shadow = (uint32_t)counts[CGRT_CNT_REPLAY_SHADOW];
    } else if (s->lastPipeline == PIPE_PATHS) {
        stats->primary_hit = (uint64_t)counts[CGRT_CNT_PATHS];
        stats->shadow = (uint64_t)counts[CGRT_CNT_HITS] * (uint64_t)P.nLights;
        stats->bounce = (uint64_t)counts[CGRT_CNT_BOUNCES];
        stats->replayed_closest = (uint32_t)counts[CGRT_CNT_REPLAY_PATHS];
        stats->replayed_shadow = (uint32_t)counts[CGRT_CNT_REPLAY_SHADOW];
    } else { // PIPE_COUNT
        stats->primary_hit = (uint64_t)counts[CGRT_CNT_HIT + 0];
        for (int l = 0; l < P.traceLimit; l++) {
            stats->shadow += (uint64_t)counts[CGRT_CNT_HIT + l] * (uint64_t)P.nLights;
            if (l >= 1) stats->bounce += (uint64_t)counts[CGRT_CNT_BOUNCE + l];
        }
    }
    if (P.traceLimit == 0) stats->primary = 0;
    stats->kernel_launches = s->lastLaunches;
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    stats->device_ms = ms;
    for (int c = 0; c < 4; c++) stats->class_launches[c] = (uint32_t)s->trace.launches[c];
    // device time per kernel class = length of the UNION of its launches' intervals (launches of different chains overlap);
    // timestamps are taken relative to the frame's first event, which works across streams
    {
        std::vector<std::pair<float, float>> iv[4];
        for (int k = 0; k < s->trace.n; k++) {
            float t0 = 0.0f, t1 = 0.0f;
            CK(cudaEventElapsedTime(&t0, s->ev0, s->trace.ev[2 * k]));
            CK(cudaEventElapsedTime(&t1, s->ev0, s->trace.ev[2 * k + 1]));
            iv[s->trace.cls[k]].push_back(std::make_pair(t0, t1));
        }
        for (int c = 0; c < 4; c++) {
            std::sort(iv[c].begin(), iv[c].end());
            float total = 0.0f, curEnd = -1.0f, curBeg = 0.0f;
            bool open = false;
            for (const auto& x : iv[c]) {
                if (!open || x.first > curEnd) {
                    if (open) total += curEnd - curBeg;
                    curBeg = x.first;
                    curEnd = x.second;
                    open = true;
                } else if (x.second > curEnd) {
                    curEnd = x.second;
                }
            }
            if (open) total += curEnd - curBeg;
            stats->class_ms[c] = total;
        }
    }
    if (s->lastPipeline == PIPE_COUNT) {
        unsigned long long t[6];
        CK(cudaMemcpy(t, s->tests.p, sizeof t, cudaMemcpyDeviceToHost));
        for (int c = 0; c < 3; c++) {
            stats->box_tests[c] = t[2 * c];
            stats->tri_tests[c] = t[2 * c + 1];
        }
    }
    return CGRT_OK;
}

int cgrt_render(cgrt_scene* s, const cgrt_camera* cam, const cgrt_render_params* p, float* rgb, cgrt_render_stats* stats)
{
    if (!s || !cam || !rgb) return fail(CGRT_ERR_INVALID, "null argument");
    RC(checkRenderParams(p));
    RC(useSceneDevice(s));
    if (p->world > 1 && (p->flags & CGRT_RENDER_SCREEN_LAYOUT))
        return fail(CGRT_ERR_INVALID, "CGRT_RENDER_SCREEN_LAYOUT is a device-pointer mode (cgrt_render_device)");
    const size_t frameFloats = (size_t)p->width * p->height * 3;
    const size_t outFloats = cgrt_tile_buffer_floats(p);
    std::lock_guard<std::mutex> hostLock(s->hostMu);
    {
        std::lock_guard<std::mutex> lk(s->mu);
        RC(s->frame.ensure(std::max(frameFloats, outFloats)));
    }
    // Overlapped delivery (whole frame, page-locked destination, a pipeline that keeps pathDepth per pixel slot): the caller's
    // frame is blanked by a copy-engine transfer of zeros on a second stream WHILE the frame renders - most pixels of these
    // scenes are black - and the bounding box of the pixels the shading pass coloured is then written straight into it by a
    // small kernel (zero-copy stores in full 128-byte runs). The synchronous call costs the device time plus that last step instead of the device time plus a
    // 25 MB copy.
    float* dHost = nullptr;
    bool overlapped = false;
    if (p->world == 1 && p->trace_limit > 0 && s->dev.fastRoot != 0u && !(p->flags & CGRT_RENDER_COUNT) && !getenv("CGRT_PLAIN_D2H")) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, rgb) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer)
            dHost = (float*)at.devicePointer;
        else
            cudaGetLastError();
    }
    if (dHost) {
        std::lock_guard<std::mutex> lk(s->mu);
        if (!s->copyStream) {
            CK(cudaStreamCreateWithFlags(&s->copyStream, cudaStreamNonBlocking));
            for (int k = 0; k < 2; k++) {
                CK(cudaEventCreateWithFlags(&s->renderDone[k], cudaEventDisableTiming));
                CK(cudaEventCreateWithFlags(&s->copyDone[k], cudaEventDisableTiming));
            }
        }
        // (a copy-engine transfer: a memset kernel would queue behind the persistent render kernel, which owns every SM)
        if (!s->zeroFrame.p || s->zeroFrame.n < frameFloats) {
            RC(s->zeroFrame.ensure(frameFloats));
            CK(cudaMemset(s->zeroFrame.p, 0, frameFloats * sizeof(float)));
            CK(uploadsDone());
        }
        CK(cudaMemcpyAsync(rgb, s->zeroFrame.p, frameFloats * sizeof(float), cudaMemcpyDeviceToHost, s->copyStream));
        CK(cudaEventRecord(s->copyDone[0], s->copyStream));
        overlapped = true;
    }
    RC(cgrt_render_device(s, cam, p, s->frame.p, s->stream));
    if (overlapped && !hasSlotRecords(s->lastPipeline)) { // (path pipeline: no per-slot depth) plain copy after all
        CK(cudaStreamSynchronize(s->copyStream));
        overlapped = false;
    }
    if (overlapped) {
        CK(cudaStreamWaitEvent(s->stream, s->copyDone[0], 0));
        launchDeliverBox(s->counts.p + CGRT_CNT_BBOX, p->width, p->height, s->frame.p, dHost, s->di.numSMs, s->stream);
        CK(cudaGetLastError());
        bool fetched = false;
        if (stats) { // the statistics ride behind the frame: one synchronisation for both
            std::lock_guard<std::mutex> lk(s->mu);
            if (!s->hStats && cudaHostAlloc((void**)&s->hStats, sizeof(int) * (CGRT_CNT_TOTAL * CGRT_MAX_CHAINS + 1), cudaHostAllocDefault) != cudaSuccess) {
                s->hStats = nullptr;
                cudaGetLastError();
            }
            if (s->hStats) {
                CK(cudaMemcpyAsync(s->hStats, s->counts.p, sizeof(int) * CGRT_CNT_TOTAL * chainsOf(s), cudaMemcpyDeviceToHost, s->stream));
                s->hStats[CGRT_CNT_TOTAL * CGRT_MAX_CHAINS] = 0;
                if (s->lastPipeline == PIPE_WAVE)
                    CK(cudaMemcpyAsync(s->hStats + CGRT_CNT_TOTAL * CGRT_MAX_CHAINS, s->waveCtl.p + WCTL_ERR, sizeof(int), cudaMemcpyDeviceToHost, s->stream));
                fetched = true;
            }
        }
        CK(cudaStreamSynchronize(s->stream));
        if (fetched) {
            std::lock_guard<std::mutex> lk(s->mu);
            s->statsOnHost = true;
        }
    } else if (p->world == 1) {
        CK(cudaMemcpyAsync(rgb, s->frame.p, frameFloats * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
        CK(cudaStreamSynchronize(s->stream));
    } else {
        // scatter this rank's tiles into the caller's full-size frame (other pixels untouched)
        std::vector<float> tiles(outFloats);
        CK(cudaMemcpyAsync(tiles.data(), s->frame.p, outFloats * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
        CK(cudaStreamSynchronize(s->stream));
        TileLayout L;
        makeTileLayout(*p, L);
        const std::vector<int>& mine = L.lists[p->rank];
        const int tpx = L.tileW * L.tileH;
        for (size_t lt = 0; lt < mine.size(); lt++) {
            const int g = mine[lt], ty = g / L.tilesX, tx = g % L.tilesX;
            for (int q = 0; q < tpx; q++) {
                const int x = tx * L.tileW + q % L.tileW, y = ty * L.tileH + q / L.tileW;
                if (x >= p->width || y >= p->height) continue;
                const float* src = tiles.data() + 3 * (lt * tpx + q);
                float* dst = rgb + 3 * ((size_t)(p->height - 1 - y) * p->width + x);
                dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2];
            }
        }
    }
    if (stats) RC(cgrt_render_collect_stats(s, stats));
    return CGRT_OK;
}

// ---- several views of one scene in one frame --------------------------------------------------------------------------------
int cgrt_render_views(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p, float* rgb,
                      cgrt_render_stats* stats)
{
    RC(checkViews(s, cams, n_views, p, rgb));
    RC(useSceneDevice(s));
    std::lock_guard<std::mutex> hostLock(s->hostMu);
    const size_t floats = (size_t)n_views * p->width * p->height * 3;
    {
        std::lock_guard<std::mutex> lk(s->mu);
        RC(s->frame.ensure(floats));
    }
    RC(renderDevice(s, cams, n_views, p, s->frame.p, s->stream));
    CK(cudaMemcpyAsync(rgb, s->frame.p, floats * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    if (stats) RC(cgrt_render_collect_stats(s, stats));
    return CGRT_OK;
}

// ---- renderRayTracing's optional passes around the path (SURVEY.md §8 f1) -------------------------------------------------
int cgrt_render_effects(cgrt_scene* s, const cgrt_camera* cam, const cgrt_render_params* p, int32_t effects, float* rgb,
                        cgrt_render_stats* stats)
{
    if (!s || !cam || !rgb) return fail(CGRT_ERR_INVALID, "null argument");
    RC(checkRenderParams(p));
    if (p->world != 1) return fail(CGRT_ERR_INVALID, "cgrt_render_effects renders whole frames (world == 1)");
    if (effects & ~(CGRT_EFFECT_ANTIALIAS | CGRT_EFFECT_MOTION_BLUR | CGRT_EFFECT_BLOOM)) return fail(CGRT_ERR_INVALID, "unknown effect bits");
    if ((effects & CGRT_EFFECT_BLOOM) && (effects & CGRT_EFFECT_ANTIALIAS))
        return fail(CGRT_ERR_INVALID, "bloom with anti-aliasing is not offered: the reference's combination thresholds on an uninitialised "
                                      "accumulator (src/main.cpp:663-687)");
    if (!effects) return cgrt_render(s, cam, p, rgb, stats);
    RC(useSceneDevice(s));
    std::lock_guard<std::mutex> hostLock(s->hostMu);
    const int W = p->width, H = p->height;
    const size_t n = (size_t)W * H * 3;
    cudaStream_t st = s->stream;
    cgrt_render_stats total;
    std::memset(&total, 0, sizeof total);
    auto addStats = [&](const cgrt_render_stats& a) {
        total.primary += a.primary; total.primary_hit += a.primary_hit; total.shadow += a.shadow; total.bounce += a.bounce;
        total.kernel_launches += a.kernel_launches; total.device_ms += a.device_ms;
        total.replayed_closest += a.replayed_closest; total.replayed_shadow += a.replayed_shadow;
    };
    bool haveBloom = false; // fxC = bloom output of the un-shifted frame, fxA = that frame
    if (effects & CGRT_EFFECT_BLOOM) {
        // the pixel loop's frame, then bloomEffect (main.cpp:698-705, 586-628) on the device
        if ((int64_t)H > (int64_t)s->di.numSMs * 16 * 4) return fail(CGRT_ERR_INVALID, "frame too tall for the bloom pass");
        RC(s->fxA.ensure(n));
        RC(s->fxC.ensure(n));
        RC(s->fxM.ensure(n));
        RC(s->fxProg.ensure((size_t)H));
        RC(cgrt_render_device(s, cam, p, s->fxA.p, st));
        launchBloom(s->fxA.p, W, H, s->fxM.p, s->fxProg.p, s->fxC.p, s->di.numSMs, st);
        CK(cudaGetLastError());
        if (stats) {
            cgrt_render_stats one;
            RC(cgrt_render_collect_stats(s, &one));
            addStats(one);
            total.kernel_launches += 2;
        }
        haveBloom = true;
        if (!(effects & CGRT_EFFECT_MOTION_BLUR)) {
            CK(cudaMemcpyAsync(rgb, s->fxC.p, n * sizeof(float), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (stats) *stats = total;
            return CGRT_OK;
        }
    }
    if (effects & CGRT_EFFECT_MOTION_BLUR) {
        // blurEffect runs after the pixel loop and overwrites every pixel (main.cpp:716-719, :581), whatever the loop drew
        static const double shift[15] = {0.01, 0.02, 0.03, 0.04, 0.05, 0.06, 0.07, 0.08, 0.09, 0.10, 0.11, 0.12, 0.13, 0.14, 0.15};
        RC(s->fxA.ensure(n));
        RC(s->fxB.ensure(n));
        if (haveBloom) { // with bloom, matrixPixels enters blurEffect as colour + (bloom matrix + colour) (main.cpp:700, :622)
            launchAccumulate(s->fxB.p, s->fxA.p, n, true, st);
            launchAccumulate(s->fxB.p, s->fxC.p, n, false, st);
            total.kernel_launches += 2;
        }
        for (int k = 0; k < 15; k++) {
            cgrt_camera c = *cam;
            c.look_at[0] = (float)shift[k]; // cameraNew.setLookAt(glm::vec3(0.0k, 0, 0)), main.cpp:344-568
            c.look_at[1] = 0.0f;
            c.look_at[2] = 0.0f;
            RC(cgrt_render_device(s, &c, p, s->fxA.p, st));
            launchAccumulate(s->fxB.p, s->fxA.p, n, k == 0 && !haveBloom, st);
            if (stats) {
                cgrt_render_stats one;
                RC(cgrt_render_collect_stats(s, &one));
                addStats(one);
            }
        }
        launchDivide(s->fxB.p, n, 16.0f, s->fxA.p, st);
        total.kernel_launches += 16;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(rgb, s->fxA.p, n * sizeof(float), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    } else { // anti-aliasing
        if ((int64_t)W * 2 * H * 2 > (int64_t)1 << 28) return fail(CGRT_ERR_INVALID, "frame too large for 2x2 supersampling");
        cgrt_render_params big = *p;
        big.width = 2 * W;
        big.height = 2 * H;
        RC(s->fxA.ensure(n * 4));
        RC(s->fxB.ensure(n));
        RC(cgrt_render_device(s, cam, &big, s->fxA.p, st)); // aspect stays cam->aspect (W/H)
        launchAADownsample(s->fxA.p, W, H, s->fxB.p, st);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(rgb, s->fxB.p, n * sizeof(float), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (stats) {
            cgrt_render_stats one;
            RC(cgrt_render_collect_stats(s, &one));
            addStats(one);
            total.kernel_launches += 1;
        }
    }
    if (stats) *stats = total;
    return CGRT_OK;
}

// ---- streaming form: up to two frames in flight, the D2H copy of frame k overlaps the kernels of frame k+1 -----------------
int cgrt_render_submit(cgrt_scene* s, const cgrt_camera* cam, const cgrt_render_params* p, float* rgb_host)
{
    if (!s || !cam || !rgb_host) return fail(CGRT_ERR_INVALID, "null argument");
    RC(checkRenderParams(p));
    if (p->world != 1) return fail(CGRT_ERR_INVALID, "cgrt_render_submit renders whole frames (world == 1)");
    RC(useSceneDevice(s));
    std::lock_guard<std::mutex> hostLock(s->hostMu);
    const size_t frameFloats = (size_t)p->width * p->height * 3;
    int slot;
    {
        std::lock_guard<std::mutex> lk(s->mu);
        if (!s->copyStream) {
            CK(cudaStreamCreateWithFlags(&s->copyStream, cudaStreamNonBlocking));
            for (int k = 0; k < 2; k++) {
                CK(cudaEventCreateWithFlags(&s->renderDone[k], cudaEventDisableTiming));
                CK(cudaEventCreateWithFlags(&s->copyDone[k], cudaEventDisableTiming));
            }
        }
        slot = (int)(s->submitSeq++ & 1);
        if (s->slotUsed[slot]) {
            CK(cudaEventSynchronize(s->copyDone[slot])); // at most two frames in flight: frame k-2 has been delivered
        }
        RC(s->streamFrame[slot].ensure(frameFloats));
        s->slotUsed[slot] = true;
    }
    RC(cgrt_render_device(s, cam, p, s->streamFrame[slot].p, s->stream));
    CK(cudaEventRecord(s->renderDone[slot], s->stream));
    CK(cudaStreamWaitEvent(s->copyStream, s->renderDone[slot], 0));
    CK(cudaMemcpyAsync(rgb_host, s->streamFrame[slot].p, frameFloats * sizeof(float), cudaMemcpyDeviceToHost, s->copyStream));
    CK(cudaEventRecord(s->copyDone[slot], s->copyStream));
    return CGRT_OK;
}

int cgrt_render_wait(cgrt_scene* s)
{
    if (!s) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useSceneDevice(s));
    if (s->copyStream) CK(cudaStreamSynchronize(s->copyStream));
    CK(cudaStreamSynchronize(s->stream));
    return CGRT_OK;
}

// cached tile lists of every rank for the assemble step on rank 0
struct AssembleCache {
    int key[6] = {0, 0, 0, 0, 0, 0};
    int* dLists = nullptr;
    int* dCounts = nullptr;
    TileLayout L;
};
static std::mutex g_asmMu;
static std::map<int, AssembleCache> g_asm; // per device

int cgrt_assemble_tiles(int device, const cgrt_render_params* p, const float* d_gathered, float* d_frame, void* stream)
{
    if (!d_gathered || !d_frame) return fail(CGRT_ERR_INVALID, "null argument");
    RC(checkRenderParams(p));
    RC(useDevice(device));
    DeviceInfo di;
    RC(deviceInfo(device, di));
    std::lock_guard<std::mutex> lk(g_asmMu);
    AssembleCache& c = g_asm[device];
    TileLayout L;
    makeTileLayout(*p, L);
    const int key[6] = {p->width, p->height, L.tileW, L.tileH, L.world, 1};
    if (std::memcmp(key, c.key, sizeof key) != 0) {
        CK(cudaDeviceSynchronize());
        if (c.dLists) cudaFree(c.dLists);
        if (c.dCounts) cudaFree(c.dCounts);
        c.dLists = c.dCounts = nullptr;
        std::vector<int> lists((size_t)L.world * std::max(L.maxTiles, 1), 0), counts(L.world, 0);
        for (int r = 0; r < L.world; r++) {
            counts[r] = (int)L.lists[r].size();
            std::copy(L.lists[r].begin(), L.lists[r].end(), lists.begin() + (size_t)r * L.maxTiles);
        }
        CK(cudaMalloc((void**)&c.dLists, lists.size() * sizeof(int)));
        CK(cudaMalloc((void**)&c.dCounts, counts.size() * sizeof(int)));
        CK(cudaMemcpy(c.dLists, lists.data(), lists.size() * sizeof(int), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(c.dCounts, counts.data(), counts.size() * sizeof(int), cudaMemcpyHostToDevice));
        CK(uploadsDone());
        std::memcpy(c.key, key, sizeof key);
        c.L = L;
    }
    const size_t perRank = (size_t)L.maxTiles * L.tileW * L.tileH * 3;
    launchAssemble(d_gathered, perRank, c.dLists, c.dCounts, L.maxTiles, L.world, L.tileW, L.tileH, L.tilesX, p->width,
                   p->height, d_frame, di.numSMs, (cudaStream_t)stream);
    CK(cudaGetLastError());
    return CGRT_OK;
}

int cgrt_quantize_rgba8(int device, const float* d_frame, size_t n_pixels, uint8_t* d_rgba8, void* stream)
{
    if (n_pixels && (!d_frame || !d_rgba8)) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useDevice(device));
    launchQuantize(d_frame, n_pixels, d_rgba8, (cudaStream_t)stream);
    CK(cudaGetLastError());
    return CGRT_OK;
}

// timeline of the last k_wave frame (CGRT_WAVE_TRACE=1): out[k][8] = {valid, rays in flight, ray queue head, tail, finish queue
// head, tail, second-part head, tail} for the k-th 4.096 us bucket since the kernel started; returns the number of buckets copied
int cgrt_debug_wave_timeline(cgrt_scene* s, int32_t* out, int32_t cap)
{
    if (!s || !out || !s->waveTrace.p) return 0;
    if (useSceneDevice(s) != CGRT_OK) return 0;
    const int n = std::min<int>(cap, WAVE_TRACE_SAMPLES);
    if (cudaMemcpy(out, s->waveTrace.p, (size_t)n * 8 * sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    return n;
}

// the finisher share the persistent wavefront currently uses for this scene's frames (WaveTuner; 0 before the first frame) and
// the device times it has measured per setting: out[0] = current setting, out[f] = ms of setting f (f = 2..14), 0 = not tried
int cgrt_debug_wave_tuner(cgrt_scene* s, float* out, int32_t cap)
{
    if (!s || !out || cap < WaveTuner::HI + 1) return 0;
    std::lock_guard<std::mutex> lk(s->mu);
    out[0] = (float)s->tuner.cur;
    out[1] = (float)s->tuner.frames;
    for (int f = WaveTuner::LO; f <= WaveTuner::HI; f++) out[f] = s->tuner.ms[f];
    return WaveTuner::HI + 1;
}

#ifdef CGRT_WAVE_LAT
// instrumented builds: per-ticket latency records of the last k_wave frame (layout in cgrt_wave.cuh); returns tickets copied
int cgrt_debug_wave_latency(cgrt_scene* s, uint32_t* out, int32_t cap)
{
    if (!s || !out || !s->waveLat.p) return 0;
    if (useSceneDevice(s) != CGRT_OK) return 0;
    const int n = (int)std::min<size_t>((size_t)cap, s->waveLat.n / 16);
    if (cudaMemcpy(out, s->waveLat.p, (size_t)n * 16 * sizeof(unsigned), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    return n;
}
#endif
#ifdef CGRT_INSTRUMENT
void cgrt_debug_instrumentation(unsigned long long* out, int reset) { cgrt::readInstrumentation(out, reset != 0); }
void cgrt_debug_timeline(unsigned int* out, int reset) { cgrt::readTimeline(out, reset != 0); }
void cgrt_debug_step_hist(unsigned int* out, int reset) { cgrt::readStepHist(out, reset != 0); }
#endif

// ---- peer memory + frame hand-off flags (multi-GPU, one process per GPU) ---------------------------------------------
int cgrt_peer_export(int device, void* d_ptr, uint8_t* handle)
{
    if (!d_ptr || !handle) return fail(CGRT_ERR_INVALID, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == CGRT_IPC_HANDLE_BYTES, "IPC handle size");
    RC(useDevice(device));
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, d_ptr));
    std::memcpy(handle, &h, sizeof h);
    return CGRT_OK;
}
int cgrt_peer_open(int device, const uint8_t* handle, void** out)
{
    if (!handle || !out) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useDevice(device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof h);
    CK(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    return CGRT_OK;
}
int cgrt_peer_close(int device, void* p)
{
    RC(useDevice(device));
    CK(cudaIpcCloseMemHandle(p));
    return CGRT_OK;
}
int cgrt_flag_signal(int device, uint32_t* const* d_flags, int32_t n, uint32_t seq, void* stream)
{
    if (n < 0 || n > CGRT_MAX_PEERS || (n && !d_flags)) return fail(CGRT_ERR_INVALID, "bad flag list");
    RC(useDevice(device));
    launchFlagSignal(d_flags, n, seq, (cudaStream_t)stream);
    CK(cudaGetLastError());
    return CGRT_OK;
}
int cgrt_flag_wait(int device, const uint32_t* d_flags, int32_t n, uint32_t seq, uint32_t timeout_ms, uint32_t* d_status,
                   void* stream)
{
    if (n < 0 || n > 1024 || (n && !d_flags)) return fail(CGRT_ERR_INVALID, "bad flag list");
    RC(useDevice(device));
    launchFlagWait(d_flags, n, seq, (unsigned long long)timeout_ms * 1000000ull, d_status, (cudaStream_t)stream);
    CK(cudaGetLastError());
    return CGRT_OK;
}
int cgrt_memset_device(int device, void* p, int value, size_t bytes, void* stream)
{
    RC(useDevice(device));
    CK(cudaMemsetAsync(p, value, bytes, (cudaStream_t)stream));
    return CGRT_OK;
}
int cgrt_memcpy_d2h_async(int device, void* dst, const void* src, size_t bytes, void* stream)
{
    RC(useDevice(device));
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return CGRT_OK;
}

// ---- memory helpers ------------------------------------------------------------------------------------------------
int cgrt_device_malloc(int device, size_t bytes, void** out)
{
    if (!out) return fail(CGRT_ERR_INVALID, "null argument");
    RC(useDevice(device));
    cudaError_t e = cudaMalloc(out, bytes ? bytes : 1);
    if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? CGRT_ERR_OOM : CGRT_ERR_CUDA, cudaGetErrorString(e));
    return CGRT_OK;
}
int cgrt_device_free(int device, void* p)
{
    RC(useDevice(device));
    CK(cudaFree(p));
    return CGRT_OK;
}
int cgrt_host_alloc_pinned(size_t bytes, void** out)
{
    if (!out) return fail(CGRT_ERR_INVALID, "null argument");
    CK(cudaMallocHost(out, bytes ? bytes : 1));
    return CGRT_OK;
}
int cgrt_host_free_pinned(void* p)
{
    CK(cudaFreeHost(p));
    return CGRT_OK;
}
int cgrt_memcpy_h2d(int device, void* dst, const void* src, size_t bytes)
{
    RC(useDevice(device));
    CK(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
    CK(uploadsDone()); // (the caller launches on streams of its own next)
    return CGRT_OK;
}
int cgrt_memcpy_d2h(int device, void* dst, const void* src, size_t bytes)
{
    RC(useDevice(device));
    CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return CGRT_OK;
}
int cgrt_device_synchronize(int device)
{
    RC(useDevice(device));
    CK(cudaDeviceSynchronize());
    return CGRT_OK;
}

} // extern "C"
