// Host-visible declarations of the kernel launchers (cgrt_kernels.cu) and the structures they share with cgrt_capi.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

// ---- HBM layout -----------------------------------------------------------------------------------------------------------
// nodes     : 2 x float4 per node (32 B, 32-byte aligned):  [lo.xyz | a]  [hi.xyz | b]
//               inner node: a = index of the left child (right child = a + 1, createTree pushes them consecutively,
//                           src/bounding_volume_hierarchy.cpp:358-364), b = 0
//               leaf      : a = first triangle (leaf order), b = triangle count (> 0)
// triPl     : float4 per triangle (leaf order): plane normal.xyz, D     (trianglePlane, src/ray_tracing.cpp:74-82, precomputed
//             on the device with the same expression tree -> same bits as the reference's per-test recomputation)
// triV0/1/2 : float4 per triangle: position.xyz ; triV0.w = global triangle id (bit-cast), triV1.w = mesh/material id,
//             triV2.w = rank of the triangle in the reference's own leaf order (tie-break, see cgrt_device.cuh)
//             Inside a reference leaf the triangles are stored in sub-tree order (bvh_build.cpp buildLeafSubTrees).
// pairs     : the production traversal's reference-node array: one entry of 4 x float4 per inner reference node holding both
//             children: [l.lo | l.w0] [l.hi | l.w1] [r.lo | r.w0] [r.hi | r.w1]; w0 = id to visit the child with (encoding
//             in cgrt_device.cuh), w1 = reference node index of the child. rootId = id of the root.
// wide      : 8-wide nodes of the culling sub-trees that refine the reference leaves, 14 x float4 each:
//             lo.x[0..3] lo.x[4..7] lo.y.. lo.z.. hi.x.. hi.y.. hi.z.. id[0..3] id[4..7]; boxes pre-expanded (bvh_build.cpp)
// triN0/1/2 : float4 per triangle: vertex normal.xyz (read only for the final hit); triN0.w = reference leaf node of the triangle
//             The top of `wide` also holds the FAST TREE (bvh_build.cpp buildFastTree): the reference tree collapsed into
//             8-wide conservative nodes whose leaves are the sub-tree roots above - one tree over all triangles.
// mats      : 2 x float4 per mesh:  [kd.xyz | shininess] [ks.xyz | transparency]        (src/mesh.h:17-23)
// spheres   : 3 x float4 per sphere: [center | radius] [kd | shininess] [ks | transparency]  (src/scene.h:36-40)
struct DevScene {
    const float4* nodes;
    const float4* triPl;
    const float4* triV0;
    const float4* triV1;
    const float4* triV2;
    const float4* tri4;   // 4 x float4 per triangle (64 B, one cache line half): [plane] [v0|gid] [v1|mesh] [v2|rank] - the
                          // traversal's copy of triPl/triV0/1/2, so that one triangle test touches one line instead of four
    const float4* tri4f;  // the same records in the FAST TREE's triangle order, with [v2 | position in tri4] - read by the
                          // speculative search only (identity order unless the fast tree is the independent SAH tree)
    const float4* triN0;
    const float4* triN1;
    const float4* triN2;
    const float4* mats;
    const float4* spheres;
    const float4* pairs;
    const float4* wide;
    const float4* wide8;  // the same 8-wide nodes child-major: child j = [lo.xyz | id] [hi.xyz | -] at float4 2j, 2j+1 (256 B per
                          // node), for the cooperative search where lane j of a ray's group owns child j
    const int* origToLeaf; // global triangle id -> leaf-order index (brute-force path only)
    const int* alwaysTri;  // positions of the triangles the fast tree does not cover (unboundable accept region): every ray tests them
    int nAlways;
    const int* refParent;  // reference node -> parent (-1 for the root): certification of the speculative traversal
    uint32_t fastRoot;     // id of the root of the fast tree in `wide` (0 = none: exact traversal only)
    int nNodes;
    int nTris;
    int nSpheres;
    int nMeshes;
    int rootId;
};


namespace cgrt {

#define CGRT_STACK 32                           // traversal stack: one pending sibling per level below the root (reference depth 12)
#define CGRT_MAX_BVH_DEPTH (CGRT_STACK + 1)     // largest cgrt_scene_options::bvh_max_depth the stack supports
#define CGRT_MAX_LEVELS 16                      // upper bound on cgrt_render_params::trace_limit
#define CGRT_CNT_HIT 0                          // counts[CGRT_CNT_HIT + level]    = hits found at `level`
#define CGRT_CNT_BOUNCE CGRT_MAX_LEVELS         // counts[CGRT_CNT_BOUNCE + level] = rays queued for `level` (level >= 1)
#define CGRT_CNT_WORK (2 * CGRT_MAX_LEVELS + 1)  // counts[CGRT_CNT_WORK + k] = work counter of the k-th persistent launch of the frame
#define CGRT_CNT_PATHS (CGRT_CNT_WORK + 2 * CGRT_MAX_LEVELS + 2) // path pipeline: pixels whose primary ray hit (= paths)
#define CGRT_CNT_HITS (CGRT_CNT_PATHS + 1)                      // path pipeline: hit records of all levels
#define CGRT_CNT_BOUNCES (CGRT_CNT_PATHS + 2)                   // path pipeline: reflection rays traced
#define CGRT_CNT_REPLAY_PATHS (CGRT_CNT_PATHS + 3)              // rays the speculative closest-hit kernel deferred to the exact one
#define CGRT_CNT_REPLAY_SHADOW (CGRT_CNT_PATHS + 4)             // shadow rays deferred to the exact any-hit kernel
#define CGRT_CNT_BBOX (CGRT_CNT_PATHS + 5) // 4 ints, bounding box of the pixels the shading pass coloured (whole frames in Screen
                                          // layout): max of x + 1, row + 1, W - x, H - row; 0 = no pixel (counters start at zero)
#define CGRT_CNT_TOTAL (CGRT_CNT_PATHS + 9)
#define CGRT_MAX_PEERS 32                       // flags one signal launch can write (GPUs of one box)
#define CGRT_PARAM_BLOCK_HEADER 128             // bytes reserved for FrameParams in the per-frame block; lights, then cameras follow

// Per-frame constants, evaluated on the host with libm exactly as Trackball does (framework/src/trackball.cpp:70-73, 92-103)
// so that device sinf/cosf/tanf never enter the picture. Uploaded once per render together with the lights.
struct FrameParams {
    float camX, camY, camZ; // Trackball::position()
    float halfW, halfH;     // aspect * tan(fovy/2), tan(fovy/2)
    float qx, qy, qz, qw;   // glm::quat(m_rotationEulerAngles)
    int width, height;
    int nLights;
    int traceLimit;
    int nSlots;             // local pixel slots = owned tiles * tileW * tileH
    int tileW, tileH, tilesX;
    int world, rank;
    int screenLayout;       // 1: pixels are written at their Screen position (row H-1-y); 0: tile-major buffer of this rank
    int nSph;               // spherical lights (2 x float4 each, after the point lights in the parameter block)
    int nViews;             // cameras of the frame (cgrt_render_views; 1 otherwise). nSlots counts the slots of all views; the
                            // views' camera constants follow the lights in the parameter block (CGRT_VIEW_F4 x float4 each)
};
// camera constants of one view in the parameter block: [camX camY camZ | halfW] [qx qy qz qw] [halfH | - - -]
#define CGRT_VIEW_F4 3
#define CGRT_MAX_VIEWS 1024

// Four kernel sets render a frame; cgrt_capi.cu choosePipeline picks one per frame (all give the same pixels and ray counts):
//   counting wavefront  CGRT_RENDER_COUNT                                         launchCountingFrame, CountBuffers
//   path pipeline       scenes without a fast tree; frames too large for rounds   launchPathPipeline, PathBuffers
//   round pipeline      large shallow frames of scenes with a fast tree           launchRoundPipeline, RoundBuffers per chain
//   k_wave              every other frame of a scene with a fast tree             launchWavePipeline, RoundBuffers + WaveQ

// Queues of the counting wavefront (all sized for the worst case `cap` = nSlots; only the used prefix is ever touched).
struct CountBuffers {
    float4* hitQ;      // 3 x float4 per hit:   [P | matId] [N | outIdx] [D | pathId]
    float4* bounceQ;   // 2 x float4 per ray:   [origin | tmax] [direction | pathId]
    uint8_t* lit;      // [hit][light] 1 = light reaches the point
    int* pathPix;      // [pathId] output index of the path's pixel
    float4* pathState; // [level][pathId] 2 x float4: directColor, ks of the shade() frame waiting for its reflection
    int* counts;       // CGRT_CNT_TOTAL queue lengths
    unsigned long long* tests; // [class 0..2][box, tri] reference test counts
    size_t cap;
};

// Queues of the path pipeline (cgrt_kernels.cu "path pipeline"): one persistent closest-hit kernel follows every
// path from its primary ray through its mirror bounces and leaves one hit record per (path, level); all shadow rays of the
// frame are then traced by one any-hit launch and one shading launch folds each path back to its pixel.
struct PathBuffers {
    float4* hitRec;    // [path * levels + level] 3 x float4: [P | matId] [N | t] [D | id] (hitRecordId)
    int* hitList;      // [i] = path * levels + level, compacted list of all hit records (shadow work items)
    uint8_t* lit;      // [(path * levels + level) * nLights + light] 1 = light reaches the point
    int* pathPix;      // [path] output index of the path's pixel
    int* pathDepth;    // [path] number of levels that recorded a hit
    float4* replayQ;   // 3 x float4 per deferred ray: [origin | tmax] [direction | level] [path, outIdx, -, -]
    int* replayShadow; // deferred shadow work items (index of the lit flag)
    int* counts;       // shared with CountBuffers::counts
    size_t cap;        // paths the buffers can hold (= local pixel slots)
    int levels;        // trace limit the buffers are laid out for
};

// Buffers of the ROUND pipeline (cgrt_kernels.cu "round pipeline"; k_wave uses the records and counters, not the ray lists):
//   k_gen      : one thread per pixel slot: primary ray, the reference's root-box test, compacted list of rays that enter
//   round r    : k_trace  - persistent warps, speculative search ONLY (no prologue / epilogue code in the hot loop) over the
//                           closest-hit rays of level r and the shadow rays of the hits of level r-1
//                k_finish - one thread per traced ray, converged: certificate (or exact replay), sphere loop, hit epilogue,
//                           hit record, emission of the next level's reflection ray and of the shadow rays
//   k_shade_slots : one thread per pixel slot folds the levels back to the pixel
// Ray record: 3 x float4  [origin | tmax] [direction | maxDist] [slot, level / lit index, eps, -]; result: [state, t, tri, -]
struct RoundBuffers {
    float4* cRay[2];   // closest-hit rays, double-buffered by level parity
    float4* cRes[2];
    float4* sRay[2];   // shadow rays, double-buffered by level parity
    float4* sRes[2];
    float4* hitRec;    // [slot * levels + level] 3 x float4: [P | matId] [N | t] [D | id] (hitRecordId)
    uint8_t* lit;      // [(slot * levels + level) * nLights + light]
    int* pathDepth;    // [slot] number of levels that recorded a hit (0: the pixel is already final)
    int* counts;
    int levels;
    // spherical-light soft shadows (src/main.cpp:168-218), scenes with Scene::sphericalLight only
    int* softList;     // hit records of the frame (slot * levels + level), compacted; softList[cap * levels] = their number
    float* soft;       // [(slot * levels + level) * nSph + light] fraction of the 200 sample rays that reach the light
    unsigned softSeed;
};
// hitRecordId: D.w of a hit record (bit-cast int) = the triangle's LEAF-ORDER index (global id: triV0[id].w), or -2 - s for
// sphere s. N.w = t of the hit. The shading passes read neither lane; the AOV pass reads both.

// Per-pixel buffers of a frame (cgrt_render_aovs, cgrt_render_paths), Screen layout, view after view; a null pointer is not
// written. Level l of the pixel's mirror path (the ray trace(l) cast and its hit) is at pixel l * levelPixels + the pixel's
// index; cgrt_render_aovs is the one-level case without ray, position and visibility.
struct AovBuffers {
    float* depth;   // t of the level's closest hit; the ray's t on a miss, FLT_MAX where the level cast no ray
    int* tri;       // global triangle id of that hit, -1 miss or no ray, -2 - s sphere s
    float* normal;  // 3 floats: shading normal of that hit, 0 on a miss or no ray
    uint8_t* hits;  // levels of the pixel's path that recorded a hit (pathDepth); one per pixel, not per level
    float4* ray;        // 2 float4s: the level's ray [origin | t] [direction | 0]; all +0 where the level cast no ray
    float* position;    // 3 floats: the hit record's P (the point shading() used), 0 where the level did not hit
    float* visibility;  // nLights floats: each light's shadow factor at that point, point lights then spherical lights (1 / 0
                        // lit / shadowed, k / 200 of the soft-shadow samples), 0 where the level did not hit
    int levels;         // levels written (1..max(trace limit, 1))
    size_t levelPixels; // pixels of all views
    int nLights;        // cgrt_render_paths: the caller's light count, checked again when the frame reads the lights; -1: not given
};

// Light-group buffers of a frame (cgrt_render_lights): group g's [n_views][H][W][3] at rgb + g * groupFloats, Screen layout.
// A light's group is the bit-cast int in the w lane of its colour in the parameter block (-1: no group); no other pass reads it.
struct LightGroupBuffers {
    float* rgb;
    size_t groupFloats; // 3 x pixels of all views
    int nGroups;
};
#define CGRT_MAX_LIGHT_GROUPS 64

// ---- persistent wavefront (cgrt_wave.cuh): control block + ticket queue of the single-kernel frame ----------------------------
#define WCTL_PENDING 0  // u64 at int index 0: (CTAs done with phase A << 32) | rays in flight
#define WCTL_ERR 2      // watchdog: a warp waited longer than WaveQ::timeoutNs
#define WCTL_HEAD 32    // ray queue: tickets handed out           (every counter on its own 128-byte line)
#define WCTL_TAIL 64    // ray queue: tickets reserved by producers
#define WCTL_FHEAD 96   // finish queue: tickets handed out
#define WCTL_FTAIL 128  // finish queue: tickets reserved
#define WCTL_HEAD2 160  // ray queue, second part (after the change-over to the cooperative search form): own counters
#define WCTL_TAIL2 192
#define WCTL_FINCOUNT 288 // finish warps of the frame / finish warps that have left their loop (phase C waits for equality);
#define WCTL_FINEXIT 289  // own 128-byte line
#define WCTL_T0 4       // low 32 bits of %globaltimer of the first CTA that started (timeline origin)
#define WCTL_CLOSEAT 224 // 1 + the first ticket of the first part that will never be served (0 = the first part is open)
#define WCTL_RESUME 256  // search states handed over from the LANE form to the GROUP form at the change-over (WaveQ::resume)
#define WCTL_DONE 320   // 32 copies of the done flag, one per 128-byte line (ctl[WCTL_DONE + 32 k])
#define WCTL_SCRATCH (WCTL_DONE + 32 * 32) // 32 words, one per 128-byte line: targets of the release reductions (waveRelease)
#define WCTL_INTS (WCTL_SCRATCH + 32 * 32)

struct WaveQ {
    float4* rays;   // ray queue: 3 x float4 per ticket (layout in cgrt_wave.cuh)
    float4* fin;    // finish queue: 2 x float4 per ticket
    int* ctl;       // WCTL_INTS ints, zeroed before every frame
    uint32_t seq;   // sequence number of this frame on these queues (never 0)
    int cap;        // tickets each array can hold
    int mode;       // search form of the frame: 1 LANE (one lane per ray) first, 2 GROUP (eight lanes per ray) throughout
    int switchBelow; // mode 1: change over to GROUP when fewer rays than this are in flight (0 = never)
    int finEvery;   // SMs with %smid % finEvery == 0 run the finish warps, the others the search warps
    unsigned long long timeoutNs;
    int resumeCap;  // states the side array holds
    float4* resume; // search states of rays handed over at the change-over: WAVE_RESUME_F4 x float4 each, one per LANE-form lane of
                    // the grid (a lane hands over at most once per frame); nullptr = rays finish in the form they started in
    unsigned* lat;  // instrumented builds only (-DCGRT_WAVE_LAT): 8 timestamps / counters per ray ticket (tools/wave_latency.py)
    int* trace;     // optional (CGRT_WAVE_TRACE=1): WAVE_TRACE_SAMPLES x 8 ints, one sample of the counters per 4.096 us of the frame
};
#define WAVE_TRACE_SAMPLES 1024
#define WAVE_RESUME_STACK 32                        // deepest traversal stack that is handed over (deeper: the ray stays where it is)
#define WAVE_RESUME_F4 (1 + WAVE_RESUME_STACK / 2)  // [t, tri, t2, node] + two stack entries (node, entry distance) per float4

#define CGRT_TRACE_MAX_KERNELS (8 * (2 * (CGRT_MAX_LEVELS + 1) + 1) + 2) // chains x (k_gen + 2 per round) + shade
// optional per-kernel event trace of one wavefront (classes: 0 primary, 1 bounce closest-hit, 2 shadow, 3 shade)
struct WaveTrace {
    cudaEvent_t* ev;   // 2 * maxKernels events
    int maxKernels;
    int classMask;
    int n;             // traced kernels
    int cls[CGRT_TRACE_MAX_KERNELS];
    int launches[4];
};

void launchSetupPlanes(const float4* v0, const float4* v1, const float4* v2, float4* pl, float4* tri4, int n, cudaStream_t st);
void launchPermuteTri4(const float4* tri4, const int* fastOrder, float4* tri4f, int n, cudaStream_t st);
void launchClosestBatch(const DevScene& S, const float4* rays, size_t n, float4* hits, uint32_t* counts, int numSMs,
                        cudaStream_t st);
void launchAnyBatch(const DevScene& S, const float4* rays, const float* maxDist, float eps, size_t n, uint8_t* occluded,
                    int numSMs, cudaStream_t st);
void launchBruteBatch(const DevScene& S, const float4* rays, size_t n, float4* hits, int numSMs, cudaStream_t st);
void launchUnitAabb(const float* boxes, const float4* rays, size_t n, uint8_t* hit, float* t, cudaStream_t st);
void launchUnitTriangle(const float* tris, const float4* rays, size_t n, float4* out, cudaStream_t st);
void launchUnitPlane(const float4* planes, const float4* rays, size_t n, uint8_t* hit, float* t, cudaStream_t st);
void launchUnitTrianglePlane(const float* tris, size_t n, float4* planes, cudaStream_t st);
void launchUnitPointInTriangle(const float* in, size_t n, uint8_t* inside, cudaStream_t st);
void launchUnitSphere(const float4* spheres, const float4* rays, size_t n, float* out, cudaStream_t st);
void launchGenerateRays(const FrameParams* dP, int nPixels, float4* rays, cudaStream_t st);
// The launchers return the kernels they launched (cgrt_render_stats::kernel_launches).
int launchCountingFrame(const DevScene& S, const FrameParams* dP, const FrameParams& hP, const float4* dLights,
                        const CountBuffers& B, const int* dTileList, float* fb, int numSMs, WaveTrace* tr, cudaStream_t st);
int launchPathPipeline(const DevScene& S, const FrameParams* dP, const FrameParams& hP, const float4* dLights,
                       const PathBuffers& B, const int2* dTileSeq, float* fb, int numSMs, WaveTrace* tr, cudaStream_t st);
#define CGRT_MAX_CHAINS 8
// streams / events of the round pipeline's chains (chain 0 runs on the caller's stream)
struct ChainSync {
    cudaStream_t streams[CGRT_MAX_CHAINS];
    cudaEvent_t fork, join[CGRT_MAX_CHAINS];
};
int roundPipelineChains(int nSlots); // number of chains the round pipeline uses for a frame share of nSlots pixels (CGRT_TUNE chains=N overrides)
int launchRoundPipeline(const DevScene& S, const FrameParams* dP, const FrameParams& hP, const float4* dLights,
                        const RoundBuffers* chains, int nChains, const ChainSync& sync, const int2* dTileSeq, float* fb,
                        int numSMs, WaveTrace* tr, cudaStream_t st);
// one kernel per frame: phase A ray generation, phase B search + finish over the device-side queue, phase C shading
int waveGridBlocks(int numSMs); // co-resident CTAs of k_wave on this device (occupancy x SMs; CGRT_TUNE waveblocks=N caps the per-SM count)
int launchWavePipeline(const DevScene& S, const FrameParams* dP, const FrameParams& hP, const float4* dLights,
                       const RoundBuffers& B, const WaveQ& Q, const int2* dTileSeq, float* fb, int numSMs, WaveTrace* tr,
                       cudaStream_t st);
// The AOV / mirror-path pass after a frame of the path, round or wave pipeline (whole frames in Screen layout). pathDepth ==
// nullptr: no records (trace limit 0), every pixel is a miss; perPath: the path pipeline's records (per path, pathPix gives the
// pixel), else one record chain per pixel slot. lit / soft: the frame's lit flags and soft-shadow fractions (read for
// A.visibility only; soft: the round pipeline with spherical lights). Returns the kernels it launched.
int launchAovPass(const DevScene& S, const FrameParams* dP, const FrameParams& hP, const float4* dLights, const float4* hitRec,
                  const uint8_t* lit, const float* soft, const int* pathDepth, bool perPath, const int* pathPix, const int* counts,
                  const int2* dTileSeq, const AovBuffers& A, int numSMs, cudaStream_t st);
// The light-group pass after a frame of the path, round or wave pipeline with trace limit > 0 (whole frames in Screen layout).
// perPath: the path pipeline's records, written through pathPix into buffers the caller has cleared to +0 (misses have no
// record); else every pixel slot's chain, misses included. soft: the round pipeline's soft-shadow fractions (spherical lights).
// Returns the kernels it launched.
int launchLightPass(const DevScene& S, const FrameParams* dP, const FrameParams& hP, const float4* dLights, const float4* hitRec,
                    const uint8_t* lit, const float* soft, const int* pathDepth, bool perPath, const int* pathPix, const int* counts,
                    const int2* dTileSeq, const LightGroupBuffers& G, int numSMs, cudaStream_t st);
void launchDeliverBox(const int* bbox, int W, int H, const float* frame, float* hostFrame, int numSMs, cudaStream_t st);
void launchAssemble(const float* gathered, size_t perRankFloats, const int* tileLists, const int* tileCounts, int maxTiles,
                    int world, int tileW, int tileH, int tilesX, int width, int height, float* frame, int numSMs,
                    cudaStream_t st);
void launchFlagSignal(uint32_t* const* flags, int n, uint32_t seq, cudaStream_t st);
void launchFlagWait(const uint32_t* flags, int n, uint32_t seq, unsigned long long timeoutNs, uint32_t* status, cudaStream_t st);
// bloom of nViews frames [nViews][H][W][3] into out (same layout); M: nViews x W x H x 3 floats, progress: nViews x H + 1 ints
void launchBloom(const float* frame, int W, int H, int nViews, float* M, int* progress, float* out, int numSMs, cudaStream_t st);
// big [nViews][2H][2W][3] -> out [nViews][H][W][3]
void launchAADownsample(const float* big, int W, int H, int nViews, float* out, cudaStream_t st);
// motion blur of several views: frames holds cameras c0..c1-1 of the flattened (view, k) list (15 per view, view-major), each
// W x H x 3 floats; acc = [views][W x H x 3]. bloomIn (optional): the un-shifted frames, whose bloom output acc holds before k = 0.
void launchBlurViews(const float* frames, int c0, int c1, size_t n, const float* bloomIn, float* acc, float div, cudaStream_t st);
void launchAccumulate(float* acc, const float* frame, size_t n, bool first, cudaStream_t st);
void launchDivide(const float* acc, size_t n, float div, float* out, cudaStream_t st);
void launchQuantize(const float* frame, size_t nPixels, uint8_t* rgba, cudaStream_t st);

} // namespace cgrt
