/* cgrt_b200.h — C ABI of the B200-native hot path of CG-RayTracer (libcgrt_b200.so).
 *
 * Scope: BVH traversal + ray/AABB + ray/triangle intersection driven by the per-pixel getFinalColor recursion
 * (Phong shading, hard shadow rays, mirror bounces), i.e. SURVEY.md §8 rows (a)-(e). Everything behind this header is
 * hand-written CUDA for sm_100a; there is NO CPU fallback: every entry returns CGRT_ERR_NO_DEVICE / CGRT_ERR_CUDA when no
 * usable GPU is present. No torch / C++ types cross this boundary: plain pointers and sizes only.
 *
 * Each entry cites the reference interface it replaces (paths relative to the reference checkout).
 * The reference has no FFI layer (in-process C++), so these are the symbols a maintainer binds from the C++ shims in
 * cg-raytracer_b200/host/ (same class / function names as the reference) — see INTEGRATION.md.
 *
 * Conventions: return 0 (CGRT_OK) on success, non-zero error code otherwise; never throws; cgrt_last_error() returns a
 * thread-local human-readable message for the last failing call on this thread. Host callers own host buffers, the
 * library owns device memory. All entry points may be called concurrently from several host threads on the same scene
 * (the reference's intersect() is const and called from all OpenMP threads, src/main.cpp:653-656 -> :276). The query entries
 * (cgrt_intersect_closest / _any and their _device forms) share nothing between threads: each host thread has its own stream
 * and device scratch, kept between calls, so concurrent queries overlap on the device. Renders of ONE scene are serialised
 * (they share the scene's ray queues; the reference calls renderRayTracing from the UI thread only), renders of different
 * scenes are not. cgrt_render_device enqueues on the caller's stream: frames of one scene must be enqueued on one stream
 * (or ordered by the caller) - the next frame reuses the queues of the previous one.
 */
#ifndef CGRT_B200_H
#define CGRT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CGRT_VERSION 100

enum {
    CGRT_OK = 0,
    CGRT_ERR_INVALID = 1,   /* bad argument */
    CGRT_ERR_NO_DEVICE = 2, /* no CUDA device / driver: the product has no CPU path */
    CGRT_ERR_CUDA = 3,      /* a CUDA runtime call failed (message in cgrt_last_error) */
    CGRT_ERR_OOM = 4
};

/* ---- data types on the boundary ---------------------------------------------------------------------------------- */

/* struct Ray, framework/include/ray.h:9-13 (origin, direction, t = max distance in / hit distance out), padded to 32 B
 * so a ray is two 128-bit loads. */
typedef struct cgrt_ray {
    float origin[3];
    float t;
    float direction[3];
    float pad;
} cgrt_ray;

/* HitInfo, src/ray_tracing.h:4-8, extended with what the parity checks need (triangle id, barycentrics).
 *   t      : hit distance (ray.t after intersect()); the input ray's t on a miss
 *   tri    : global triangle id (mesh order, then triangle order inside the mesh) of the closest triangle; -1 = miss;
 *            (-2 - s) when the closest primitive is sphere s (then `alpha` carries, bit-cast to int32, the id of the last
 *            accepted triangle or -1: the reference leaves hitInfo.material at that triangle's material,
 *            src/bounding_volume_hierarchy.cpp:878-879 + src/ray_tracing.cpp:154-157)
 *   alpha, beta, gamma : area-ratio barycentrics exactly as src/ray_tracing.cpp:94-96 computes them
 *   normal : interpolated shading normal flipped towards the ray (src/ray_tracing.cpp:97-106); untouched (0) on a miss */
typedef struct cgrt_hit {
    float t;
    int32_t tri;
    float alpha, beta, gamma;
    float normal[3];
} cgrt_hit;

/* Flattened Scene (src/scene.h:53-60) = Mesh list (src/mesh.h:12-35) + spheres (src/scene.h:36-40). */
typedef struct cgrt_scene_desc {
    int32_t n_meshes;
    const int32_t* mesh_vertex_count;   /* [n_meshes] */
    const int32_t* mesh_triangle_count; /* [n_meshes] */
    const float* vertices;              /* [sum v][6]  Vertex{p,n}        src/mesh.h:12-15 */
    const uint32_t* triangles;          /* [sum t][3]  mesh-local indices src/mesh.h:25    */
    const float* materials;             /* [n_meshes][8] kd, ks, shininess, transparency   src/mesh.h:17-23 */
    int32_t n_spheres;
    const float* spheres;               /* [n_spheres][12] center, radius, Material(8)     src/scene.h:36-40 */
} cgrt_scene_desc;

typedef struct cgrt_scene_options {
    int32_t device;        /* CUDA device ordinal this scene lives on */
    int32_t bvh_max_depth; /* reference literal 12 (src/bounding_volume_hierarchy.cpp:48); 0 = 12 */
    int32_t flags;         /* CGRT_SCENE_* */
    int32_t reserved[5];
} cgrt_scene_options;
/* Build the BVH on the host and keep it for introspection only (cgrt_bvh_*): no CUDA call is made, so the host builder
 * can be checked on machines without a GPU. Every query / render entry refuses such a scene with CGRT_ERR_NO_DEVICE. */
#define CGRT_SCENE_HOST_ONLY 1
/* Do not refine the reference leaves with culling sub-trees: every visited leaf is scanned triangle by triangle exactly as
 * intersectLeaf does (A/B switch for tests and profiling; results are identical either way). */
#define CGRT_SCENE_NO_SUBTREES 2
/* Do not use the speculative traversal (fast conservative tree + certification, see DESIGN.md): every ray takes the exact
 * reference-order traversal. A/B switch for tests and profiling; results are identical either way. */
#define CGRT_SCENE_EXACT_ONLY 4

/* PointLight, src/scene.h:42-45 */
typedef struct cgrt_point_light {
    float position[3];
    float color[3];
} cgrt_point_light;

/* Trackball private state (framework/include/trackball.h:47-53) + Window::aspectRatio (framework/src/window.cpp:334-337) */
typedef struct cgrt_camera {
    float fovy, aspect, dist;
    float look_at[3];
    float euler[3];
} cgrt_camera;

typedef struct cgrt_render_params {
    int32_t width, height;
    int32_t trace_limit; /* recursion limit, reference literal 2 (src/main.cpp:267) */
    int32_t rank, world; /* interleaved screen-tile partition over the GPUs of one box; world=1 -> whole frame */
    int32_t tile_w, tile_h; /* 0 = default 8x8 */
    int32_t flags;          /* CGRT_RENDER_* */
    int32_t reserved[4];
} cgrt_render_params;

/* kernel classes of the wavefront, in launch order within a level */
enum { CGRT_K_PRIMARY = 0, CGRT_K_BOUNCE = 1, CGRT_K_SHADOW = 2, CGRT_K_SHADE = 3, CGRT_K_CLASSES = 4 };
/* flags: bits 0..3 = record CUDA events around the kernels of that class (device time per class in the stats) */
#define CGRT_RENDER_PROFILE(cls) (1 << (cls))
#define CGRT_RENDER_PROFILE_ALL 0xF
/* run the counting variants of the traversal kernels: stats.box_tests / tri_tests receive the number of ray/AABB and
 * ray/triangle tests the REFERENCE traversal performs for the primary, bounce and shadow rays of the frame (shadow rays are
 * charged the reference's full closest-hit work, src/main.cpp:115). Same image; slower; meant for the roofline arithmetic. */
#define CGRT_RENDER_COUNT 0x100
/* world > 1 only: d_out of cgrt_render_device is a full [H][W][3] frame in Screen layout (typically the frame of rank 0,
 * mapped into this process with cgrt_peer_open) and the kernels store this rank's pixels straight at their final position -
 * the framebuffer "gather" is fused into the shading stores, no tile-major staging buffer, no assemble pass. */
#define CGRT_RENDER_SCREEN_LAYOUT 0x200

typedef struct cgrt_render_stats {
    uint64_t primary, primary_hit, shadow, bounce; /* logical rays, SURVEY.md §8(d) (shadow rays counted once) */
    uint64_t kernel_launches;                      /* kernels of this library launched by the call */
    uint64_t box_tests[3], tri_tests[3];           /* CGRT_RENDER_COUNT only: [primary, bounce, shadow] */
    float device_ms;                               /* CUDA-event time of the whole wavefront on its stream */
    float class_ms[4];                             /* CGRT_RENDER_PROFILE only: summed device time per kernel class */
    uint32_t class_launches[4];                    /* kernels launched per class */
    uint32_t replayed_closest, replayed_shadow;    /* rays the speculative traversal could not certify and handed to the
                                                      exact reference-order traversal (same results, more work) */
    uint32_t pipeline;                             /* which kernel set rendered the frame: 0 counting wavefront (CGRT_RENDER_COUNT),
                                                      1 path pipeline (scenes without a fast tree), 2 round pipeline,
                                                      3 persistent wavefront k_wave (chosen per frame, DESIGN 4.4;
                                                      CGRT_PIPELINE=wave|rounds forces one) */
} cgrt_render_stats;

typedef struct cgrt_scene cgrt_scene; /* opaque: flattened scene + BVH resident in HBM */

/* ---- library ------------------------------------------------------------------------------------------------------ */
int cgrt_version(void);
const char* cgrt_last_error(void);
/* number of visible CUDA devices (0 and CGRT_ERR_NO_DEVICE when there is none) */
int cgrt_device_count(int* count);

/* ---- scene + BVH ---------------------------------------------------------------------------------------------------
 * cgrt_scene_create replaces BoundingVolumeHierarchy::BoundingVolumeHierarchy(Scene*)
 * (src/bounding_volume_hierarchy.cpp:42-76 and build helpers :88-207, :235-389): host build with the reference split rule
 * on index ranges, then a 32-byte node layout + leaf-ordered SoA triangle buffers uploaded once. Meshes are copied
 * (bvh.cpp:50: later edits to meshes are not seen); lights and spheres can be replaced between renders because the
 * reference reads them live through Scene (src/main.cpp:835-876, bvh.cpp:878). */
int cgrt_scene_create(const cgrt_scene_desc* desc, const cgrt_scene_options* opt, cgrt_scene** out);
void cgrt_scene_destroy(cgrt_scene* s);
int cgrt_scene_set_lights(cgrt_scene* s, const cgrt_point_light* lights, int32_t n);
int cgrt_scene_set_spheres(cgrt_scene* s, const float* spheres /* [n][12] */, int32_t n);
/* Scene::sphericalLight (src/scene.h:47-51, preset CornellBoxSphericalLight src/scene.cpp:27-32) and the soft shadows of
 * shading() (src/main.cpp:168-218): per hit and spherical light 200 sample rays towards random points of the light's sphere
 * (randomUnitVector :46-59), the light's diffuse + specular term scaled by the fraction that arrives; spherical lights come
 * before the point lights in the sum. The reference draws the samples from std::random_device (non-deterministic): here a
 * counter-based generator keyed by (hit, light, sample, seed) - same distribution, reproducible frames; parity with the
 * reference is statistical by nature. lights[n][7] = position, radius, colour; n <= 64. Read at the next render. */
int cgrt_scene_set_spherical_lights(cgrt_scene* s, const float* lights /* [n][7] */, int32_t n, uint32_t seed);

/* BoundingVolumeHierarchy::numLevels() src/bounding_volume_hierarchy.cpp:214-224 */
int cgrt_bvh_num_levels(const cgrt_scene* s);
int cgrt_bvh_num_nodes(const cgrt_scene* s);
int64_t cgrt_scene_num_triangles(const cgrt_scene* s);
/* node export for debugDraw(level) (bvh.cpp:469-525) and for parity tests:
 * meta[n][5] = isLeaf, level, child0, child1, triangle count (leaves); aabb[n][6] = lower, upper */
int cgrt_bvh_export_nodes(const cgrt_scene* s, int32_t* meta, float* aabb);
/* global triangle ids of leaf `node` in the leaf's visiting order (intersectLeaf bvh.cpp:535-553); returns the count */
int cgrt_bvh_leaf_triangles(const cgrt_scene* s, int32_t node, int32_t* out, int32_t cap);

/* Structural self-check of the speculative traversal's tree (the conservative 8-wide tree over all triangles, see
 * DESIGN.md), evaluated on the host at build time: out[8] = wide nodes reachable, triangles reachable, triangles not reached
 * exactly once, vertices outside the box they hang under, depth in wide levels, certificate-chain errors, 1 if the scene has
 * such a tree (0 with CGRT_SCENE_NO_SUBTREES / CGRT_SCENE_EXACT_ONLY), reserved. Callable without a GPU. */
int cgrt_bvh_fast_tree_stats(const cgrt_scene* s, int64_t* out);

/* ---- queries -------------------------------------------------------------------------------------------------------
 * cgrt_intersect_closest replaces BoundingVolumeHierarchy::intersect(Ray&, HitInfo&) const
 * (src/bounding_volume_hierarchy.cpp:850-881) for a batch of n rays: same visiting order, same pruning, same accept/reject
 * arithmetic (strict build: -fmad=false, IEEE div/sqrt), then the sphere loop. counts (optional, [n][2]) receives the
 * number of ray/AABB and ray/triangle tests performed per ray (the quantities of SURVEY.md §8(d)).
 * Host-pointer form copies in/out around the kernel; *_device form takes device pointers and a cudaStream_t. */
int cgrt_intersect_closest(cgrt_scene* s, const cgrt_ray* rays, size_t n, cgrt_hit* hits, uint32_t* counts);
int cgrt_intersect_closest_device(cgrt_scene* s, const cgrt_ray* d_rays, size_t n, cgrt_hit* d_hits, uint32_t* d_counts,
                                  void* stream);
/* Any-hit form of the shadow query pointInShadow (src/main.cpp:104-135): occluded[i] = 1 iff the reference's closest hit
 * along rays[i] (searched with rays[i].t as initial bound) satisfies  t + eps < max_dist[i]; the traversal is the closest-hit
 * traversal with an early exit, so the answer is identical by construction. */
int cgrt_intersect_any(cgrt_scene* s, const cgrt_ray* rays, const float* max_dist, float eps, size_t n, uint8_t* occluded);
int cgrt_intersect_any_device(cgrt_scene* s, const cgrt_ray* d_rays, const float* d_max_dist, float eps, size_t n,
                              uint8_t* d_occluded, void* stream);
/* intersectRayWithShape(const Mesh&, Ray&, HitInfo&) src/ray_tracing.cpp:202-213 applied to every mesh of the scene in
 * order: brute force over all triangles (the reference's own cross-check of the BVH). */
int cgrt_intersect_brute(cgrt_scene* s, const cgrt_ray* rays, size_t n, cgrt_hit* hits);

/* ---- the free functions of src/ray_tracing.h:10-20, batched (element i of every array belongs to call i) ---------------- */
/* intersectRayWithShape(const AxisAlignedBox&, Ray&)  src/ray_tracing.cpp:162-200 ; boxes[n][6] = lower, upper */
int cgrt_ray_aabb(int device, const float* boxes, const cgrt_ray* rays, size_t n, uint8_t* hit, float* t);
/* intersectRayWithTriangle  src/ray_tracing.cpp:86-114 ; tris[n][18] = v0 v1 v2 n0 n1 n2 ; out[i].tri = 1 on hit, 0 on miss */
int cgrt_ray_triangle(int device, const float* tris, const cgrt_ray* rays, size_t n, cgrt_hit* out);
/* intersectRayWithPlane  src/ray_tracing.cpp:40-72 ; planes[n][4] = normal, D */
int cgrt_ray_plane(int device, const float* planes, const cgrt_ray* rays, size_t n, uint8_t* hit, float* t);
/* trianglePlane  src/ray_tracing.cpp:74-82 ; tris[n][9] -> planes[n][4] */
int cgrt_triangle_plane(int device, const float* tris, size_t n, float* planes);
/* pointInTriangle  src/ray_tracing.cpp:23-38 ; in[n][15] = v0 v1 v2 n p */
int cgrt_point_in_triangle(int device, const float* in, size_t n, uint8_t* inside);
/* intersectRayWithShape(const Sphere&, Ray&, HitInfo&)  src/ray_tracing.cpp:118-158 ; spheres[n][4] ; out[n][5] = t, hit, normal */
int cgrt_ray_sphere(int device, const float* spheres, const cgrt_ray* rays, size_t n, float* out);

/* ---- rendering -----------------------------------------------------------------------------------------------------
 * Trackball::generateRay over the pixel grid of renderRayTracing (framework/src/trackball.cpp:92-103, src/main.cpp:691-694);
 * rays[H*W], pixel (x,y) at y*W+x. */
int cgrt_generate_rays(int device, const cgrt_camera* cam, int32_t width, int32_t height, cgrt_ray* rays);

/* cgrt_render replaces renderRayTracing(scene, camera, bvh, screen) (src/main.cpp:648-720, non-AA/non-bloom branch) and the
 * recursion below it (getFinalColor/trace/shade/shading/pointInShadow, src/main.cpp:61-310) as a wavefront of kernels:
 * ray generation + closest hit, any-hit shadow rays (one per hit per light), shading, compacted reflection-bounce queues.
 * rgb receives the float framebuffer in Screen's layout (row H-1-y, src/screen.cpp:30-36), [H][W][3].
 * With world > 1 the call renders only this rank's interleaved tiles; cgrt_render (host form) then returns only those
 * pixels (others untouched); use the *_device form + cgrt_assemble_tiles for the gathered multi-GPU path. */
int cgrt_render(cgrt_scene* s, const cgrt_camera* cam, const cgrt_render_params* p, float* rgb, cgrt_render_stats* stats);
/* world==1: d_out = frame [H][W][3] (Screen layout).  world>1: d_out = this rank's tile-major buffer of
 * cgrt_tile_buffer_floats(p) floats (tiles owned by the rank, in increasing global tile id, tile_h*tile_w*3 floats each,
 * padded to the largest per-rank tile count so that all ranks send equal sizes). Asynchronous on `stream`;
 * stats (optional) are valid after the stream is synchronised and cgrt_render_collect_stats is called. */
int cgrt_render_device(cgrt_scene* s, const cgrt_camera* cam, const cgrt_render_params* p, float* d_out, void* stream);
/* Several camera views of one scene in one call (turntables, stereo pairs, sets of viewpoints, motion-blur cameras): the
 * n_views cameras share the width, height, trace limit and lights of p and render as ONE frame of n_views x width x height
 * pixel slots, so the views share the per-frame costs and the tail of the last mirror chains. The views are interleaved tile by
 * tile in the centre-out tile order (DESIGN.md 4.4).
 *   Output   rgb / d_out = [n_views][H][W][3], each view in Screen layout (row H-1-y).
 *   Equality view v is bit for bit the frame cgrt_render(s, &cams[v], p, ...) returns, with spherical-light soft shadows too;
 *            the ray statistics are the sums of those frames'.
 *   Pipeline the kernel set is chosen as for one frame of that many pixel slots (cgrt_render_stats::pipeline; CGRT_PIPELINE
 *            forces it as for cgrt_render). stats: sums over the views; kernel_launches counts the launches of the whole call.
 *   Limits   a batch has the limits of one frame of its total size (n_views x width x height <= 2^28, the persistent
 *            wavefront's 30-bit ray tickets); the scene's reserved buffers grow with the batch and stay, as for a large frame.
 *   Refused  (CGRT_ERR_INVALID, before any CUDA call): null cams / rgb / d_out, n_views outside 1..1024, n_views x width x
 *            height > 2^28, pixel slots of whole tiles (n_views x tiles x tile_w x tile_h) >= 2^31, world != 1, any flag
 *            but CGRT_RENDER_PROFILE_*.
 * The _device form is asynchronous on `stream`; its statistics come from cgrt_render_collect_stats after the stream has been
 * synchronised, as for cgrt_render_device.
 * Measured on one B200 (1000 W power limit), device time per view for 8 views batched vs one by one: C1 (Cornell 512^2, trace
 * limit 2) 0.034 vs 0.119 ms, C2 (monkey 1080p, limit 1) 0.229 vs 0.300 ms, C3 (1080p, limit 5) 0.736 vs 0.971 ms; one view
 * costs what cgrt_render does (DESIGN.md 4.4). */
int cgrt_render_views(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p, float* rgb,
                      cgrt_render_stats* stats);
int cgrt_render_views_device(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p,
                             float* d_out, void* stream);
/* Per-pixel buffers of a frame ("AOVs", a G-buffer): what each pixel's primary ray hit, for picking, depth-based passes and
 * masks. Any pointer may be NULL: that buffer is not produced. */
typedef struct cgrt_aov_buffers {
    float* depth;   /* [n_views][H][W]    t of the primary ray's closest hit; the ray's t (FLT_MAX) on a miss */
    int32_t* tri;   /* [n_views][H][W]    cgrt_hit.tri of that hit: global triangle id, -1 miss, -2 - s sphere s */
    float* normal;  /* [n_views][H][W][3] cgrt_hit.normal of that hit (shading normal towards the ray); 0 on a miss */
    uint8_t* hits;  /* [n_views][H][W]    trace() levels of the pixel's path that hit: 0 = primary miss, .. trace_limit */
} cgrt_aov_buffers;
/* cgrt_render_views with per-pixel buffers: the frame's renderer keeps the hit distance and the hit's id in its level-0 hit
 * records, and one small pass after the frame writes the requested buffers from them (DESIGN.md 4.5).
 *   Layout   every buffer is in Screen layout (row H-1-y), view after view, like rgb; n_views = 1 is a single frame.
 *   Equality rgb is bit for bit what cgrt_render_views returns for the same arguments; so are the stats, except
 *            kernel_launches, which also counts the AOV pass (device_ms covers it), and the reported pipeline is the same.
 *            Per pixel, depth, tri and normal are bit for bit the t, tri and normal cgrt_intersect_closest returns for that
 *            pixel's ray from cgrt_generate_rays(cams[v]).
 *   Limit 0  the frame traces nothing: every pixel reports a miss and hits is 0.
 *   Refused  (CGRT_ERR_INVALID, before any CUDA call): everything cgrt_render_views refuses (so whole frames only, no
 *            CGRT_RENDER_COUNT, no CGRT_RENDER_SCREEN_LAYOUT), a null aov, an aov whose four pointers are all NULL.
 * The host form copies rgb and each requested buffer back on the scene's stream and synchronises once. The _device form takes
 * device pointers and is asynchronous on `stream`; its statistics come from cgrt_render_collect_stats.
 * Measured on one B200 (1000 W power limit): the pass adds 0.018-0.024 ms to a 1080p frame (C3, trace limit 5: 1.072 vs
 * 1.095 ms, DESIGN.md 4.5). */
int cgrt_render_aovs(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p, float* rgb,
                     const cgrt_aov_buffers* aov, cgrt_render_stats* stats);
int cgrt_render_aovs_device(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p,
                            float* d_rgb, const cgrt_aov_buffers* d_aov, void* stream);
/* Mirror paths and shadow factors: every level of each pixel's getFinalColor recursion (the ray trace(level) cast, what it hit
 * and where) and, at each hit, each light's shadow factor. Any pointer may be NULL: that buffer is not produced. */
typedef struct cgrt_path_buffers {
    cgrt_ray* ray;       /* [n_levels][n_views][H][W]           the ray trace(level) cast */
    float* depth;        /* [n_levels][n_views][H][W]           t of its closest hit */
    int32_t* tri;        /* [n_levels][n_views][H][W]           cgrt_hit.tri of that hit */
    float* normal;       /* [n_levels][n_views][H][W][3]        cgrt_hit.normal of that hit */
    float* position;     /* [n_levels][n_views][H][W][3]        the shading point of the hit */
    float* visibility;   /* [n_levels][n_views][H][W][n_lights] each light's shadow factor at the hit */
} cgrt_path_buffers;
/* cgrt_render_views with the frame's mirror paths: the frame keeps one hit record per pixel and level, one lit flag per record
 * and point light and (round pipeline) one soft-shadow fraction per record and spherical light; one pass after the frame walks
 * each pixel's records and writes the requested buffers (DESIGN.md 4.5).
 *   Layout   every buffer is in Screen layout (row H-1-y), view after view, level after level: level l of pixel (x, y) of view
 *            v is element (l * n_views + v) * H * W + (H-1-y) * W + x. Lights come in the order of cgrt_render_lights: the
 *            point lights (cgrt_scene_set_lights order), then the spherical lights.
 *   Equality rgb is bit for bit what cgrt_render_views returns for the same arguments; so are the stats, except
 *            kernel_launches, which also counts the pass (device_ms covers it).
 *   Contract for level l of pixel (x, y) of view v:
 *            (1) ray: level 0 is the ray of cgrt_generate_rays(cams[v]) whenever trace_limit > 0. Level l >= 1 exists when
 *            level l-1 hit, that hit's material has ks.z > 0.01 and l < trace_limit: it is shade()'s reflection ray off the
 *            level l-1 hit, origin P + 0.001 r, direction r = normalize(reflect(D, N)), t = |D| with D the incoming direction
 *            (src/main.cpp:246-256). A level for which the recursion cast no ray (a miss or a non-mirror before it, the trace
 *            limit, limit 0) is all +0 in ray.
 *            (2) hit: depth, tri and normal are bit for bit what cgrt_intersect_closest returns for ray[l], so a miss reports
 *            the ray's own t (FLT_MAX for a primary ray), tri -1 and normal 0. A level without a ray reports FLT_MAX, -1 and
 *            0. Level 0 is therefore bit for bit the depth / tri / normal of cgrt_render_aovs, limit 0 included.
 *            (3) position: the hit's shading point origin + t * direction (src/main.cpp:164); 0 where the level did not hit.
 *            (4) visibility: the factor that level's shading() applied to each light's diffuse + specular term: 1 or 0 for a
 *            point light (lit, or pointInShadow), k / 200 for a spherical light whose k of 200 samples arrived (the frame's
 *            own samples, cgrt_scene_set_spherical_lights); 0 where the level did not hit.
 *            (5) every level of every pixel is written on every call: levels past a pixel's path hold no data of an earlier
 *            frame.
 *   Refused  (CGRT_ERR_INVALID, before any CUDA call): everything cgrt_render_views refuses (so whole frames only, no
 *            CGRT_RENDER_COUNT, no CGRT_RENDER_SCREEN_LAYOUT), a null paths or one whose six pointers are all NULL, n_levels
 *            outside 1..max(trace_limit, 1), n_levels x n_views x W x H > 2^28, a requested visibility with n_levels x n_views
 *            x W x H x n_lights > 2^28, and n_lights other than the scene's point plus spherical lights (checked again when the
 *            frame reads the lights, which may change in between).
 * The host form stages the buffers on the device, copies rgb and each requested buffer back on the scene's stream and
 * synchronises once. The _device form takes device pointers and is asynchronous on `stream`; its statistics come from
 * cgrt_render_collect_stats.
 * Measured on one B200 (1000 W power limit), every buffer, n_levels = trace limit: the pass adds 0.22-0.28 ms to a 1080p view
 * (C3, trace limit 5: 1.076 vs 1.293 ms for one view, 0.738 vs 1.018 ms per view for 8; DESIGN.md 4.5). */
int cgrt_render_paths(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p, int32_t n_levels,
                      int32_t n_lights, float* rgb, const cgrt_path_buffers* paths, cgrt_render_stats* stats);
int cgrt_render_paths_device(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p,
                             int32_t n_levels, int32_t n_lights, float* d_rgb, const cgrt_path_buffers* d_paths, void* stream);
/* Light groups: cgrt_render_views with each group's share of every pixel in its own buffer, so that a light's colour can be
 * edited (relit) without tracing the frame again. One pass after the frame shades the hit records, lit flags and soft-shadow
 * fractions the frame left once per group, with the frame's arithmetic, restricted to the group's lights (DESIGN.md 4.5).
 *   Groups   light_group[n_lights] (host memory, read before the call returns) gives each light's group: the scene's point
 *            lights in cgrt_scene_set_lights order, then its spherical lights in cgrt_scene_set_spherical_lights order. An
 *            entry is a group 0..n_groups-1, or -1: the light is in no group (it lights rgb, no group buffer). n_groups is
 *            1..64; a group without lights is +0 everywhere.
 *   Layout   groups is [n_groups][n_views][H][W][3], each view in Screen layout (row H-1-y) like rgb.
 *   Equality rgb is bit for bit what cgrt_render_views returns for the same arguments; so are the stats, except
 *            kernel_launches, which also counts the group pass (device_ms covers it).
 *   Exact    (1) group g of view v is bit for bit view v of cgrt_render_views with every light outside g given colour
 *            (0,0,0), positions, radii, the spherical-light seed and the order of the lights unchanged (soft-shadow samples
 *            are keyed by the light's index, which does not change). (2) So a group holding every light equals rgb bit for
 *            bit. Reason: a light of colour 0 adds +-0 to a sum that is never -0, and the pass skips it. Precondition:
 *            finite material values and light colours, and shininess >= 0 (every preset and fixture meets it).
 *   Approx.  (3) the sum of the groups plus the share of the lights in no group equals rgb up to float reassociation
 *            only: a pixel sums its lights in one order, the groups split that sum. Scaling a group buffer by a colour gain
 *            likewise matches a render with that light colour scaled up to rounding.
 *   Limit 0  the frame traces nothing: every group buffer is +0.
 *   Refused  (CGRT_ERR_INVALID, before any CUDA call): everything cgrt_render_views refuses (so whole frames only, no
 *            CGRT_RENDER_COUNT, no CGRT_RENDER_SCREEN_LAYOUT), a null light_group or groups, n_groups outside 1..64,
 *            n_groups x n_views x W x H > 2^28, n_lights other than the scene's point plus spherical lights (checked again
 *            when the frame reads the lights, which may change in between), and an entry outside -1..n_groups-1.
 * The host form stages the group buffers on the device, copies rgb and them back on the scene's stream and synchronises once.
 * The _device form takes device pointers and is asynchronous on `stream`; its statistics come from cgrt_render_collect_stats.
 * Measured on one B200 (1000 W power limit): one group adds 0.034-0.050 ms to a 1080p frame (C3, trace limit 5: 1.077 vs
 * 1.127 ms, DESIGN.md 4.5). */
int cgrt_render_lights(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p,
                       const int32_t* light_group, int32_t n_lights, int32_t n_groups, float* rgb, float* groups,
                       cgrt_render_stats* stats);
int cgrt_render_lights_device(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p,
                              const int32_t* light_group, int32_t n_lights, int32_t n_groups, float* d_rgb, float* d_groups,
                              void* stream);
int cgrt_render_collect_stats(cgrt_scene* s, cgrt_render_stats* stats);
/* renderRayTracing's optional passes around the path (UI toggles, default off, src/main.cpp:33-35):
 *   CGRT_EFFECT_ANTIALIAS   src/main.cpp:663-687: four rays per pixel = the pixel-corner rays of the (2W x 2H) frame, summed in
 *                           the reference's order and divided by level * 2.5 = 5 (sic). The reference never initialises its
 *                           accumulator `color` (undefined behaviour); this implementation starts it at zero.
 *   CGRT_EFFECT_MOTION_BLUR blurEffect, src/main.cpp:318-584: the frames of 15 cameras whose look-at point is REPLACED by
 *                           (0.01 k, 0, 0), k = 1..15, added in that order and divided by 16; as in the reference it overwrites
 *                           whatever the pixel loop drew, so it wins over CGRT_EFFECT_ANTIALIAS.
 *   CGRT_EFFECT_BLOOM       bloomEffect, src/main.cpp:586-628 with the bookkeeping of :698-705: pixels whose colour sums to more
 *                           than 1 are kept (else black), every entry is then replaced IN PLACE, in scan order, by the average of its
 *                           clipped 21 x 21 neighbourhood (so it sees the new values below / left of it and the old ones elsewhere),
 *                           and the pixel becomes that average + the ray-traced colour. Bit-exact to the sequential loop: the
 *                           recurrence is run as a wavefront, one warp per image row, rows 11 columns apart, every entry's terms
 *                           added in the reference's order. With CGRT_EFFECT_MOTION_BLUR the running sum starts from
 *                           colour + (bloom + colour) as in the reference (:700, :622, :581). Not offered together with
 *                           CGRT_EFFECT_ANTIALIAS (the reference's combination thresholds on an uninitialised accumulator).
 * world must be 1. stats (optional): sums over the rendered frames. */
#define CGRT_EFFECT_ANTIALIAS 1
#define CGRT_EFFECT_MOTION_BLUR 2
#define CGRT_EFFECT_BLOOM 4
int cgrt_render_effects(cgrt_scene* s, const cgrt_camera* cam, const cgrt_render_params* p, int32_t effects, float* rgb,
                        cgrt_render_stats* stats);
/* The effects of cgrt_render_effects for several views of one scene in one call, on the caller's stream (turntables, datasets,
 * a UI that keeps its frames on the GPU). Every render inside the call is one frame of a views batch (cgrt_render_views) of at
 * most 2^25 pixel slots: the 15 motion-blur cameras of as many whole views as fit (a view whose 15 cameras do not fit, e.g. 4K,
 * spreads them over several batches in order), the un-shifted views of bloom, the 2W x 2H views of anti-aliasing. One kernel
 * adds each batch's motion-blur frames into the views' running sums, one bloom pass runs the row recurrences of all views.
 *   Output   rgb / d_out = [n_views][H][W][3], each view in Screen layout (row H-1-y).
 *   Equality view v is bit for bit what cgrt_render_effects(s, &cams[v], p, effects, ...) returns, for every accepted
 *            combination of effects, with spherical-light soft shadows too, and at trace limit 0. effects == 0 is
 *            cgrt_render_views.
 *   Stats    primary, primary_hit, shadow and bounce are the sums of those calls' statistics; kernel_launches counts every
 *            launch of this call; device_ms runs from the call's first event to its last; pipeline is that of the last
 *            render; no per-class times (there is no profiling mode).
 *   Refused  (CGRT_ERR_INVALID): what cgrt_render_effects refuses for one view (unknown effect bits, bloom with
 *            anti-aliasing, 4 x width x height > 2^28 for anti-aliasing, a frame too tall for the bloom pass) and, before any
 *            CUDA call, null cams / rgb / d_out, n_views outside 1..1024, n_views x width x height > 2^28, world != 1, any
 *            p->flags other than 0.
 * The scene's effect buffers grow with the call and stay. The _device form is asynchronous on `stream`: after the stream has
 * synchronised, cgrt_render_collect_stats returns the sums above for the whole call (CGRT_ERR_CUDA if the persistent
 * wavefront's watchdog fired in any of its renders). Frames of one scene are enqueued on one stream or ordered by the caller.
 * The host form is the device form on the scene's stream, one copy to rgb and one synchronisation. */
int cgrt_render_effects_views(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p,
                              int32_t effects, float* rgb, cgrt_render_stats* stats);
int cgrt_render_effects_views_device(cgrt_scene* s, const cgrt_camera* cams, int32_t n_views, const cgrt_render_params* p,
                                     int32_t effects, float* d_out, void* stream);
/* Streaming form of cgrt_render for hosts that render frame after frame (the reference re-renders every UI frame in
 * ViewMode::RayTracing, src/main.cpp:907-914): cgrt_render_submit enqueues the frame (per-frame camera + lights upload, the
 * kernels, the device->host copy into rgb_host) and returns; up to two frames are in flight, so the copy of frame k overlaps
 * the kernels of frame k+1 (the call blocks only until frame k-2 has been delivered). cgrt_render_wait returns when every
 * submitted frame has arrived. rgb_host should be page-locked (cgrt_host_alloc_pinned) and must stay valid until delivery;
 * frames are delivered in submission order. world must be 1. Same pixels as cgrt_render. */
int cgrt_render_submit(cgrt_scene* s, const cgrt_camera* cam, const cgrt_render_params* p, float* rgb_host);
int cgrt_render_wait(cgrt_scene* s);
size_t cgrt_tile_buffer_floats(const cgrt_render_params* p);
/* global ids (ty * tilesX + tx, tilesX = ceil(width / tile_w)) of the tiles `rank` owns, increasing; returns the count
 * (-1 on bad arguments). Pure host arithmetic: callable without a GPU. */
int cgrt_tile_list(const cgrt_render_params* p, int32_t rank, int32_t* out, int32_t cap);
/* rank 0 after the gather: d_gathered = [world][cgrt_tile_buffer_floats] -> d_frame [H][W][3] in Screen layout */
int cgrt_assemble_tiles(int device, const cgrt_render_params* p, const float* d_gathered, float* d_frame, void* stream);
/* Screen::writeBitmapToFile quantisation (src/screen.cpp:38-49): clamp to [0,1], *255, truncate; rgba8[H*W*4], alpha 255 */
int cgrt_quantize_rgba8(int device, const float* d_frame, size_t n_pixels, uint8_t* d_rgba8, void* stream);

/* ---- multi-GPU frame hand-off over NVLink peer memory (one process per GPU) ------------------------------------------
 * The path shards by pixels (src/main.cpp:656-697 has no inter-pixel dependence); its single exchange step is the
 * framebuffer. Instead of a gather collective, every rank renders with CGRT_RENDER_SCREEN_LAYOUT into the frame of rank 0,
 * which rank 0 exports and the others map:
 *   rank 0 : cgrt_device_malloc(frame), cgrt_peer_export -> 64-byte handle, sent to the peers by the host's own plumbing
 *   rank r : cgrt_peer_open(handle) -> device pointer valid in this process (NVLink / NVSwitch peer mapping)
 * Completion and buffer reuse are 32-bit sequence numbers in device memory (local or peer-mapped):
 *   cgrt_flag_signal : after everything enqueued on `stream` so far, store `seq` to each of the n flags (system-scope release)
 *   cgrt_flag_wait   : `stream` does not proceed until all n consecutive flags are >= seq (wrap-safe); gives up after
 *                      timeout_ms and increments *d_status (optional) so that a lost peer cannot hang the GPU. */
#define CGRT_IPC_HANDLE_BYTES 64
int cgrt_peer_export(int device, void* d_ptr, uint8_t* handle /* [CGRT_IPC_HANDLE_BYTES] */);
int cgrt_peer_open(int device, const uint8_t* handle, void** out);
int cgrt_peer_close(int device, void* p);
int cgrt_flag_signal(int device, uint32_t* const* d_flags, int32_t n, uint32_t seq, void* stream);
int cgrt_flag_wait(int device, const uint32_t* d_flags, int32_t n, uint32_t seq, uint32_t timeout_ms, uint32_t* d_status,
                   void* stream);

/* ---- device memory helpers for hosts that do not link the CUDA runtime themselves (ctypes / C callers) ---------------- */
int cgrt_device_malloc(int device, size_t bytes, void** out);
int cgrt_device_free(int device, void* p);
int cgrt_host_alloc_pinned(size_t bytes, void** out);
int cgrt_host_free_pinned(void* p);
int cgrt_memcpy_h2d(int device, void* dst, const void* src, size_t bytes);
int cgrt_memcpy_d2h(int device, void* dst, const void* src, size_t bytes);
int cgrt_device_synchronize(int device);
int cgrt_memset_device(int device, void* p, int value, size_t bytes, void* stream);
int cgrt_memcpy_d2h_async(int device, void* dst, const void* src, size_t bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CGRT_B200_H */
