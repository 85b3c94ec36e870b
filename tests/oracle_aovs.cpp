// TEST INFRASTRUCTURE for tests/test_render_aovs.py: the per-pixel buffers of cgrt_render_aovs, computed by the restatement.
// The restatement (oracle/cgrt_oracle.cpp) is included whole, so its camera, intersect() and Tracer run unchanged; this file only
// adds one export. tests/test_render_aovs.py compiles it into a temporary directory with the oracle's flags.
#include "../oracle/cgrt_oracle.cpp"

extern "C" {

// orc_render's pixel loop (no duplicate shading) that also records per pixel, in Screen layout (row H-1-y):
//   depth / tri / normal: the primary ray's closest hit as orc_intersect reports it on the ray of orc_generate_rays (canonical
//                         triangle id, -2 - s for sphere s); a miss at trace limit 0, which casts no ray
//   hits                : the trace() calls of the pixel's path that reached shade(). Each shade() casts one shadow ray per point
//                         light and 200 per spherical light (RenderCounters::shadow), so the count is the pixel's shadow rays
//                         over that number.
// Returns 0, or -1 for a scene without lights (the count cannot be read off the shadow rays).
int orc_render_aovs(void* h, const CameraDesc* c, int W, int H, int traceLimit, float* rgb, float* depth, int32_t* tri,
                    float* normal, uint8_t* hits, int nthreads)
{
    OrcBVH* b = (OrcBVH*)h;
    const uint64_t perShade = b->bvh.scene->pointLights.size() + 200 * (uint64_t)b->bvh.scene->sphericalLight.size();
    if (perShade == 0) return -1;
    Camera cam = makeCamera(c);
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#pragma omp parallel num_threads(nthreads)
#endif
    {
        RenderCounters rc;
        g_cnt = Counters();
        Tracer tr{&b->bvh, traceLimit, false, &rc, true};
        int tid = 0;
#ifdef _OPENMP
        tid = omp_get_thread_num();
#endif
        std::mt19937 gen(g_softSeed * 7919u + (unsigned)tid);
        tr.rng = &gen;
#ifdef _OPENMP
#pragma omp for
#endif
        for (int y = 0; y < H; y++) {
            for (int x = 0; x != W; x++) {
                float px = float(x) / W * 2.0f - 1.0f;
                float py = float(y) / H * 2.0f - 1.0f;
                Ray cameraRay = cam.generateRay(px, py);
                const size_t i = (size_t)(H - 1 - y) * W + x;
                Ray ray = cameraRay;
                HitInfo hi = Tracer::freshHitInfo();
                int sphere = -1;
                const bool hit = traceLimit > 0 && intersect(b->bvh, ray, hi, &sphere);
                float rec[8];
                fillHit(b->os, cameraRay, ray, hit, hi, sphere, rec);
                int32_t id;
                std::memcpy(&id, &rec[1], 4);
                if (hit && sphere >= 0) id = -2 - sphere;
                depth[i] = rec[0];
                tri[i] = id;
                normal[3 * i] = rec[5]; normal[3 * i + 1] = rec[6]; normal[3 * i + 2] = rec[7];
                const uint64_t before = rc.shadow;
                vec3 color;
                tr.trace(0, cameraRay, color);
                hits[i] = (uint8_t)((rc.shadow - before) / perShade);
                rgb[3 * i] = color.x; rgb[3 * i + 1] = color.y; rgb[3 * i + 2] = color.z;
            }
        }
    }
    return 0;
}

} // extern "C"
