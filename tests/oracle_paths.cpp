// TEST INFRASTRUCTURE for tests/test_render_paths.py: the mirror paths of cgrt_render_paths, computed by the restatement.
// The restatement (oracle/cgrt_oracle.cpp) is included whole, so its camera, intersect() and Tracer run unchanged; this file only
// adds one export. tests/test_render_paths.py compiles it into a temporary directory with the oracle's flags.
#include "../oracle/cgrt_oracle.cpp"

namespace {
// Tracer::trace / shade / shading (src/main.cpp:160-295) with the same arithmetic in the same order, that also record each
// level's ray, hit, shading point and per-light shadow factors of one pixel. Buffers are [nLevels][H][W](...); the caller has
// filled every level of the pixel as "no ray".
struct PathWalk {
    Tracer& tr;
    const OrcScene* os;
    int nLevels;
    size_t px, i; // pixels of one level, this pixel's index
    float *rays, *depth, *normal, *position, *visibility;
    int32_t* tri;

    vec3 shading(int level, Ray& ray, HitInfo& hitInfo)
    { // Tracer::shading, recording the factor of each light: point lights, then spherical lights
        const Scene& sc = *tr.bvh->scene;
        const size_t nPoint = sc.pointLights.size();
        float* vis = level < nLevels ? visibility + ((size_t)level * px + i) * (nPoint + sc.sphericalLight.size()) : nullptr;
        vec3 pointOn = ray.origin + ray.direction * ray.t;
        vec3 result = V(0, 0, 0);
        for (size_t k = 0; k < sc.sphericalLight.size(); k++) {
            const SphericalLight& spherical = sc.sphericalLight[k];
            const PointLight light = {spherical.position, spherical.color};
            const vec3 fromPosToLight = normalize(light.position - pointOn);
            vec3 diffuse = tr.diffuseOneLight(ray, light, fromPosToLight, hitInfo);
            vec3 specular = tr.specularOneLight(ray, light, fromPosToLight, hitInfo);
            float softShadowCounter = 0.0f;
            for (int s = 1; s <= 200; s++) {
                vec3 randomPointOnSphere = spherical.position + spherical.radius * tr.randomUnitVector();
                Ray newRay;
                newRay.origin = pointOn + (float)(0.001) * (normalize(randomPointOnSphere - pointOn));
                newRay.direction = normalize(randomPointOnSphere - pointOn);
                newRay.t = length(newRay.origin - randomPointOnSphere);
                HitInfo newHitInfo = Tracer::freshHitInfo();
                float lightT = length(newRay.origin - randomPointOnSphere);
                if (!intersect(*tr.bvh, newRay, newHitInfo)) softShadowCounter += 1.0f;
                else if (newRay.t > lightT) softShadowCounter += 1.0f;
            }
            softShadowCounter = softShadowCounter / 200.0f;
            if (vis) vis[nPoint + k] = softShadowCounter;
            result = result + diffuse * softShadowCounter;
            result = result + specular * softShadowCounter;
        }
        for (size_t k = 0; k < nPoint; k++) {
            const PointLight& light = sc.pointLights[k];
            const vec3 fromPosToLight = normalize(light.position - pointOn);
            const bool shadowed = tr.pointInShadow(pointOn, light);
            if (vis) vis[k] = shadowed ? 0.0f : 1.0f;
            if (shadowed) continue;
            vec3 diffuse = tr.diffuseOneLight(ray, light, fromPosToLight, hitInfo);
            vec3 specular = tr.specularOneLight(ray, light, fromPosToLight, hitInfo);
            result = result + diffuse;
            result = result + specular;
        }
        if (level < nLevels) {
            float* p = position + 3 * ((size_t)level * px + i);
            p[0] = pointOn.x; p[1] = pointOn.y; p[2] = pointOn.z;
        }
        return result;
    }
    void shade(int level, Ray ray, vec3& color, HitInfo& hitInfo)
    { // Tracer::shade
        vec3 directColor = shading(level, ray, hitInfo);
        if (hitInfo.material.ks.z <= 0.01f) {
            color = directColor;
            return;
        }
        vec3 fromCamToPos = ray.direction;
        vec3 reflected = normalize(reflect(fromCamToPos, hitInfo.normal));
        Ray reflectedRay = {ray.origin + ray.direction * ray.t, reflected, length(fromCamToPos)};
        float epsilon = 0.001;
        reflectedRay.origin = reflectedRay.origin + epsilon * reflectedRay.direction;
        vec3 reflectedColor;
        trace(level + 1, reflectedRay, reflectedColor);
        color = directColor + reflectedColor * hitInfo.material.ks;
    }
    void trace(int level, Ray ray, vec3& color)
    { // Tracer::trace: the level's ray, then its hit as orc_intersect reports it (canonical id, -2 - s for sphere s)
        if (level >= tr.traceLimit) {
            color = V(0, 0, 0);
            return;
        }
        const Ray in = ray;
        HitInfo hitInfo = Tracer::freshHitInfo();
        int sphere = -1;
        const bool hit = intersect(*tr.bvh, ray, hitInfo, &sphere);
        if (level < nLevels) {
            const size_t j = (size_t)level * px + i;
            float* r = rays + 8 * j;
            r[0] = in.origin.x; r[1] = in.origin.y; r[2] = in.origin.z; r[3] = in.t;
            r[4] = in.direction.x; r[5] = in.direction.y; r[6] = in.direction.z; r[7] = 0.0f;
            float rec[8];
            fillHit(os, in, ray, hit, hitInfo, sphere, rec);
            int32_t id;
            std::memcpy(&id, &rec[1], 4);
            if (hit && sphere >= 0) id = -2 - sphere;
            depth[j] = rec[0];
            tri[j] = id;
            normal[3 * j] = rec[5]; normal[3 * j + 1] = rec[6]; normal[3 * j + 2] = rec[7];
        }
        if (hit) shade(level, ray, color, hitInfo);
        else color = V(0, 0, 0);
    }
};
} // namespace

extern "C" {

// orc_render's pixel loop walked by PathWalk: rgb (Screen layout) and, per level l < nLevels of each pixel, in Screen layout
// [nLevels][H][W]: ray[8] (origin, t, direction, 0; all 0 where the recursion cast no ray), depth / tri / normal of that ray's
// hit (FLT_MAX, -1, 0 without a ray), position (the shading point, 0 where the level did not hit) and visibility[nLights]
// (point lights, then spherical lights: 1 / 0 lit / in shadow, k / 200 arriving samples; 0 where the level did not hit).
void orc_render_paths(void* h, const CameraDesc* c, int W, int H, int traceLimit, int nLevels, float* rgb, float* ray, float* depth,
                      int32_t* tri, float* normal, float* position, float* visibility, int nthreads)
{
    OrcBVH* b = (OrcBVH*)h;
    const size_t pix = (size_t)W * H;
    const size_t nLights = b->bvh.scene->pointLights.size() + b->bvh.scene->sphericalLight.size();
    const size_t n = pix * nLevels;
    std::fill(ray, ray + 8 * n, 0.0f);
    std::fill(depth, depth + n, std::numeric_limits<float>::max());
    std::fill(tri, tri + n, -1);
    std::fill(normal, normal + 3 * n, 0.0f);
    std::fill(position, position + 3 * n, 0.0f);
    std::fill(visibility, visibility + nLights * n, 0.0f);
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
        PathWalk walk{tr, b->os, nLevels, pix, 0, ray, depth, normal, position, visibility, tri};
#ifdef _OPENMP
#pragma omp for
#endif
        for (int y = 0; y < H; y++) {
            for (int x = 0; x != W; x++) {
                float px = float(x) / W * 2.0f - 1.0f;
                float py = float(y) / H * 2.0f - 1.0f;
                Ray cameraRay = cam.generateRay(px, py);
                walk.i = (size_t)(H - 1 - y) * W + x;
                vec3 color;
                walk.trace(0, cameraRay, color);
                rgb[3 * walk.i] = color.x; rgb[3 * walk.i + 1] = color.y; rgb[3 * walk.i + 2] = color.z;
            }
        }
    }
}

} // extern "C"
