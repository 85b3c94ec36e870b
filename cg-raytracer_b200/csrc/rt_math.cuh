// Strict fp32 vector math + the reference's intersection predicates as device functions.
// Build flags that this file relies on (see __graft_entry__.build): -fmad=false (no FMA contraction),
// default -prec-div=true -prec-sqrt=true -ftz=false, no --use_fast_math. Expression trees follow glm 0.9.9.8's scalar
// paths and the reference source literally (SURVEY.md Appendix A); never fminf/fmaxf/rsqrtf/reciprocal-multiply here.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#define RT_DEV __device__ __forceinline__

struct V3 {
    float x, y, z;
};
RT_DEV V3 mk3(float x, float y, float z)
{
    V3 r;
    r.x = x; r.y = y; r.z = z;
    return r;
}
RT_DEV V3 mk3(const float4& v) { return mk3(v.x, v.y, v.z); }
RT_DEV V3 operator+(const V3& a, const V3& b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
RT_DEV V3 operator-(const V3& a, const V3& b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
RT_DEV V3 operator*(const V3& a, const V3& b) { return mk3(a.x * b.x, a.y * b.y, a.z * b.z); }
RT_DEV V3 operator*(const V3& a, float s) { return mk3(a.x * s, a.y * s, a.z * s); }
RT_DEV V3 operator*(float s, const V3& a) { return mk3(s * a.x, s * a.y, s * a.z); }
RT_DEV V3 operator-(const V3& a) { return mk3(-a.x, -a.y, -a.z); }
// glm: dot = (x*x' + y*y') + z*z' ; cross ; length = sqrt(dot) ; normalize = v * (1/sqrt(dot)) ; reflect = I - (N*dot(N,I))*2
RT_DEV float dot3(const V3& a, const V3& b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
RT_DEV V3 cross3(const V3& x, const V3& y)
{
    return mk3(x.y * y.z - y.y * x.z, x.z * y.x - y.z * x.x, x.x * y.y - y.x * x.y);
}
RT_DEV float length3(const V3& v) { return sqrtf(dot3(v, v)); }
RT_DEV V3 normalize3(const V3& v) { return v * (1.0f / sqrtf(dot3(v, v))); }
RT_DEV V3 reflect3(const V3& I, const V3& N) { return I - (N * dot3(N, I)) * 2.0f; }

// ---- intersectRayWithShape(const AxisAlignedBox&, Ray&)  src/ray_tracing.cpp:162-200 ------------------------------------
// Returns true and writes the entry distance into tHit iff the reference would return true for a ray whose current
// ray.t is rayT. Ternaries are kept literally: with NaN operands the SECOND alternative is chosen, as in the reference.
RT_DEV bool slabTest(const V3& lo, const V3& hi, const V3& o, const V3& d, float rayT, float& tHit)
{
    const float tMinX = (lo.x - o.x) / d.x, tMinY = (lo.y - o.y) / d.y, tMinZ = (lo.z - o.z) / d.z;
    const float tMaxX = (hi.x - o.x) / d.x, tMaxY = (hi.y - o.y) / d.y, tMaxZ = (hi.z - o.z) / d.z;
    const float tInX = tMinX < tMaxX ? tMinX : tMaxX;
    const float tOutX = tMinX > tMaxX ? tMinX : tMaxX;
    const float tInY = tMinY < tMaxY ? tMinY : tMaxY;
    const float tOutY = tMinY > tMaxY ? tMinY : tMaxY;
    const float tInZ = tMinZ < tMaxZ ? tMinZ : tMaxZ;
    const float tOutZ = tMinZ > tMaxZ ? tMinZ : tMaxZ;
    const float tIn = tInX > tInY ? (tInX > tInZ ? tInX : tInZ) : (tInY > tInZ ? tInY : tInZ);
    const float tOut = tOutX < tOutY ? (tOutX < tOutZ ? tOutX : tOutZ) : (tOutY < tOutZ ? tOutY : tOutZ);
    float currentT;
    if (tIn > tOut || tOut < 0) return false;
    else if (tIn < 0) currentT = tOut;
    else currentT = tIn;
    if (currentT >= rayT) return false;
    tHit = currentT;
    return true;
}

// startsInBox  src/bounding_volume_hierarchy.cpp:647-661 (strict inequalities: on-face origins are outside)
RT_DEV bool startsInBox(const V3& o, const V3& lo, const V3& hi)
{
    const bool inX = lo.x < o.x && o.x < hi.x;
    const bool inY = lo.y < o.y && o.y < hi.y;
    const bool inZ = lo.z < o.z && o.z < hi.z;
    return inX && inY && inZ;
}

// ---- trianglePlane  src/ray_tracing.cpp:74-82 ---------------------------------------------------------------------------
RT_DEV float4 trianglePlaneDev(const V3& v0, const V3& v1, const V3& v2)
{
    const V3 u = v1 - v0;
    const V3 v = v2 - v0;
    const V3 n = normalize3(cross3(u, v));
    return make_float4(n.x, n.y, n.z, dot3(v0, n));
}

// ---- intersectRayWithPlane  src/ray_tracing.cpp:40-72 : candidate distance or reject ------------------------------------
// Returns true with tt = the value the reference would store in ray.t.
RT_DEV bool planeTest(const V3& n, float D, const V3& o, const V3& d, float rayT, float& tt)
{
    const float on = dot3(o, n);
    if (on == D) { // origin lies in the plane: t = 0 even when ray.t is already 0 (quirk, SURVEY Appendix B.8)
        tt = 0.0f;
        return true;
    }
    const float denominator = dot3(d, n);
    if (denominator == 0) return false;
    const float numerator = D - on;
    const float t = numerator / denominator;
    if (t < 0) return false;
    if (t >= rayT) return false;
    tt = t;
    return true;
}

// ---- pointInTriangle  src/ray_tracing.cpp:23-38 (edges inclusive) --------------------------------------------------------
RT_DEV bool pointInTriangleDev(const V3& v0, const V3& v1, const V3& v2, const V3& n, const V3& p)
{
    const V3 v0v1 = v1 - v0;
    const V3 v1v2 = v2 - v1;
    const V3 v2v0 = v0 - v2;
    const V3 v0p = p - v0;
    const V3 v1p = p - v1;
    const V3 v2p = p - v2;
    return dot3(n, cross3(v0v1, v0p)) >= 0 && dot3(n, cross3(v1v2, v1p)) >= 0 && dot3(n, cross3(v2v0, v2p)) >= 0;
}

// ---- magnitude / area  src/ray_tracing.cpp:13-21 : pow(float,int) promotes to double, sqrt in double, narrowed ----------
RT_DEV float areaDev(const V3& a, const V3& b, const V3& c)
{
    const V3 k = cross3(b - a, c - a);
    const double s = ((double)k.x * (double)k.x + (double)k.y * (double)k.y) + (double)k.z * (double)k.z;
    const float m = (float)sqrt(s);
    return m / 2.0f;
}

// ---- accepted-hit epilogue of intersectRayWithTriangle  src/ray_tracing.cpp:92-107 ---------------------------------------
// The reference evaluates this for every accepted candidate; only the last accepted one survives, so the wavefront
// evaluates it once for the final hit (same inputs -> same bits).
RT_DEV void hitEpilogue(const V3& v0, const V3& v1, const V3& v2, const V3& n0, const V3& n1, const V3& n2,
                     const V3& planeN, const V3& o, const V3& d, float t, float& alpha, float& beta, float& gamma,
                     V3& normal)
{
    const V3 p = o + d * t;
    const float whole = areaDev(v0, v1, v2);
    alpha = areaDev(p, v1, v2) / whole;
    beta = areaDev(p, v0, v2) / whole;
    gamma = areaDev(p, v0, v1) / whole;
    const V3 ni = normalize3((alpha * n0 + beta * n1) + gamma * n2);
    normal = dot3(planeN, -d) > 0 ? ni : -ni;
}

// ---- intersectRayWithShape(const Sphere&, Ray&, HitInfo&)  src/ray_tracing.cpp:118-158 -----------------------------------
// Unqualified sqrt(float) resolves to ::sqrt(double) under g++/glibc (the oracle's compiler), so the two roots are
// evaluated in double and narrowed on assignment; reproduced literally.
RT_DEV bool sphereTest(const V3& center, float radius, const V3& o, const V3& d, float rayT, float& tHit, V3& normal)
{
    const V3 oc = o - center;
    const float a = dot3(d, d);
    const float b = 2 * dot3(d, oc);
    const float c = dot3(oc, oc) - radius * radius;
    const float D = b * b - 4 * a * c;
    if (D < 0) return false;
    const float smallerT = (float)(((double)(-b) - sqrt((double)D)) / (double)(2 * a));
    const float biggerT = (float)(((double)(-b) + sqrt((double)D)) / (double)(2 * a));
    float currentT;
    if (smallerT >= 0) currentT = smallerT;
    else if (biggerT >= 0) currentT = biggerT;
    else return false;
    if (currentT >= rayT) return false;
    tHit = currentT;
    normal = normalize3((o + d * currentT) - center);
    return true;
}
