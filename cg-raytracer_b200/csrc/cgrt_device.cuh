// Device-side BVH traversal shared by every kernel: the reference's exact visiting order over the reference tree, with the
// (large) reference leaves refined by conservative culling sub-trees. Results are identical to the reference's sequential
// leaf scan by construction; see the comments on leaf evaluation below.
#pragma once
#include "rt_math.cuh"
#include "cgrt_kernels.h"

RT_DEV int f2i(float f) { return __float_as_int(f); }
RT_DEV float i2f(int i) { return __int_as_float(i); }

struct TraceResult {
    float t;      // ray.t after the query
    int tri;      // position (leaf-ordered arrays) of the last accepted triangle, -1 none
    int sphere;   // index of the last accepted sphere (closer than every triangle), -1 none
    V3 sphereN;   // its normal
};

// ---- leaf evaluation ----------------------------------------------------------------------------------------------------------
// intersectLeaf (src/bounding_volume_hierarchy.cpp:535-553) scans the leaf's triangles in order and accepts a triangle iff
// its plane distance tt is >= 0 and < the CURRENT ray.t and the hit point is inside (src/ray_tracing.cpp:40-114). The state
// after the scan is therefore: among the triangles that are acceptable against the ray.t at leaf ENTRY, the one with the
// smallest tt, ties broken by the earliest position in the leaf ("rank"). That characterisation does not depend on the order
// in which the triangles are examined, which is what lets the sub-tree skip triangles that cannot be accepted.
// One quirk: when the origin lies exactly in the triangle's plane (dot(o,n) == D) the reference takes t = 0 WITHOUT comparing
// against ray.t (:43-47), so among such "shortcut" candidates the LAST one in leaf order wins, and it beats every other.
struct LeafBest {
    float t;      // best distance so far (initially ray.t at leaf entry)
    int pos;      // position of the best triangle, -1 = none accepted in this leaf yet
    int rank;     // its rank in the reference's leaf order
    bool shortcut;
};

// Exact accept arithmetic for one triangle (same expression trees as planeTest + pointInTriangleDev), folded into `best`.
// Returns true iff the triangle became the new best.
RT_DEV bool leafCandidate(const DevScene& S, int i, const V3& o, const V3& d, LeafBest& best)
{
    const float4* tr = S.tri4 + 4 * (size_t)i;
    const float4 pl = __ldg(tr);
    const V3 n = mk3(pl);
    const float on = dot3(o, n);
    float tt;
    bool shortcut = false;
    if (on == pl.w) {
        tt = 0.0f;
        shortcut = true;
    } else {
        const float denominator = dot3(d, n);
        if (denominator == 0) return false;
        tt = (pl.w - on) / denominator;
        if (tt < 0) return false;
        // cannot win: farther than the best, or a shortcut candidate already holds the leaf, or equal to ray.t at leaf
        // entry (rejected by the reference's `t >= ray.t`)
        if (!(tt <= best.t)) return false;
        if (best.shortcut) return false;
        if (tt == best.t && best.pos < 0) return false;
    }
    const float4 v0 = __ldg(tr + 1), v1 = __ldg(tr + 2), v2 = __ldg(tr + 3);
    const int rank = f2i(v2.w);
    if (shortcut) {
        if (best.shortcut && rank < best.rank) return false; // the last shortcut candidate in leaf order wins
    } else if (tt == best.t && rank > best.rank) {
        return false; // equally close: the reference keeps the one it reached first
    }
    const V3 p = o + d * tt;
    if (!pointInTriangleDev(mk3(v0), mk3(v1), mk3(v2), n, p)) return false;
    best.t = tt;
    best.pos = i;
    best.rank = rank;
    best.shortcut = shortcut;
    return true;
}

#define CGRT_SUBSTACK 40

// ---- the production traversal ---------------------------------------------------------------------------------------------
// Same visiting order, pruning and accept arithmetic as traverseStrict below (which documents the mapping to the reference's
// functions); the difference is structural:
//  * One node per step, resumable (persistent warps hand a finished lane a new ray between steps, cgrt_kernels.cu).
//  * Reference nodes and the nodes of the culling sub-trees live in ONE array of child pairs (DevScene::pairs, 4 x float4:
//    both children's boxes, each with a 2-word descriptor), so a step is one 64-byte fetch, and the inner-node step is the
//    same instruction stream for both kinds: slab distances as (box - o) * fl(1/d), then a short kind-specific decision.
//      - sub-tree pair: tolerant test against pre-expanded boxes, nearer child first, pruned against the leaf's best distance;
//      - reference pair: the reference's exact decisions (intersectNonLeaf / intersectDeeper, bvh.cpp:679-736). The slab
//        distances computed this way differ from the reference's correctly rounded quotients by at most 3 ulp, so with
//        rho = 1e-6 relative (+ tau absolute) slack every comparison of slabTest (ray_tracing.cpp:162-200) is either decided
//        with certainty or declared ambiguous; ambiguous cases (and rays with extreme direction components) evaluate
//        slabTest itself. Its numeric result matters only for ordering two hit children and for pruning a pending sibling;
//        there too the approximate value is used when it is decisive and the exact one is computed otherwise.
//    Outcomes are therefore exactly the reference's; divisions are only executed when they can matter.
//  * Stack entries carry a key: for a reference sibling the entry distance tSecond (skipped iff ray.t < tSecond,
//    intersectChildrenHierarchically), for a sub-tree node its tolerant entry distance (skipped iff beyond the leaf's best).
//    A reference leaf's result is committed when its sub-tree entries are gone.
//
// Node ids (child descriptors w0, stack entries, Trav::node):
//   bits 0..25 index: pair index (inner nodes) | first triangle position (CGRT_TRI) | reference node index (CGRT_REFSCAN)
//   bits 26..28 count-1 of a CGRT_TRI leaf (ids with CGRT_TRI only)
//   bit 27  CGRT_KEYAPPROX (reference stack entries only: the key is an approximate distance)
//   bit 28  CGRT_REFLEAF: a reference leaf entered through its sub-tree (index = wide node of the sub-tree root)
//   bit 29  CGRT_TRI: sub-tree leaf           bit 30  CGRT_SUB: sub-tree node (index = wide node unless CGRT_TRI)
//   bit 31  CGRT_REFSCAN: reference leaf scanned triangle by triangle (leaves too small for a sub-tree, or rays excluded
//   from the tolerant tests)
#define CGRT_IDX_MASK 0x03ffffffu
#define CGRT_TRICNT_SHIFT 26
#define CGRT_KEYAPPROX 0x08000000u
#define CGRT_REFLEAF 0x10000000u
#define CGRT_TRI 0x20000000u
#define CGRT_SUB 0x40000000u
#define CGRT_REFSCAN 0x80000000u

#define CGRT_WIDE_STRIDE 16 // float4 per 8-wide node: 14 used, padded to 256 B = exactly two 128-byte lines

#define CGRT_RHO 1e-6f
#define CGRT_TAU 1e-30f
RT_DEV float errBound(float x) { return fabsf(x) * CGRT_RHO + CGRT_TAU; }

struct Trav {
    V3 o, d, inv;
    float t;
    int hitTri;
    int sp, subBase;
    uint32_t node;
    bool useSub;  // the ray may use the culling sub-trees (tolerant tests are safe for it)
    bool fastRef; // reference box tests may be decided from (box - o) * inv for this ray
    bool inLeaf;
    LeafBest best;
};
// the traversal stack lives outside the struct so that the scalars above stay in registers
struct TravStack {
    uint32_t n[CGRT_STACK + CGRT_SUBSTACK];
    float t[CGRT_STACK + CGRT_SUBSTACK];
    int r[CGRT_STACK + CGRT_SUBSTACK]; // reference node index of a reference entry (exact re-evaluation of its key)
};

enum { TRAV_CONTINUE = 0, TRAV_DONE = 1, TRAV_FIRED = 2, TRAV_DEFER = 3 };
enum { CLS_REF = 0, CLS_WIDE = 1, CLS_LEAF = 2, CLS_NONE = 3 };
RT_DEV int travClass(uint32_t node)
{
    if (node & (CGRT_TRI | CGRT_REFSCAN)) return CLS_LEAF;
    return (node & (CGRT_SUB | CGRT_REFLEAF)) ? CLS_WIDE : CLS_REF;
}

// intersectDataStructure (bvh.cpp:831-844): returns true iff the tree has to be traversed for this ray.
RT_DEV bool travBegin(const DevScene& S, Trav& T, const V3& o, const V3& d, float tIn)
{
    T.o = o;
    T.d = d;
    T.t = tIn;
    T.hitTri = -1;
    T.sp = 0;
    T.subBase = 0;
    T.inLeaf = false;
    T.best.t = tIn; T.best.pos = -1; T.best.rank = -1; T.best.shortcut = false;
    if (S.nNodes <= 0) return false;
    const float4 rq0 = __ldg(S.nodes + 0), rq1 = __ldg(S.nodes + 1);
    bool enter = startsInBox(o, mk3(rq0), mk3(rq1));
    if (!enter) {
        float tmp;
        enter = slabTest(mk3(rq0), mk3(rq1), o, d, tIn, tmp);
    }
    if (!enter) return false;
    const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    // tolerant sub-tree tests: zero components are fine (huge finite reciprocal), extreme magnitudes are not
    const bool okx = (ax == 0.0f) || (ax >= 1e-20f && ax <= 1e20f);
    const bool oky = (ay == 0.0f) || (ay >= 1e-20f && ay <= 1e20f);
    const bool okz = (az == 0.0f) || (az >= 1e-20f && az <= 1e20f);
    const bool fin = fabsf(o.x) <= 1e30f && fabsf(o.y) <= 1e30f && fabsf(o.z) <= 1e30f; // false for NaN
    T.useSub = okx && oky && okz && fin;
    T.inv.x = ax == 0.0f ? 1e30f : 1.0f / d.x;
    T.inv.y = ay == 0.0f ? 1e30f : 1.0f / d.y;
    T.inv.z = az == 0.0f ? 1e30f : 1.0f / d.z;
    // filtered reference box tests need finite non-zero reciprocals and no overflow in (box - o) * inv
    T.fastRef = ax >= 1e-15f && ax <= 1e15f && ay >= 1e-15f && ay <= 1e15f && az >= 1e-15f && az <= 1e15f &&
                fabsf(o.x) <= 1e15f && fabsf(o.y) <= 1e15f && fabsf(o.z) <= 1e15f;
    const uint32_t root = (uint32_t)S.rootId;
    T.node = ((root & CGRT_REFLEAF) && !T.useSub) ? (CGRT_REFSCAN | 0u) : root;
    return true;
}

// the reference's distance of a box that is known to be hit (used when an approximate distance is not decisive)
RT_DEV float boxExactT(const float4& lo, const float4& hi, const V3& o, const V3& d)
{
    float te = 0.0f;
    slabTest(mk3(lo), mk3(hi), o, d, __int_as_float(0x7f800000), te);
    return te;
}

// pop: next pending node that is not pruned, committing the reference leaf when its sub-tree entries are gone
RT_DEV int travPop(const DevScene& S, Trav& T, TravStack& K)
{
    const float slack = 1.000001f;
    while (true) {
        if (T.inLeaf && T.sp == T.subBase) {
            if (T.best.pos >= 0) { T.t = T.best.t; T.hitTri = T.best.pos; }
            T.inLeaf = false;
        }
        if (T.sp == 0) return TRAV_DONE;
        T.sp--;
        const uint32_t n = K.n[T.sp];
        const float key = K.t[T.sp];
        if (n & CGRT_SUB) {
            if (key > T.best.t * slack) continue;
            T.node = n;
            return TRAV_CONTINUE;
        }
        // reference sibling: skipped iff ray.t < tSecond (intersectChildrenHierarchically, bvh.cpp:572-595)
        if (n & CGRT_KEYAPPROX) {
            const float e = errBound(key);
            if (T.t < key - e) continue;
            if (!(T.t >= key + e)) { // not decisive: compare with the reference's exact distance of that box
                const int ri = K.r[T.sp];
                const float tS = boxExactT(__ldg(S.nodes + 2 * ri), __ldg(S.nodes + 2 * ri + 1), T.o, T.d);
                if (T.t < tS) continue;
            }
        } else {
            if (T.t < key) continue;
        }
        T.node = n & ~CGRT_KEYAPPROX;
        return TRAV_CONTINUE;
    }
}

// slab distances of one child box from the per-ray reciprocals
RT_DEV void slabApprox(const float4& lo, const float4& hi, const V3& o, const V3& inv, float& tin, float& tout)
{
    const float q0x = (lo.x - o.x) * inv.x, q1x = (hi.x - o.x) * inv.x;
    const float q0y = (lo.y - o.y) * inv.y, q1y = (hi.y - o.y) * inv.y;
    const float q0z = (lo.z - o.z) * inv.z, q1z = (hi.z - o.z) * inv.z;
    tin = fmaxf(fmaxf(fminf(q0x, q1x), fminf(q0y, q1y)), fminf(q0z, q1z));
    tout = fminf(fminf(fmaxf(q0x, q1x), fmaxf(q0y, q1y)), fmaxf(q0z, q1z));
}

// the reference's box test decided from approximate slab distances when that is certain, else by slabTest itself.
// hit: the reference's boolean; t: its distance (exact when `exact`, otherwise within errBound(t) of it)
RT_DEV void refBoxDecide(const float4& lo, const float4& hi, const V3& o, const V3& d, bool fast, float tin, float tout,
                         float rayT, bool& hit, float& t, bool& exact)
{
    if (fast) {
        const float ein = errBound(tin), eout = errBound(tout);
        if (tout + eout < 0.0f || tin - ein > tout + eout) { // certainly `tOut < 0` or `tIn > tOut`
            hit = false;
            return;
        }
        float cur = 0.0f, ecur = 0.0f;
        bool branch = false;
        if (tin + ein < 0.0f) { cur = tout; ecur = eout; branch = true; }        // certainly tIn < 0
        else if (tin - ein >= 0.0f) { cur = tin; ecur = ein; branch = true; }   // certainly tIn >= 0
        if (branch) {
            if (cur - ecur >= rayT) { // certainly `currentT >= ray.t`
                hit = false;
                return;
            }
            if (tin + ein <= tout - eout && tout - eout >= 0.0f && cur + ecur < rayT) { // certainly a hit
                hit = true;
                t = cur;
                exact = false;
                return;
            }
        }
    }
    float te = 0.0f;
    hit = slabTest(mk3(lo), mk3(hi), o, d, rayT, te);
    t = te;
    exact = true;
}

// one step on a reference inner node: intersectNonLeaf + intersectDeeper with the reference's exact outcomes
RT_DEV int travStepRef(const DevScene& S, Trav& T, TravStack& K)
{
    const float4* pr = S.pairs + 4 * (size_t)(T.node & CGRT_IDX_MASK);
    const float4 l0 = __ldg(pr), l1 = __ldg(pr + 1), r0 = __ldg(pr + 2), r1 = __ldg(pr + 3);
    const V3 o = T.o, d = T.d;
    float tinL, toutL, tinR, toutR;
    slabApprox(l0, l1, o, T.inv, tinL, toutL);
    slabApprox(r0, r1, o, T.inv, tinR, toutR);
    uint32_t idL = (uint32_t)f2i(l0.w), idR = (uint32_t)f2i(r0.w);
    if (!T.useSub) { // this ray scans reference leaves instead of using their sub-trees
        if (idL & CGRT_REFLEAF) idL = CGRT_REFSCAN | (uint32_t)f2i(l1.w);
        if (idR & CGRT_REFLEAF) idR = CGRT_REFSCAN | (uint32_t)f2i(r1.w);
    }
    bool hL, hR, exL = true, exR = true;
    float tL = -1.0f, tR = -1.0f;
    refBoxDecide(l0, l1, o, d, T.fastRef, tinL, toutL, T.t, hL, tL, exL);
    refBoxDecide(r0, r1, o, d, T.fastRef, tinR, toutR, T.t, hR, tR, exR);
    const bool inL = startsInBox(o, mk3(l0), mk3(l1));
    const bool inR = startsInBox(o, mk3(r0), mk3(r1));
    uint32_t first = 0u, second = 0u;
    bool haveFirst = false, haveSecond = false, keyApprox = false, secondIsRight = false;
    float key = -1.0f;
    if (inL && inR) { // both visited unconditionally, left operand of `|` first (g++ order)
        first = idL; second = idR; haveFirst = haveSecond = true; secondIsRight = true; key = -1.0f;
    } else if (inL) {
        first = idL; haveFirst = true;
        if (hR) { second = idR; haveSecond = true; secondIsRight = true; key = tR; keyApprox = !exR; }
    } else if (inR) {
        first = idR; haveFirst = true;
        if (hL) { second = idL; haveSecond = true; key = tL; keyApprox = !exL; }
    } else if (hL && hR) {
        // nearer child first: `tLeft < tRight` (bvh.cpp:626), from the approximate distances when they are separated
        // by more than their error bounds, otherwise from the exact ones
        bool leftFirst;
        if (!(exL && exR) && tL + errBound(tL) < tR - errBound(tR)) leftFirst = true;
        else if (!(exL && exR) && tL - errBound(tL) >= tR + errBound(tR)) leftFirst = false;
        else {
            if (!exL) { tL = boxExactT(l0, l1, o, d); exL = true; }
            if (!exR) { tR = boxExactT(r0, r1, o, d); exR = true; }
            leftFirst = tL < tR;
        }
        haveFirst = haveSecond = true;
        if (leftFirst) { first = idL; second = idR; secondIsRight = true; key = tR; keyApprox = !exR; }
        else { first = idR; second = idL; key = tL; keyApprox = !exL; }
    } else if (hL) {
        first = idL; haveFirst = true;
    } else if (hR) {
        first = idR; haveFirst = true;
    }
    if (haveSecond) {
        K.n[T.sp] = keyApprox ? (second | CGRT_KEYAPPROX) : second;
        K.t[T.sp] = key;
        K.r[T.sp] = f2i(secondIsRight ? r1.w : l1.w);
        T.sp++;
    }
    if (haveFirst) {
        T.node = first;
        return TRAV_CONTINUE;
    }
    return travPop(S, T, K);
}

// one step on an 8-wide sub-tree node: tolerant tests of all children against their pre-expanded boxes (never a miss for a
// box that holds a point the reference could accept); the nearest hit child is visited next, the others are stacked with
// their entry distance and pruned against the leaf's best distance when popped
RT_DEV int travStepWide(const DevScene& S, Trav& T, TravStack& K)
{
    uint32_t id = T.node;
    if (id & CGRT_REFLEAF) { // entering a reference leaf through its sub-tree (intersectLeaf, evaluated order-independently)
        T.best.t = T.t; T.best.pos = -1; T.best.rank = -1; T.best.shortcut = false;
        T.inLeaf = true;
        T.subBase = T.sp;
    }
    const float4* w = S.wide + CGRT_WIDE_STRIDE * (size_t)(id & CGRT_IDX_MASK);
    const float slack = 1.000001f;
    const float bt = T.best.t * slack;
    const V3 o = T.o, inv = T.inv;
    float tin[8];
    uint32_t cid[8];
    unsigned hitMask = 0u;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const float4 lx = __ldg(w + 0 + h), ly = __ldg(w + 2 + h), lz = __ldg(w + 4 + h);
        const float4 hx = __ldg(w + 6 + h), hy = __ldg(w + 8 + h), hz = __ldg(w + 10 + h);
        const float4 ci = __ldg(w + 12 + h);
        const float lox[4] = {lx.x, lx.y, lx.z, lx.w}, loy[4] = {ly.x, ly.y, ly.z, ly.w}, loz[4] = {lz.x, lz.y, lz.z, lz.w};
        const float hix[4] = {hx.x, hx.y, hx.z, hx.w}, hiy[4] = {hy.x, hy.y, hy.z, hy.w}, hiz[4] = {hz.x, hz.y, hz.z, hz.w};
        const float cw[4] = {ci.x, ci.y, ci.z, ci.w};
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const float q0x = (lox[c] - o.x) * inv.x, q1x = (hix[c] - o.x) * inv.x;
            const float q0y = (loy[c] - o.y) * inv.y, q1y = (hiy[c] - o.y) * inv.y;
            const float q0z = (loz[c] - o.z) * inv.z, q1z = (hiz[c] - o.z) * inv.z;
            const float ti = fmaxf(fmaxf(fminf(q0x, q1x), fminf(q0y, q1y)), fminf(q0z, q1z));
            const float to = fminf(fminf(fmaxf(q0x, q1x), fmaxf(q0y, q1y)), fmaxf(q0z, q1z));
            const uint32_t ii = (uint32_t)f2i(cw[c]);
            const bool hit = ii != 0u && !(to < 0.0f || ti > to * slack || ti > bt);
            tin[4 * h + c] = ti;
            cid[4 * h + c] = ii;
            if (hit) hitMask |= 1u << (4 * h + c);
        }
    }
    if (hitMask == 0u) return travPop(S, T, K);
    // nearest hit child first
    int best = -1;
    float bestT = 0.0f;
#pragma unroll
    for (int c = 0; c < 8; c++) {
        if ((hitMask >> c & 1u) && (best < 0 || tin[c] < bestT)) { best = c; bestT = tin[c]; }
    }
#pragma unroll
    for (int c = 0; c < 8; c++) {
        if ((hitMask >> c & 1u) && c != best) {
            K.n[T.sp] = cid[c];
            K.t[T.sp] = tin[c];
            T.sp++;
        }
    }
    T.node = cid[best];
    return TRAV_CONTINUE;
}

// one step on a leaf: the triangles of a sub-tree leaf (folded into the reference leaf's running best), or a whole
// reference leaf scanned in order
template <bool ANY>
RT_DEV int travStepLeaf(const DevScene& S, Trav& T, TravStack& K, float eps, float maxDist)
{
    const uint32_t id = T.node;
    int first, count;
    const bool scan = (id & CGRT_REFSCAN) != 0u;
    if (scan) {
        const int ri = (int)(id & CGRT_IDX_MASK);
        first = f2i(__ldg(S.nodes + 2 * ri).w);
        count = f2i(__ldg(S.nodes + 2 * ri + 1).w);
        T.best.t = T.t; T.best.pos = -1; T.best.rank = -1; T.best.shortcut = false;
    } else {
        first = (int)(id & CGRT_IDX_MASK);
        count = (int)((id >> CGRT_TRICNT_SHIFT) & 7u) + 1;
    }
#pragma unroll 1
    for (int i = first; i < first + count; i++) {
        if (leafCandidate(S, i, T.o, T.d, T.best)) {
            if (ANY && !(T.best.t + eps >= maxDist)) return TRAV_FIRED;
        }
    }
    if (scan && T.best.pos >= 0) { T.t = T.best.t; T.hitTri = T.best.pos; }
    return travPop(S, T, K);
}

template <bool ANY>
RT_DEV int travStep(const DevScene& S, Trav& T, TravStack& K, float eps, float maxDist)
{
    const int cls = travClass(T.node);
    if (cls == CLS_REF) return travStepRef(S, T, K);
    if (cls == CLS_WIDE) return travStepWide(S, T, K);
    return travStepLeaf<ANY>(S, T, K, eps, maxDist);
}

// After the tree: the sphere loop of BoundingVolumeHierarchy::intersect (bvh.cpp:878-879) and the result record.
// `state` is TRAV_FIRED when the any-hit predicate already fired inside the tree. Returns hit (closest) / shadowed (ANY).
template <bool ANY>
RT_DEV bool travFinish(const DevScene& S, Trav& T, int state, float eps, float maxDist, TraceResult& R)
{
    R.sphere = -1;
    if (ANY && state == TRAV_FIRED) {
        R.t = T.best.t;
        R.tri = T.best.pos;
        return true;
    }
    float t = T.t;
    for (int s = 0; s < S.nSpheres; s++) {
        const float4 c = __ldg(S.spheres + 3 * s);
        float ts;
        V3 nn;
        if (sphereTest(mk3(c), c.w, T.o, T.d, t, ts, nn)) {
            t = ts;
            R.sphere = s;
            R.sphereN = nn;
            if (ANY && !(ts + eps >= maxDist)) {
                R.t = t;
                R.tri = T.hitTri;
                return true;
            }
        }
    }
    R.t = t;
    R.tri = T.hitTri;
    if (ANY) return false;
    return T.hitTri >= 0 || R.sphere >= 0;
}

// one ray, start to finish (batch entry points that do not use persistent warps)
template <bool ANY>
RT_DEV bool traverseFast(const DevScene& S, const V3& o, const V3& d, float tIn, float eps, float maxDist, TraceResult& R)
{
    Trav T;
    TravStack K;
    int state = TRAV_DONE;
    if (travBegin(S, T, o, d, tIn)) {
        do {
            state = travStep<ANY>(S, T, K, eps, maxDist);
        } while (state == TRAV_CONTINUE);
    }
    return travFinish<ANY>(S, T, state, eps, maxDist, R);
}

// ---- the speculative traversal ------------------------------------------------------------------------------------------------
// The exact traversal above pays for reproducing the reference's visiting ORDER (two exact box decisions per reference node,
// three node classes). For almost every ray the order is irrelevant: the reference's result is simply the acceptable
// triangle with the smallest distance, where "acceptable" means that the reference's own arithmetic (leafCandidate: plane
// distance in [0, ray.t at entry), point inside) accepts it. The speculative traversal therefore
//   1. searches ONE conservative 8-wide tree over all triangles (DevScene::fastRoot, bvh_build.cpp buildFastTree) for the
//      acceptable triangle of smallest distance t* - tolerant box tests that can never cull an acceptable triangle, the
//      reference's exact triangle arithmetic, plain nearest-first order with pruning against t*;
//   2. CERTIFIES that the reference finds the same triangle (certifyChain): the reference reaches a leaf unless one of the
//      boxes on the way from the root is rejected (`currentT >= ray.t`, or a miss) or pruned as a pending sibling
//      (`ray.t < tSecond`). Before tri* is accepted ray.t is the distance of some other acceptable triangle or the initial
//      bound, i.e. > t*. So if for every node on the path root -> leaf(tri*) the origin is strictly inside the box
//      (startsInBox: visited unconditionally, bvh.cpp:685-696) or the reference's own slabTest with ray.t := t* reports a hit
//      with distance < t*, every one of those decisions comes out "descend" whatever the order of the visits, the leaf scan
//      accepts tri* (its distance is below the current ray.t) and nothing accepted later can replace it (nothing acceptable is
//      closer). A miss needs no certificate: the reference only ever accepts acceptable triangles.
//   3. DEFERS the ray to the exact traversal whenever the outcome could depend on the visiting order: two acceptable triangles
//      at exactly the same distance, a candidate through the in-plane shortcut (ray_tracing.cpp:43-47, accepted regardless of
//      ray.t), a box on the chain that is entered exactly at t* (axis-aligned geometry lying in a box face), or a ray the
//      tolerant tests are not safe for (useSub). Deferred rays are replayed by the exact kernels; results are identical to
//      the reference's in every case, only the cost differs.
// Any-hit (pointInShadow): an acceptable triangle X with !(t_X + eps >= maxDist) whose chain certifies with t* := t_X proves
// "shadowed" - the reference either visits leaf(X) with ray.t > t_X and accepts X, or its ray.t is already below t_X; its
// final distance is <= t_X either way and the predicate is monotone. No such X among ALL acceptable triangles proves that
// the tree does not shadow; the search may prune with min(t*, maxDist) because eps > 0.
struct FastTrav {
    V3 o, d, inv;
    float t;     // distance of the best acceptable triangle so far (initially the ray's bound)
    int hitTri;  // position of the best triangle, -1 none
    int sp;
    uint32_t node;
};
// acceptable triangles up to this factor beyond the best are still examined, so that the certificate knows every acceptable
// triangle closer than t* (1 + 1e-6) (the pruning of the search uses the same factor)
#define CGRT_NEAR 1.000001f
#define CGRT_FASTSTACK 64
struct FastStack {
    uint2 e[CGRT_FASTSTACK]; // (node id, entry distance): one 8-byte local-memory access per push / pop
    float t2; // smallest distance of any OTHER acceptable triangle met so far (runner-up), +inf none: see certifyClosest. Lives
              // here (local memory) because it is touched only when a candidate is accepted; a register in the hot loop is not
};

// intersectDataStructure (bvh.cpp:831-844) evaluated exactly, then the fast tree's root.
// TRAV_DONE: the reference does not enter the tree (certain miss); TRAV_DEFER: this ray must take the exact traversal.
RT_DEV int fastBegin(const DevScene& S, FastTrav& T, const V3& o, const V3& d, float tIn)
{
    T.o = o;
    T.d = d;
    T.t = tIn;
    T.hitTri = -1;
    T.sp = 0;
    T.node = 0u;
    if (S.nNodes <= 0) return TRAV_DONE;
    const float4 rq0 = __ldg(S.nodes + 0), rq1 = __ldg(S.nodes + 1);
    bool enter = startsInBox(o, mk3(rq0), mk3(rq1));
    if (!enter) {
        float tmp;
        enter = slabTest(mk3(rq0), mk3(rq1), o, d, tIn, tmp);
    }
    if (!enter) return TRAV_DONE;
    const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    const bool okx = (ax == 0.0f) || (ax >= 1e-20f && ax <= 1e20f);
    const bool oky = (ay == 0.0f) || (ay >= 1e-20f && ay <= 1e20f);
    const bool okz = (az == 0.0f) || (az >= 1e-20f && az <= 1e20f);
    const bool fin = fabsf(o.x) <= 1e30f && fabsf(o.y) <= 1e30f && fabsf(o.z) <= 1e30f; // false for NaN
    // a negative or NaN ray bound is garbage the reference still has defined behaviour for (its in-plane shortcut accepts t = 0
    // whatever ray.t is, and `t >= NaN` never rejects); the search prunes with the bound, so such rays take the exact traversal
    if (!(okx && oky && okz && fin) || !(tIn >= 0.0f) || S.fastRoot == 0u) return TRAV_DEFER;
    T.inv.x = ax == 0.0f ? 1e30f : 1.0f / d.x;
    T.inv.y = ay == 0.0f ? 1e30f : 1.0f / d.y;
    T.inv.z = az == 0.0f ? 1e30f : 1.0f / d.z;
    T.node = S.fastRoot;
    return TRAV_CONTINUE;
}

RT_DEV int fastPop(FastTrav& T, FastStack& K, float bound)
{
    while (T.sp > 0) {
        T.sp--;
        const uint2 e = K.e[T.sp];
        if (__uint_as_float(e.y) > bound) continue;
        T.node = e.x;
        return TRAV_CONTINUE;
    }
    return TRAV_DONE;
}

// search bound: boxes entered beyond it cannot hold a closer acceptable triangle (ANY: nor one within maxDist)
template <bool ANY>
RT_DEV float fastBound(const FastTrav& T, float maxDist)
{
    const float slack = 1.000001f;
    return (ANY ? fminf(T.t, maxDist) : T.t) * slack;
}

RT_DEV int fastStepWideDyn(const DevScene& S, FastTrav& T, FastStack& K, bool any, float maxDist)
{
    const float4* w = S.wide + CGRT_WIDE_STRIDE * (size_t)(T.node & CGRT_IDX_MASK);
    const float slack = 1.000001f;
    const float bt = (any ? fminf(T.t, maxDist) : T.t) * slack; // = fastBound<ANY>
    const V3 o = T.o, inv = T.inv;
    float tin[8];
    uint32_t cid[8];
    unsigned hitMask = 0u;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const float4 lx = __ldg(w + 0 + h), ly = __ldg(w + 2 + h), lz = __ldg(w + 4 + h);
        const float4 hx = __ldg(w + 6 + h), hy = __ldg(w + 8 + h), hz = __ldg(w + 10 + h);
        const float4 ci = __ldg(w + 12 + h);
        const float lox[4] = {lx.x, lx.y, lx.z, lx.w}, loy[4] = {ly.x, ly.y, ly.z, ly.w}, loz[4] = {lz.x, lz.y, lz.z, lz.w};
        const float hix[4] = {hx.x, hx.y, hx.z, hx.w}, hiy[4] = {hy.x, hy.y, hy.z, hy.w}, hiz[4] = {hz.x, hz.y, hz.z, hz.w};
        const float cw[4] = {ci.x, ci.y, ci.z, ci.w};
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const float q0x = (lox[c] - o.x) * inv.x, q1x = (hix[c] - o.x) * inv.x;
            const float q0y = (loy[c] - o.y) * inv.y, q1y = (hiy[c] - o.y) * inv.y;
            const float q0z = (loz[c] - o.z) * inv.z, q1z = (hiz[c] - o.z) * inv.z;
            const float ti = fmaxf(fmaxf(fminf(q0x, q1x), fminf(q0y, q1y)), fminf(q0z, q1z));
            const float to = fminf(fminf(fmaxf(q0x, q1x), fmaxf(q0y, q1y)), fmaxf(q0z, q1z));
            const uint32_t ii = (uint32_t)f2i(cw[c]);
            const bool hit = ii != 0u && !(to < 0.0f || ti > to * slack || ti > bt);
            tin[4 * h + c] = ti;
            cid[4 * h + c] = ii;
            if (hit) hitMask |= 1u << (4 * h + c);
        }
    }
    if (hitMask == 0u) return fastPop(T, K, bt);
    if (T.sp + 7 > CGRT_FASTSTACK) return TRAV_DEFER; // pathological depth: let the exact traversal handle the ray
    int best = -1;
    float bestT = 0.0f;
#pragma unroll
    for (int c = 0; c < 8; c++) {
        if ((hitMask >> c & 1u) && (best < 0 || tin[c] < bestT)) { best = c; bestT = tin[c]; }
    }
#pragma unroll
    for (int c = 0; c < 8; c++) {
        if ((hitMask >> c & 1u) && c != best) {
            K.e[T.sp] = make_uint2(cid[c], __float_as_uint(tin[c]));
            T.sp++;
        }
    }
    T.node = cid[best];
    return TRAV_CONTINUE;
}
template <bool ANY>
RT_DEV int fastStepWide(const DevScene& S, FastTrav& T, FastStack& K, float maxDist)
{
    return fastStepWideDyn(S, T, K, ANY, maxDist);
}

// One triangle against the search state, with the reference's accept arithmetic (same expression trees as leafCandidate).
// Returns TRAV_CONTINUE (state possibly updated), TRAV_DEFER (the outcome depends on the reference's visiting order: exact
// tie with the best, or the in-plane shortcut) or TRAV_FIRED (ANY: the shadow predicate holds for the new best).
template <bool ANY>
RT_DEV int fastTriangle(const DevScene& S, FastTrav& T, float& t2, int i, float eps, float maxDist)
{
    if (i == T.hitTri) return TRAV_CONTINUE; // already the best candidate (always-list triangles are met twice): not a tie
    // the whole 64-byte record at once: one memory round trip per triangle
    const float4* tr = S.tri4 + 4 * (size_t)i;
    const float4 pl = __ldg(tr), v0 = __ldg(tr + 1), v1 = __ldg(tr + 2), v2 = __ldg(tr + 3);
    const V3 o = T.o, d = T.d;
    const V3 n = mk3(pl);
    const float on = dot3(o, n);
    float tt = 0.0f;
    const bool shortcut = (on == pl.w);
    if (!shortcut) {
        const float denominator = dot3(d, n);
        if (denominator == 0) return TRAV_CONTINUE;
        tt = (pl.w - on) / denominator;
        if (tt < 0) return TRAV_CONTINUE;
        if (T.hitTri < 0) {
            if (!(tt < T.t)) return TRAV_CONTINUE;             // T.t is the ray's own bound: `t >= ray.t` (or NaN)
        } else if (!(tt <= T.t * CGRT_NEAR)) return TRAV_CONTINUE; // clearly farther than the best
        // (a runner-up at or beyond the ray's own bound is not acceptable; recording it anyway only makes the certificate
        // more cautious, and saves carrying the bound through the search)
    }
    const V3 p = o + d * tt;
    if (!pointInTriangleDev(mk3(v0), mk3(v1), mk3(v2), n, p)) return TRAV_CONTINUE;
    if (shortcut) return TRAV_DEFER;
    if (T.hitTri >= 0) {
        if (tt == T.t) return TRAV_DEFER;                  // exact tie: the reference keeps whichever it reaches first
        if (tt > T.t) {                                    // acceptable runner-up just behind the best
            t2 = fminf(t2, tt);
            return TRAV_CONTINUE;
        }
        t2 = fminf(t2, T.t);                               // the old best becomes the runner-up
    }
    T.t = tt;
    T.hitTri = i;
    if (ANY && !(tt + eps >= maxDist)) return TRAV_FIRED;
    return TRAV_CONTINUE;
}

// the triangles of one fast-tree leaf; `any` = shadow ray (early exit as soon as the shadow predicate holds for the best)
RT_DEV int fastStepLeafDyn(const DevScene& S, FastTrav& T, FastStack& K, bool any, float eps, float maxDist)
{
    const uint32_t id = T.node;
    const int first = (int)(id & CGRT_IDX_MASK);
    const int count = (int)((id >> CGRT_TRICNT_SHIFT) & 7u) + 1;
    const V3 o = T.o, d = T.d;
    // (fastTriangle written out: this is the hot loop of the search, and its shape matters to the compiler)
#pragma unroll 1
    for (int i = first; i < first + count; i++) {
        // the whole 64-byte record at once: one memory round trip per triangle (fast-tree order; v2.w = position in tri4)
        const float4* tr = S.tri4f + 4 * (size_t)i;
        const float4 pl = __ldg(tr), v0 = __ldg(tr + 1), v1 = __ldg(tr + 2), v2 = __ldg(tr + 3);
        const V3 n = mk3(pl);
        const float on = dot3(o, n);
        float tt = 0.0f;
        const bool shortcut = (on == pl.w);
        if (!shortcut) {
            const float denominator = dot3(d, n);
            if (denominator == 0) continue;
            tt = (pl.w - on) / denominator;
            if (tt < 0) continue;
            if (!(tt <= T.t * CGRT_NEAR)) continue;        // clearly farther than the best (or NaN)
            if (T.hitTri < 0 && !(tt < T.t)) continue;     // T.t is still the ray's own bound: `t >= ray.t`
        }
        const V3 p = o + d * tt;
        if (!pointInTriangleDev(mk3(v0), mk3(v1), mk3(v2), n, p)) continue;
        const int pos = f2i(v2.w);
        if (shortcut || (tt == T.t && pos != T.hitTri)) return TRAV_DEFER; // depends on the reference's visiting order
        if (tt >= T.t) {                                   // acceptable runner-up just behind the best (or the best itself again)
            if (pos != T.hitTri) K.t2 = fminf(K.t2, tt);
            continue;
        }
        if (T.hitTri >= 0) K.t2 = fminf(K.t2, T.t);        // the old best becomes the runner-up
        T.t = tt;
        T.hitTri = pos;
        if (any && !(tt + eps >= maxDist)) return TRAV_FIRED;
    }
    // search bound: fminf(t, maxDist) for shadow rays; closest-hit rays carry maxDist = +inf or are bounded by t alone
    return fastPop(T, K, (any ? fminf(T.t, maxDist) : T.t) * 1.000001f);
}
template <bool ANY>
RT_DEV int fastStepLeaf(const DevScene& S, FastTrav& T, FastStack& K, float eps, float maxDist)
{
    return fastStepLeafDyn(S, T, K, ANY, eps, maxDist);
}

// Closest hit: does the reference find tri* (position `pos`, distance tStar)? Until tri* is accepted the reference's ray.t is
// the ray's own bound tIn or the distance of another acceptable triangle. Every acceptable triangle closer than
// tStar * (1 + 8e-7) has been examined by the search (its pruning factor CGRT_NEAR minus the rounding of the slab arithmetic),
// the closest of them is t2; hence ray.t >= LB = min(tIn, t2, tStar * (1 + 5e-7)) > tStar at all those times. If every box on
// the path root -> leaf(tri*) contains the origin strictly (visited unconditionally) or is reported hit by the reference's own
// slabTest at a distance below LB, none of the reference's decisions on that path (`currentT >= ray.t` rejects, `ray.t <
// tSecond` prunes a pending sibling) can go against descending, whatever the order of its visits; the leaf scan then accepts
// tri* (tStar < ray.t) and nothing acceptable is closer. Boxes that are entered exactly where the triangle is hit (axis-aligned
// geometry lying in a box face: distance within a few ulp of tStar) pass thanks to the 5e-7 margin.
// The reference's slabTest (ray_tracing.cpp / rt_math.cuh slabTest: six IEEE divisions) decides for every box of the path. The
// certificates evaluate it in two stages: first with the reciprocal direction, tIn' / tOut' from (lo - o) * (1 / d). Each of
// the six products differs from the reference's quotient by less than 3 ulp (the subtraction is the same; reciprocal, product
// and quotient each round once), so tIn and tOut - a max and a min of them - lie within E = 4e-7 * (largest magnitude of the
// six) + 1e-30 of tIn', tOut'. If  tIn' > E  (the reference's entry distance is positive, so it reports tIn),
// tIn' + 2 E <= tOut'  (it reports a hit: tIn <= tOut, tOut >= 0)  the reference's distance is at most tIn' + E. Only when
// these margins do not hold (origin on a face, grazing rays, boxes entered within a few ulp of the bound, non-finite values:
// every comparison with a NaN fails) is the box evaluated with the reference's own arithmetic. The finish warps of the
// persistent wavefront are bound by the latency of this walk: ~160 dependent instructions per box with the divisions, ~45 without.
struct SlabFast {
    V3 inv;
};
RT_DEV SlabFast slabFastBegin(const V3& d)
{
    SlabFast F;
    // (directions whose reciprocal would lose precision - zero, denormal, beyond 1e30 - get NaN: every fast test then fails and
    // the reference's arithmetic decides)
    const float nan = __int_as_float(0x7fc00000);
    F.inv.x = (fabsf(d.x) >= 1e-30f && fabsf(d.x) <= 1e30f) ? 1.0f / d.x : nan;
    F.inv.y = (fabsf(d.y) >= 1e-30f && fabsf(d.y) <= 1e30f) ? 1.0f / d.y : nan;
    F.inv.z = (fabsf(d.z) >= 1e-30f && fabsf(d.z) <= 1e30f) ? 1.0f / d.z : nan;
    return F;
}
// true: the reference's slabTest(lo, hi, o, d, +inf) reports a hit at a distance <= teUpper (and > 0)
RT_DEV bool slabFastHit(const SlabFast& F, const V3& lo, const V3& hi, const V3& o, float& teUpper)
{
    const float ax = (lo.x - o.x) * F.inv.x, bx = (hi.x - o.x) * F.inv.x;
    const float ay = (lo.y - o.y) * F.inv.y, by = (hi.y - o.y) * F.inv.y;
    const float az = (lo.z - o.z) * F.inv.z, bz = (hi.z - o.z) * F.inv.z;
    const float tIn = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fminf(az, bz));
    const float tOut = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fmaxf(az, bz));
    const float big = fmaxf(fmaxf(fmaxf(fabsf(ax), fabsf(bx)), fmaxf(fabsf(ay), fabsf(by))), fmaxf(fabsf(az), fabsf(bz)));
    const float e = big * 4e-7f + 1e-30f;
    // (fminf / fmaxf drop NaN operands, so a NaN product is caught through `big`: the sum below is then NaN or the checks on
    // the individual products fail)
    const bool finite = (ax == ax) && (bx == bx) && (ay == ay) && (by == by) && (az == az) && (bz == bz) && big < 1e30f;
    teUpper = tIn + e;
    return finite && tIn > e && tIn + 2.0f * e <= tOut;
}

RT_DEV bool certifyClosest(const DevScene& S, const V3& o, const V3& d, int pos, float tStar, float t2, float tIn)
{
    const float lb = fminf(fminf(tIn, t2), tStar * 1.0000005f);
    if (!(lb > tStar)) return false;
    const SlabFast F = slabFastBegin(d);
    int node = f2i(__ldg(S.triN0 + pos).w);
#pragma unroll 1
    while (true) {
        const float4 q0 = __ldg(S.nodes + 2 * node), q1 = __ldg(S.nodes + 2 * node + 1);
        const int parent = node != 0 ? __ldg(S.refParent + node) : 0; // (fetched beside the box, not after its test)
        if (!startsInBox(o, mk3(q0), mk3(q1))) {
            float te = 0.0f;
            if (!(slabFastHit(F, mk3(q0), mk3(q1), o, te) && te < lb)) {
                if (!slabTest(mk3(q0), mk3(q1), o, d, lb, te)) return false;
                if (!(te < lb)) return false; // NaN distances are not certificates
            }
        }
        if (node == 0) return true;
        node = parent;
    }
}

// Any hit: X (position `pos`, distance tX) is acceptable and satisfies the shadow predicate. On the path root -> leaf(X) the
// reference either descends at every box - then it tests X and ends with ray.t <= tX - or it stops at a box because its ray.t
// is already at or below that box's entry distance. Its final distance is therefore at most M = max(tX, entry distances of the
// path's boxes), provided every box is geometrically hit; the predicate is monotone, so !(M + eps >= maxDist) proves "shadowed".
// (A NaN entry distance stays: `m == m` below; the predicate then fails.)
RT_DEV bool certifyAny(const DevScene& S, const V3& o, const V3& d, int pos, float tX, float eps, float maxDist)
{
    float m = tX; // an upper bound of the reference's final distance is enough: the predicate is monotone
    const SlabFast F = slabFastBegin(d);
    int node = f2i(__ldg(S.triN0 + pos).w);
#pragma unroll 1
    while (true) {
        const float4 q0 = __ldg(S.nodes + 2 * node), q1 = __ldg(S.nodes + 2 * node + 1);
        const int parent = node != 0 ? __ldg(S.refParent + node) : 0;
        if (!startsInBox(o, mk3(q0), mk3(q1))) {
            float te = 0.0f;
            if (!slabFastHit(F, mk3(q0), mk3(q1), o, te)) {
                if (!slabTest(mk3(q0), mk3(q1), o, d, __int_as_float(0x7f800000), te)) return false;
            }
            if (m == m && !(te <= m)) m = te; // (a NaN stays and fails the predicate below)
        }
        if (node == 0) break;
        node = parent;
    }
    return !(m + eps >= maxDist);
}

RT_DEV bool travIsLeaf(uint32_t node) { return (node & CGRT_TRI) != 0u; }

// The triangles the tree does not cover (DevScene::alwaysTri: extreme slivers / non-finite coordinates whose accept region has
// no bounding box): every ray that enters the reference tree tests them with the same accept arithmetic, before or after the
// search - the order does not matter to the search state (best, runner-up, defer on ties).
template <bool ANY>
RT_DEV int fastAlways(const DevScene& S, FastTrav& T, float& t2, float eps, float maxDist)
{
#pragma unroll 1
    for (int k = 0; k < S.nAlways; k++) {
        const int r = fastTriangle<ANY>(S, T, t2, __ldg(S.alwaysTri + k), eps, maxDist);
        if (r != TRAV_CONTINUE) return r;
    }
    return TRAV_CONTINUE;
}

// fastBegin + always-list, for the traversals that finish a ray in one place (batch kernels, path pipeline); the round
// pipeline's search kernels start with fastBegin only and k_finish applies the always-list to their result
template <bool ANY>
RT_DEV int fastStart(const DevScene& S, FastTrav& T, FastStack& K, const V3& o, const V3& d, float tIn, float eps, float maxDist)
{
    K.t2 = __int_as_float(0x7f800000);
    const int state = fastBegin(S, T, o, d, tIn);
    if (state != TRAV_CONTINUE || S.nAlways <= 0) return state;
    return fastAlways<ANY>(S, T, K.t2, eps, maxDist);
}

template <bool ANY>
RT_DEV int fastStep(const DevScene& S, FastTrav& T, FastStack& K, float eps, float maxDist)
{
    if (travIsLeaf(T.node)) return fastStepLeaf<ANY>(S, T, K, eps, maxDist);
    return fastStepWide<ANY>(S, T, K, maxDist);
}

// After the search: certificate, then the sphere loop of BoundingVolumeHierarchy::intersect (bvh.cpp:878-879).
// Returns false with `defer` set when the ray has to be replayed by the exact traversal.
template <bool ANY>
RT_DEV bool fastFinish(const DevScene& S, const FastTrav& T, float t2, int state, float tIn, float eps, float maxDist, TraceResult& R, bool& defer)
{
    R.sphere = -1;
    R.t = T.t;
    R.tri = T.hitTri;
    defer = false;
    if (state == TRAV_DEFER) {
        defer = true;
        return false;
    }
    if (ANY) {
        if (state == TRAV_FIRED) {
            if (!certifyAny(S, T.o, T.d, T.hitTri, T.t, eps, maxDist)) defer = true;
            return !defer;
        }
    } else if (T.hitTri >= 0) {
        if (!certifyClosest(S, T.o, T.d, T.hitTri, T.t, t2, tIn)) {
            defer = true;
            return false;
        }
    }
    float t = T.t;
    for (int s = 0; s < S.nSpheres; s++) {
        const float4 c = __ldg(S.spheres + 3 * s);
        float ts;
        V3 nn;
        if (sphereTest(mk3(c), c.w, T.o, T.d, t, ts, nn)) {
            t = ts;
            R.sphere = s;
            R.sphereN = nn;
            if (ANY && !(ts + eps >= maxDist)) {
                R.t = t;
                return true;
            }
        }
    }
    R.t = t;
    if (ANY) return false;
    return T.hitTri >= 0 || R.sphere >= 0;
}

// one ray, start to finish: speculative search first, exact replay when it cannot be certified
template <bool ANY>
RT_DEV bool traverseSpec(const DevScene& S, const V3& o, const V3& d, float tIn, float eps, float maxDist, TraceResult& R)
{
    {
        FastTrav T;
        FastStack K;
        int state = fastStart<ANY>(S, T, K, o, d, tIn, eps, maxDist);
        while (state == TRAV_CONTINUE) state = fastStep<ANY>(S, T, K, eps, maxDist);
        bool defer;
        const bool r = fastFinish<ANY>(S, T, K.t2, state, tIn, eps, maxDist, R, defer);
        if (!defer) return r;
    }
    return traverseFast<ANY>(S, o, d, tIn, eps, maxDist, R);
}

// Closest-hit traversal in the reference's exact visiting order (SURVEY.md §3.3 / Appendix A.7):
//   intersect            src/bounding_volume_hierarchy.cpp:850-881
//   intersectDataStructure :831-844   enter iff origin strictly inside root box OR slab test passes against ray.t
//   intersectNonLeaf     :715-736     slab-test BOTH children against the current ray.t (tLeft/tRight, -1 = miss)
//   intersectDeeper      :679-701     classify by startsInBox
//   intersectChildrenHierarchically :572-595, intersectRayThatStartsOutsideBoxes :611-635 (with the intended `return`s)
//   intersectLeaf        :535-553     (through leafCandidate, see above)
// The recursion is unrolled onto an explicit stack of (node, tSecond): the pending sibling is skipped at pop time iff
// ray.t < tSecond, which equals the reference's `hitFirst && ray.t < tSecond` because tSecond < ray.t held when it was pushed.
// ANY = true adds an early exit as soon as an accepted hit satisfies the shadow predicate !(t + eps >= maxDist)
// (pointInShadow, src/main.cpp:104-135); later accepted hits can only be closer, so the answer equals the closest-hit one.
// This variant scans every leaf sequentially (no sub-tree) and, with COUNT = true, counts the reference's box / triangle tests;
// the kernels use it for the counting passes, traverseFast above for production.
template <bool ANY, bool COUNT>
RT_DEV bool traverseStrict(const DevScene& S, const V3& o, const V3& d, float tIn, float eps, float maxDist, TraceResult& R,
                           uint32_t& nBox, uint32_t& nTri)
{
    float t = tIn;
    int hitTri = -1;
    R.sphere = -1;
    if (S.nNodes > 0) {
        float4 q0 = __ldg(S.nodes + 0), q1 = __ldg(S.nodes + 1);
        bool enter = startsInBox(o, mk3(q0), mk3(q1));
        if (!enter) {
            float tmp;
            if (COUNT) nBox++;
            enter = slabTest(mk3(q0), mk3(q1), o, d, t, tmp);
        }
        if (enter) {
            int stN[CGRT_STACK];
            float stT[CGRT_STACK];
            int sp = 0;
            int cur = 0;
            uint32_t a = (uint32_t)f2i(q0.w), b = (uint32_t)f2i(q1.w);
            while (true) {
                if (b != 0u) {
                    // ---- intersectLeaf
                    LeafBest best;
                    best.t = t;
                    best.pos = -1;
                    best.rank = -1;
                    best.shortcut = false;
                    if (COUNT) nTri += b;
                    {
                        const uint32_t end = a + b;
                        for (uint32_t i = a; i < end; i++) {
                            if (leafCandidate(S, (int)i, o, d, best)) {
                                if (ANY && !(best.t + eps >= maxDist)) {
                                    R.t = best.t;
                                    R.tri = best.pos;
                                    return true;
                                }
                            }
                        }
                    }
                    if (best.pos >= 0) {
                        t = best.t;
                        hitTri = best.pos;
                    }
                    // ---- return to the nearest pending sibling that is not pruned
                    bool found = false;
                    while (sp > 0) {
                        sp--;
                        if (t < stT[sp]) continue;
                        cur = stN[sp];
                        q0 = __ldg(S.nodes + 2 * cur);
                        q1 = __ldg(S.nodes + 2 * cur + 1);
                        a = (uint32_t)f2i(q0.w);
                        b = (uint32_t)f2i(q1.w);
                        found = true;
                        break;
                    }
                    if (!found) break;
                } else {
                    // ---- intersectNonLeaf + intersectDeeper
                    const int L = (int)a, Rn = (int)a + 1;
                    const float4 l0 = __ldg(S.nodes + 2 * L), l1 = __ldg(S.nodes + 2 * L + 1);
                    const float4 r0 = __ldg(S.nodes + 2 * L + 2), r1 = __ldg(S.nodes + 2 * L + 3);
                    float tL = -1.0f, tR = -1.0f, tmp;
                    if (COUNT) nBox += 2;
                    if (slabTest(mk3(l0), mk3(l1), o, d, t, tmp)) tL = tmp;
                    if (slabTest(mk3(r0), mk3(r1), o, d, t, tmp)) tR = tmp;
                    const bool inL = startsInBox(o, mk3(l0), mk3(l1));
                    const bool inR = startsInBox(o, mk3(r0), mk3(r1));
                    int first = -1, second = -1;
                    float tS = -1.0f;
                    if (inL && inR) { // both visited unconditionally, left operand of `|` first (g++ order)
                        first = L; second = Rn; tS = -1.0f;
                    } else if (inL) {
                        first = L;
                        if (!(tR < 0)) { second = Rn; tS = tR; }
                    } else if (inR) {
                        first = Rn;
                        if (!(tL < 0)) { second = L; tS = tL; }
                    } else {
                        if (tL < 0 && tR < 0) {
                        } else if (tL < 0) {
                            first = Rn;
                        } else if (tR < 0) {
                            first = L;
                        } else if (tL < tR) {
                            first = L; second = Rn; tS = tR;
                        } else {
                            first = Rn; second = L; tS = tL;
                        }
                    }
                    if (second >= 0) {
                        stN[sp] = second;
                        stT[sp] = tS;
                        sp++;
                    }
                    if (first >= 0) {
                        cur = first;
                        if (first == L) { a = (uint32_t)f2i(l0.w); b = (uint32_t)f2i(l1.w); }
                        else { a = (uint32_t)f2i(r0.w); b = (uint32_t)f2i(r1.w); }
                    } else {
                        bool found = false;
                        while (sp > 0) {
                            sp--;
                            if (t < stT[sp]) continue;
                            cur = stN[sp];
                            q0 = __ldg(S.nodes + 2 * cur);
                            q1 = __ldg(S.nodes + 2 * cur + 1);
                            a = (uint32_t)f2i(q0.w);
                            b = (uint32_t)f2i(q1.w);
                            found = true;
                            break;
                        }
                        if (!found) break;
                    }
                }
            }
        }
    }
    // ---- sphere loop, src/bounding_volume_hierarchy.cpp:878-879
    for (int s = 0; s < S.nSpheres; s++) {
        const float4 c = __ldg(S.spheres + 3 * s);
        float ts;
        V3 nn;
        if (sphereTest(mk3(c), c.w, o, d, t, ts, nn)) {
            t = ts;
            R.sphere = s;
            R.sphereN = nn;
            if (ANY && !(ts + eps >= maxDist)) {
                R.t = t;
                R.tri = hitTri;
                return true;
            }
        }
    }
    R.t = t;
    R.tri = hitTri;
    if (ANY) return false;
    return hitTri >= 0 || R.sphere >= 0;
}
