// Persistent wavefront: ONE kernel per frame (included by cgrt_kernels.cu after the round pipeline, whose per-ray code it shares).
//
// The round pipeline (k_gen -> { k_trace | k_trace8 -> k_finish } per level -> k_shade_slots) pays one kernel boundary per
// level and chain: every search launch ends with the warp that holds its longest rays, and nothing of level k+1 can start
// before the last ray of level k is done (profiles/r01_tuning.md: ~200 us per boundary in the one-lane search, ~65 us in the
// cooperative one; 1.50x at 8 GPUs). Here the levels overlap: the recursion of getFinalColor / trace / shade
// (src/main.cpp:241-310) becomes two device-side queues, and a finished closest-hit ray's shadow rays and reflection ray are
// picked up by whichever warp is free while the stragglers of the previous level are still searching.
//
//   phase A  every CTA generates its share of the primary rays (main.cpp:691-694, trackball.cpp:92-103; the reference's
//            root-box test bvh.cpp:831-844 culls the rays that cannot enter the tree) and appends them to the RAY queue
//   phase B  SEARCH warps: take rays from the ray queue, run the speculative search (nothing but steps), append (ray, result)
//            to the FINISH queue.  FINISH warps: take finished searches, 32 at a time, converged: certificate / exact replay,
//            sphere loop, fp64 hit epilogue, hit record, lit flag, and the emission of the hit's shadow rays and reflection ray
//            into the ray queue.
//            The two roles live on different SMs (role = f(%smid)): the first version of this kernel ran both on every warp and
//            lost more to instruction fetch than it gained (ncu: no_instruction 6.5 stalled warps per issue, 208 KB of SASS
//            against a 32 KB instruction cache per SM); with one role per SM each SM's working set is one loop.
//   phase C  when the frame's last ray has been finished: shading() / shade() per pixel slot (main.cpp:61-98, 160-264)
//
// Queues: append-only arrays indexed by TICKET. Producers reserve tickets with one atomicAdd on `tail` per warp and write
// the records: 16-byte chunks, each stored with one single-copy-atomic 128-bit access and each carrying the frame's sequence
// number, so a record needs no separate "published" flag and no fence - it is complete exactly when all its tags match.
// Consumers take tickets with one atomicAdd on `head` per warp - also tickets of records that do not exist yet - and read
// their own record (one round trip to L2: no shared hot word, no CAS loop, no flag-then-data dependency); a record that is
// produced while consumers wait is picked up by the lane that already holds its ticket.
// Termination: a 64-bit counter (CTAs that finished phase A << 32 | rays created and not yet finished); whoever brings it to
// (gridDim.x << 32) raises the done flags every waiting warp polls.
//
// Two search forms:
//   LANE   one lane per ray (k_trace's loop): highest throughput. A warp refills when CGRT_WAVE_REFILL of its lanes are free:
//          a refill is two L2 round trips (tickets + finish-queue positions, then the records) for the whole warp
//   GROUP  eight lanes per ray (k_trace8's step): one child box / one triangle per lane, ~5x lower latency per step; bursts of
//          CGRT_WAVE_GSTEPS steps between bookkeeping rounds
// Small frames (WaveQ::mode 2, chosen on the host from the size of the rank's share of the frame) use GROUP throughout. Large
// frames start in LANE form and change over ONCE, when the number of rays in flight has fallen below WaveQ::switchBelow: the
// ray queue is closed (a bit in its tail counter), later rays go to a second part of the same array with its own counters and
// a different tag. The LANE warps then (a) keep taking tickets until each has been handed one beyond the closing value - every
// record of the first part is held by a lane, however far the consumers were behind -, (b) pass rays that arrive late on to
// the second part, (c) hand the rays they are still searching over WITH their search state (best candidate, runner-up, stack:
// WaveQ::resume), and join the GROUP form - so the long tail of a frame (few rays, each many dependent steps) runs in the
// low-latency form without repeating work, while the bulk runs in the high-throughput one.
// Results do not depend on the form, on which warp handles a ray or on WaveQ::finEvery (same search, same certificate), only
// the time does: tests/test_gpu_parity.py test_scheduling_variants_render_the_same_frame, tools/wave_check.py.
#pragma once

#define WAVE_NSTAT 40
#define WAVE_STAT_PATHS 0
#define WAVE_STAT_HIT 1     // + level (CGRT_MAX_LEVELS)
#define WAVE_STAT_BOUNCE 17 // + level (CGRT_MAX_LEVELS + 1)
#define WAVE_STAT_REPLAYC 35
#define WAVE_STAT_REPLAYS 36
struct WaveShared {
    int stat[WAVE_NSTAT];             // finish warps: ray statistics of the frame, flushed once per CTA
    uint2 gstack[16][CGRT_STACK8];    // GROUP form: traversal stack of each 8-lane group
};

enum { WS_NONE = 0, WS_WAIT = 1, WS_RUN = 2, WS_PASS = 3 };

// Flags, counters and queue records are read with relaxed gpu-scope loads (served by L2, never by L1). An acquire load would
// make the SM drop its whole L1 (CCTL.IVALL in the SASS) - and with it the BVH nodes of every warp that is searching - on every
// poll; so would __threadfence() (MEMBAR.SC.GPU + CCTL.IVALL on sm_100a). Where earlier writes of a thread must be visible
// GPU-wide before something it does next (the frame's records before the counter decrement that may complete the frame),
// waveRelease() is used: a release reduction of 0 on a scratch word = MEMBAR.ALL.GPU without the invalidation.
RT_DEV unsigned ldRelaxedGpu(const unsigned* p)
{
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
RT_DEV void stRelaxedGpu(unsigned* p, unsigned v) { asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
// 128-bit accesses with the .b128 type are single-copy atomic (a reader sees all 16 bytes of one store or none of them)
RT_DEV float4 ld128(const float4* p)
{
    unsigned long long lo, hi;
    asm volatile("{ .reg .b128 t; ld.relaxed.gpu.global.b128 t, [%2]; mov.b128 {%0, %1}, t; }" : "=l"(lo), "=l"(hi) : "l"(p) : "memory");
    return make_float4(__uint_as_float((unsigned)lo), __uint_as_float((unsigned)(lo >> 32)), __uint_as_float((unsigned)hi),
                       __uint_as_float((unsigned)(hi >> 32)));
}
RT_DEV void st128(float4* p, const float4& v)
{
    const unsigned long long lo = (unsigned long long)__float_as_uint(v.x) | ((unsigned long long)__float_as_uint(v.y) << 32);
    const unsigned long long hi = (unsigned long long)__float_as_uint(v.z) | ((unsigned long long)__float_as_uint(v.w) << 32);
    asm volatile("{ .reg .b128 t; mov.b128 t, {%1, %2}; st.relaxed.gpu.global.b128 [%0], t; }" ::"l"(p), "l"(lo), "l"(hi) : "memory");
}
RT_DEV void waveRelease(const WaveQ& Q)
{
    int* scratch = Q.ctl + WCTL_SCRATCH + 32 * ((blockIdx.x * 4 + (threadIdx.x >> 5)) & 31);
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(scratch), "r"(0) : "memory");
}
RT_DEV unsigned long long globalTimerNs()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
RT_DEV unsigned smId()
{
    unsigned v;
    asm("mov.u32 %0, %%smid;" : "=r"(v));
    return v;
}

// instrumented builds (-DCGRT_WAVE_LAT): per ray ticket [emitted, search started, steps, search ended, finish loaded, finish done,
// form (1 LANE, 2 GROUP, +4 resumed), -] - times in ns since the frame's origin (low 32 bits of %globaltimer - WCTL_T0)
#ifdef CGRT_WAVE_LAT
RT_DEV void waveLat(const WaveQ& Q, int tk, int k, unsigned v)
{
    if (Q.lat != nullptr && tk >= 0 && tk < Q.cap) Q.lat[16 * (size_t)tk + k] = v;
}
RT_DEV unsigned waveNow(const WaveQ& Q) { return (unsigned)globalTimerNs() - ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_T0); }
#define WAVE_LAT(tk, k, v) waveLat(Q, tk, k, v)
#define WAVE_LAT_NOW(tk, k) waveLat(Q, tk, k, waveNow(Q))
#else
#define WAVE_LAT(tk, k, v)
#define WAVE_LAT_NOW(tk, k)
#endif

// ---- queue primitives ---------------------------------------------------------------------------------------------------------
// Ray record (3 chunks): [origin | tag] [direction | tag] [bound, meta, resume, tag]. tag = sequence number of the frame;
// resume = 0, or (1 + index of the search state this ray continues from) | stack depth << 24 (hand-over at the change-over).
//   closest-hit ray: meta = level << 26 | pixel slot, bound = ray.t on entry (FLT_MAX for primary rays, |D| for reflections,
//                    main.cpp:252-256); its search range is unbounded
//   shadow ray     : meta = CGRT_RAY_ANY | index of its lit flag, bound = distance to the light (pointInShadow casts it with
//                    t = FLT_MAX, main.cpp:104-135); eps = 0.001
// Finish record (2 chunks): [ray ticket, state, t, tag] [tri, runner-up t2, tag, tag]  - the result of the ray's search
#define WAVE_SLOT_BITS 26
#define WAVE_CLOSED 0x40000000    // bit of the ray queue's tail counter: the first part of the queue is closed
#define WAVE_TAG2 0x80000000u     // tag of records in the second part: seq | WAVE_TAG2
RT_DEV void waveStoreRay(const WaveQ& Q, int tk, unsigned tagBits, const V3& o, const V3& d, float bound, int meta)
{
    if (tk >= Q.cap) return; // (cannot happen: the array holds every ray a frame can cast)
    float4* q = Q.rays + 3 * (size_t)tk;
    const float tag = __uint_as_float(tagBits);
    st128(q, make_float4(o.x, o.y, o.z, tag));
    st128(q + 1, make_float4(d.x, d.y, d.z, tag));
    st128(q + 2, make_float4(bound, i2f(meta), 0.0f, tag));
    WAVE_LAT_NOW(tk, 0);
}
// one round trip: the record of ticket tk if it is complete. Unpacked into the (a, b, c) form the per-ray code shares with the
// round pipeline: a = [o | tIn], b = [d | maxDist], c = [slot, level or CGRT_RAY_ANY | lit index, eps, -]
// c.w = the record's resume word
RT_DEV bool waveLoadRay(const WaveQ& Q, int tk, unsigned tagBits, float4& a, float4& b, float4& c)
{
    if (tk >= Q.cap) return false; // a ticket beyond every ray the frame can produce: it is never served
    const float4* r = Q.rays + 3 * (size_t)tk;
    a = ld128(r);
    b = ld128(r + 1);
    const float4 m = ld128(r + 2);
    const unsigned s = tagBits;
    const bool ok = __float_as_uint(a.w) == s && __float_as_uint(b.w) == s && __float_as_uint(m.w) == s;
    const int meta = f2i(m.y);
    if (meta & CGRT_RAY_ANY) {
        a.w = FLT_MAX;
        b.w = m.x;
        c = make_float4(0.0f, m.y, 0.001f, m.z);
    } else {
        a.w = m.x;
        b.w = __int_as_float(0x7f800000);
        c = make_float4(i2f(meta & ((1 << WAVE_SLOT_BITS) - 1)), i2f(meta >> WAVE_SLOT_BITS), 0.0f, m.z);
    }
    return ok;
}
// cheap poll for a warp that has nothing else to do: ONE lane looks at ONE word (the last tag) of the record with the lowest
// ticket the warp is waiting for - records are served roughly in ticket order, so if that one is not there the others are not
// worth 32 x 48 bytes of loads and the instructions to check them. `mine`: this lane waits on ticket tk. Warp-uniform result.
RT_DEV bool wavePeekRay(const WaveQ& Q, bool mine, int tk, unsigned tagBits)
{
    const unsigned m = __ballot_sync(0xffffffffu, mine);
    if (m == 0u) return false;
    const int lowest = __reduce_min_sync(0xffffffffu, mine ? tk : 0x7fffffff);
    unsigned w = 0u;
    if ((threadIdx.x & 31) == 0 && lowest < Q.cap) w = ldRelaxedGpu((const unsigned*)(Q.rays + 3 * (size_t)lowest) + 11);
    return __shfl_sync(0xffffffffu, w, 0) == tagBits;
}
RT_DEV bool wavePeekFin(const WaveQ& Q, bool mine, int ftk)
{
    const unsigned m = __ballot_sync(0xffffffffu, mine);
    if (m == 0u) return false;
    const int lowest = __reduce_min_sync(0xffffffffu, mine ? ftk : 0x7fffffff);
    unsigned w = 0u;
    if ((threadIdx.x & 31) == 0 && lowest < Q.cap) w = ldRelaxedGpu((const unsigned*)(Q.fin + 2 * (size_t)lowest) + 7);
    return __shfl_sync(0xffffffffu, w, 0) == Q.seq;
}
// one thread (lane 0 of a producing warp): reserve n consecutive records of the ray array; `closedSeen` is the warp's memory
// of the change-over. Returns the array index of the first record and the tag its records must carry.
RT_DEV int waveReserve(const WaveQ& Q, int n, bool& closedSeen, unsigned& tagBits)
{
    if (!closedSeen) {
        const int old = atomicAdd(Q.ctl + WCTL_TAIL, n);
        if (!(old & WAVE_CLOSED)) {
            tagBits = Q.seq;
            return old;
        }
        closedSeen = true; // (the add went to a closed counter: harmless, the closing value is kept in WCTL_CLOSEAT)
    }
    const int t2 = atomicAdd(Q.ctl + WCTL_TAIL2, n);
    unsigned ca;
    while ((ca = ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_CLOSEAT)) == 0u) { } // written right after the closing bit
    tagBits = Q.seq | WAVE_TAG2;
    return (int)(ca - 1u) + t2;
}
// warp-converged: take n tickets of the queue whose head counter is at ctl[headIdx]
RT_DEV int waveClaim(const WaveQ& Q, int headIdx, int n)
{
    int base = 0;
    if ((threadIdx.x & 31) == 0) base = atomicAdd(Q.ctl + headIdx, n);
    return __shfl_sync(0xffffffffu, base, 0);
}
// warp-converged: the lanes with `mine` append their finished search (ray ticket, state, t, tri, t2) to the finish queue
RT_DEV void waveFinPush(const WaveQ& Q, bool mine, int tk, int state, float t, int tri, float t2)
{
    const unsigned mask = __ballot_sync(0xffffffffu, mine);
    if (mask == 0u) return;
    const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(Q.ctl + WCTL_FTAIL, __popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (mine) {
        const int pos = base + __popc(mask & ((1u << lane) - 1u));
        if (pos < Q.cap) {
            const float tag = __uint_as_float(Q.seq);
            st128(Q.fin + 2 * (size_t)pos, make_float4(i2f(tk), i2f(state), t, tag));
            st128(Q.fin + 2 * (size_t)pos + 1, make_float4(i2f(tri), t2, tag, tag));
        }
    }
}
RT_DEV bool waveLoadFin(const WaveQ& Q, int ftk, int& tk, float4& res)
{
    if (ftk >= Q.cap) return false;
    const float4 c0 = ld128(Q.fin + 2 * (size_t)ftk), c1 = ld128(Q.fin + 2 * (size_t)ftk + 1);
    const unsigned s = Q.seq;
    tk = f2i(c0.x);
    res = make_float4(c0.y, c0.z, c1.x, c1.y); // (state, t, tri, t2)
    return __float_as_uint(c0.w) == s && __float_as_uint(c1.z) == s && __float_as_uint(c1.w) == s;
}
// one thread: the frame is complete (or the watchdog fired): raise every copy of the done flag
RT_DEV void waveRaiseDone(const WaveQ& Q)
{
    waveRelease(Q);
#pragma unroll 1
    for (int k = 0; k < 32; k++) stRelaxedGpu((unsigned*)Q.ctl + WCTL_DONE + 32 * k, 1u);
}
// one thread: rays created (+) / finished (-); the thread that completes the frame raises the flags. The thread that sees the
// number of rays in flight fall below switchBelow (exact once every CTA has reported phase A) closes the first part of the queue
RT_DEV void wavePending(const WaveQ& Q, long long delta)
{
    unsigned long long* pend = (unsigned long long*)Q.ctl;
    const unsigned long long now = atomicAdd(pend, (unsigned long long)delta) + (unsigned long long)delta;
    if (now == ((unsigned long long)gridDim.x << 32)) {
        waveRaiseDone(Q);
    } else if (delta < 0 && Q.switchBelow > 0 && (now >> 32) == (unsigned long long)gridDim.x && (unsigned)now < (unsigned)Q.switchBelow) {
        if (ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_CLOSEAT) == 0u) {
            const int old = atomicOr(Q.ctl + WCTL_TAIL, WAVE_CLOSED);
            if (!(old & WAVE_CLOSED)) stRelaxedGpu((unsigned*)Q.ctl + WCTL_CLOSEAT, (unsigned)old + 1u);
        }
    }
}
// fire-and-forget form for increments (a reduction: nothing waits for it). It is issued before the atomic that reserves the
// children's records, whose result the warp does wait for, so it is performed long before a child can be finished.
RT_DEV void wavePendingAdd(const WaveQ& Q, int created) { atomicAdd((unsigned long long*)Q.ctl, (unsigned long long)created); }
// the decrement in two halves: issue now, look at the result later (on the next trip round the finish loop), so that the round
// trip overlaps the next batch's loads
RT_DEV unsigned long long wavePendingIssue(const WaveQ& Q, long long delta)
{
    return atomicAdd((unsigned long long*)Q.ctl, (unsigned long long)delta) + (unsigned long long)delta;
}
RT_DEV void wavePendingCheck(const WaveQ& Q, unsigned long long now)
{
    if (now == ((unsigned long long)gridDim.x << 32)) {
        waveRaiseDone(Q);
    } else if (Q.switchBelow > 0 && (now >> 32) == (unsigned long long)gridDim.x && (unsigned)now < (unsigned)Q.switchBelow) {
        if (ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_CLOSEAT) == 0u) {
            const int old = atomicOr(Q.ctl + WCTL_TAIL, WAVE_CLOSED);
            if (!(old & WAVE_CLOSED)) stRelaxedGpu((unsigned*)Q.ctl + WCTL_CLOSEAT, (unsigned)old + 1u);
        }
    }
}
// warp-converged and warp-uniform (phase C reads the other CTAs' records through L2 afterwards)
RT_DEV bool waveDone(const WaveQ& Q)
{
    const int w = (blockIdx.x * 4 + (threadIdx.x >> 5)) & 31;
    unsigned f = 0u;
    if ((threadIdx.x & 31) == 0) f = ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_DONE + 32 * w);
    return __shfl_sync(0xffffffffu, f, 0) != 0u;
}
// idle warps: back off a little, and give up when the frame has been running for longer than the watchdog allows (a protocol
// bug must not hang the GPU)
#ifndef CGRT_WAVE_IDLE_MAX
#define CGRT_WAVE_IDLE_MAX 1000
#endif
RT_DEV void waveIdle(const WaveQ& Q, unsigned long long t0, int& idlePolls)
{
    __nanosleep(idlePolls < 8 ? 100 : (idlePolls < 32 ? 250 : (idlePolls < 128 ? 500 : CGRT_WAVE_IDLE_MAX)));
    if ((++idlePolls & 63) == 0 && (threadIdx.x & 31) == 0 && globalTimerNs() - t0 > Q.timeoutNs) {
        atomicExch(Q.ctl + WCTL_ERR, 1);
        waveRaiseDone(Q);
    }
}

// optional timeline of the frame (CGRT_WAVE_TRACE=1): a few finish warps sample the counters once per 4.096 us bucket
RT_DEV void waveTraceSample(const WaveQ& Q, int& lastBucket)
{
    if (Q.trace == nullptr || (blockIdx.x & 15) != 0 || (threadIdx.x & 127) != 0) return;
    const unsigned t0 = ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_T0);
    const int bucket = (int)(((unsigned)globalTimerNs() - t0) >> 12);
    if (bucket == lastBucket || bucket < 0 || bucket >= WAVE_TRACE_SAMPLES) return;
    lastBucket = bucket;
    int* o = Q.trace + 8 * bucket;
    o[1] = (int)ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_PENDING);
    o[2] = (int)ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_HEAD);
    o[3] = (int)ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_TAIL);
    o[4] = (int)ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_FHEAD);
    o[5] = (int)ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_FTAIL);
    o[6] = (int)ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_HEAD2);
    o[7] = (int)ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_TAIL2);
    o[0] = 1;
}

// ---- FINISH warps ---------------------------------------------------------------------------------------------------------------
// Every lane holds a ticket of the finish queue; tickets are handed out in order, so the 32 tickets of a warp are served by 32
// consecutively finished searches - under load within a poll interval, and the batch then runs fully converged. A partly
// served warp waits a few polls for the rest, then processes what it has (the end of a frame, small frames).
#ifndef CGRT_WAVE_FIN_WAIT
#define CGRT_WAVE_FIN_WAIT 3
#endif
RT_DEV void waveFinishLoop(const DevScene& S, const FrameParams& P, const float4* __restrict__ lights, const WaveQ& Q,
                           const RoundBuffers& B, const int2* __restrict__ tileSeq, float* __restrict__ fb, WaveShared& sh,
                           unsigned long long t0)
{
    const int lane = threadIdx.x & 31;
    const unsigned ltMask = (1u << lane) - 1u;
    const int nL = P.nLights;
    int ftk = -1;        // ticket of the finish queue held by this lane
    int waited = 0, idlePolls = 0;
    bool closedSeen = false; // lane 0: this warp has seen the ray queue's change-over
    int traceBucket = -1;
    // round trips to L2 are what a batch costs (the finish warps are latency-bound), so: the tickets that replace a batch's are
    // claimed while the batch is processed (nextBase), the counter decrement of a batch is looked at one trip later (pendNow),
    // and the cheap look before the full poll is skipped while every poll finds a full batch (busy)
    int nextBase = 0, nextCount = 0; // lane 0 issued the claim; everyone knows the count
    unsigned long long pendNow = 0ull;
    bool havePend = false, busy = false;
    {
        const int base = waveClaim(Q, WCTL_FHEAD, 32);
        ftk = base + lane;
    }
    while (true) {
        waveTraceSample(Q, traceBucket);
        // ---- the tickets claimed during the last batch go to the lanes that have none
        if (nextCount) {
            const unsigned noneMask = __ballot_sync(0xffffffffu, ftk < 0);
            const int base = __shfl_sync(0xffffffffu, nextBase, 0);
            if (ftk < 0) ftk = base + __popc(noneMask & ltMask);
            nextCount = 0;
        }
        // ---- which of the warp's tickets have been served? (a cheap look first: see wavePeekRay)
        int tk = -1;
        float4 res = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        const bool ready = (busy || waited > 0 || wavePeekFin(Q, true, ftk)) && waveLoadFin(Q, ftk, tk, res);
        if (havePend) { // (lane 0) the result of the last batch's decrement: frame complete? change-over due?
            wavePendingCheck(Q, pendNow);
            havePend = false;
        }
        const unsigned readyMask = __ballot_sync(0xffffffffu, ready);
        if (readyMask == 0u) {
            busy = false;
            if (waveDone(Q)) break;
            waveIdle(Q, t0, idlePolls);
            continue;
        }
        idlePolls = 0;
        // under load the rest of a partly served batch arrives within a poll or two: wait for it; otherwise finish at once
        if (readyMask != 0xffffffffu && busy && ++waited < CGRT_WAVE_FIN_WAIT) continue;
        busy = readyMask == 0xffffffffu && waited == 0;
        waited = 0;
        // replacement tickets for the lanes of this batch: issued now, used on the next trip
        nextCount = __popc(readyMask);
        if (lane == 0) nextBase = atomicAdd(Q.ctl + WCTL_FHEAD, nextCount);
        // ---- the batch: one lane per finished search
        const int n = __popc(readyMask);
        bool hit = false, bounce = false, replayC = false, replayS = false;
        V3 pointOn = mk3(0.0f, 0.0f, 0.0f), nn = pointOn, rd = pointOn;
        int slot = 0, rec = 0, level = 0;
        if (ready) {
            ftk = -1;
            float4 a, b, c;
            WAVE_LAT_NOW(tk, 4);
            waveLoadRay(Q, tk, 0u, a, b, c); // (complete: the searcher validated it)
            const int meta = f2i(c.y);
#ifdef CGRT_WAVE_LAT
            if (a.x == 1e38f) return; // (keeps the loads above the time stamp)
            WAVE_LAT_NOW(tk, 8);
#endif
            if (meta & CGRT_RAY_ANY) { // ---- shadow ray: lit flag
                const bool shadowed = finishShadowRay<true>(S, a, b, c, res, replayS);
                WAVE_LAT_NOW(tk, 9);
                B.lit[meta & 0x3fffffff] = shadowed ? 0 : 1;
            } else { // ---- closest-hit ray of `level`
                const V3 o = mk3(a), d = mk3(b);
                slot = f2i(c.x);
                level = meta;
                TraceResult R;
                hit = finishClosestRay<true>(S, a, b, res, R, replayC);
#ifdef CGRT_WAVE_LAT
                if (R.t == -1e38f) return;
                WAVE_LAT_NOW(tk, 9);
#endif
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
                    atomicAdd(&sh.stat[WAVE_STAT_HIT + level], 1);
                    if (level == 0) atomicAdd(&sh.stat[WAVE_STAT_PATHS], 1);
                    if (bounce) atomicAdd(&sh.stat[WAVE_STAT_BOUNCE + level + 1], 1);
                    WAVE_LAT_NOW(tk, 10);
                }
                if (replayC) atomicAdd(&sh.stat[WAVE_STAT_REPLAYC], 1);
            }
            if (replayS) atomicAdd(&sh.stat[WAVE_STAT_REPLAYS], 1);
        }
        // ---- emission: tickets for the shadow rays of the batch first (lane order), then for its reflection rays, so that
        // any-hit and closest-hit rays sit in runs
        const int nShadow = hit ? nL : 0, nBounce = bounce ? 1 : 0;
        int sIncl = nShadow, bIncl = nBounce;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int vs = __shfl_up_sync(0xffffffffu, sIncl, o), vb = __shfl_up_sync(0xffffffffu, bIncl, o);
            if (lane >= o) { sIncl += vs; bIncl += vb; }
        }
        const int totS = __shfl_sync(0xffffffffu, sIncl, 31), totB = __shfl_sync(0xffffffffu, bIncl, 31);
        int base = 0;
        unsigned tagBits = 0u;
        if (lane == 0 && totS + totB > 0) {
            wavePendingAdd(Q, totS + totB); // the children are counted before they can become visible
            base = waveReserve(Q, totS + totB, closedSeen, tagBits);
        }
        base = __shfl_sync(0xffffffffu, base, 0);
        tagBits = __shfl_sync(0xffffffffu, tagBits, 0);
        if (ready) WAVE_LAT_NOW(tk, 11);
        if (hit && nL > 0) {
            const int firstS = base + sIncl - nShadow;
            for (int l = 0; l < nL; l++) {
                V3 org, dir;
                float dist;
                shadowRayOf(lights, l, pointOn, org, dir, dist);
                waveStoreRay(Q, firstS + l, tagBits, org, dir, dist, CGRT_RAY_ANY | (rec * nL + l));
            }
        }
        if (bounce) {
            V3 org, dir;
            float tIn;
            reflectionRayOf(pointOn, rd, nn, org, dir, tIn);
            waveStoreRay(Q, base + totS + bIncl - 1, tagBits, org, dir, tIn, ((level + 1) << WAVE_SLOT_BITS) | slot);
        }
        // (the children are visible as soon as their records are complete; no flag, no fence. What the batch wrote for phase C -
        // hit records, lit flags, black pixels - is released once, when this warp leaves the loop.)
        if (ready) WAVE_LAT_NOW(tk, 5);
        if (lane == 0) {
            pendNow = wavePendingIssue(Q, -(long long)n);
            havePend = true;
        }
    }
    // everything this warp wrote for phase C is visible GPU-wide before it reports out; phase C starts when every finish warp has
    waveRelease(Q);
    __syncwarp();
    if (lane == 0) atomicAdd(Q.ctl + WCTL_FINEXIT, 1);
}

// ---- SEARCH warps, LANE form: one lane per ray (the loop of k_trace on tickets) -------------------------------------------
#ifndef CGRT_WAVE_STEPS
#define CGRT_WAVE_STEPS 8
#endif
#ifndef CGRT_WAVE_REFILL
#define CGRT_WAVE_REFILL 16 // lanes that must be free before a warp refills (4 / 8 / 16 / 24 / 32: 1.22 / 1.17 / 1.06 / 1.06 / 1.16 ms on C3: a refill is two L2 round trips for the whole warp)
#endif
#ifndef CGRT_WAVE_GFIN
#define CGRT_WAVE_GFIN 1 // GROUP form: finished groups that end a burst early
#endif
#ifndef CGRT_WAVE_GSTEPS
#define CGRT_WAVE_GSTEPS 8 // GROUP form: steps per burst (measured 2 / 4 / 8: 0.44 / 0.415 / 0.40 ms on a 1/8 share of C3)
#endif
// Returns when the frame is done (true) or when the queue has changed over and this warp holds no LANE ray any more (false).
RT_DEV bool waveLaneLoop(const DevScene& S, const WaveQ& Q, unsigned long long t0)
{
    const int lane = threadIdx.x & 31;
    const unsigned ltMask = (1u << lane) - 1u;
    FastTrav T;
    FastStack K;
    int tk = -1, st = WS_NONE, state = TRAV_DONE;
    float eps = 0.0f, maxDist = 0.0f;
    bool any = false;
    int idlePolls = 0;
    int closeAt = 0x7fffffff; // tickets from this value on will never be served (known once the change-over has been seen)
    bool drained = false;     // this warp has been handed a ticket >= closeAt: the first part of the queue holds nothing for it any more
    T.t = 0.0f; T.hitTri = -1; T.node = 0u; T.sp = 0;
    K.t2 = 0.0f;
    while (true) {
        // ---- 1. finished searches go to the finish queue, idle lanes take tickets (also of rays that do not exist yet: their
        // lanes wait) - both counters in one round trip
        const bool fin = st == WS_RUN && state != TRAV_CONTINUE;
        const unsigned finMask = __ballot_sync(0xffffffffu, fin);
        const unsigned runMask = __ballot_sync(0xffffffffu, st == WS_RUN && !fin);
        const unsigned waitMask = __ballot_sync(0xffffffffu, st == WS_WAIT);
        const unsigned noneMask = __ballot_sync(0xffffffffu, st == WS_NONE || fin);
        const int nNone = __popc(noneMask), nFin = __popc(finMask);
        const bool open = closeAt == 0x7fffffff;
        // (after the change-over the warps keep taking tickets until each has been handed one beyond the closing value: every
        // record of the first part is then held by a lane, however far the consumers were behind when the queue closed)
        const int want = (!drained && (!open || nNone >= CGRT_WAVE_REFILL || runMask == 0u) && nNone > 0) ? nNone : 0;
        int fbase = 0, base = 0;
        unsigned ca = 0u;
        if (lane == 0) {
            if (nFin) fbase = atomicAdd(Q.ctl + WCTL_FTAIL, nFin);
            if (want) base = atomicAdd(Q.ctl + WCTL_HEAD, want);
            if (open && Q.switchBelow > 0 && (waitMask != 0u || want != 0)) ca = ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_CLOSEAT);
        }
        if (nFin) {
            fbase = __shfl_sync(0xffffffffu, fbase, 0);
            if (fin) {
                const int pos = fbase + __popc(finMask & ltMask);
                if (pos < Q.cap) {
                    const float tag = __uint_as_float(Q.seq);
                    st128(Q.fin + 2 * (size_t)pos, make_float4(i2f(tk), i2f(state), T.t, tag));
                    st128(Q.fin + 2 * (size_t)pos + 1, make_float4(i2f(T.hitTri), K.t2, tag, tag));
                }
                WAVE_LAT_NOW(tk, 3);
                st = WS_NONE;
                tk = -1;
            }
        }
        if (want) {
            base = __shfl_sync(0xffffffffu, base, 0);
            if (st == WS_NONE) {
                tk = base + __popc(noneMask & ltMask);
                st = WS_WAIT;
            }
        }
        if (open && Q.switchBelow > 0) {
            ca = __shfl_sync(0xffffffffu, ca, 0);
            if (ca != 0u) closeAt = (int)(ca - 1u);
        }
        const bool closed = closeAt != 0x7fffffff;
        if (closed && want != 0 && base + want > closeAt) drained = true;
        if (st == WS_WAIT && tk >= closeAt) { st = WS_NONE; tk = -1; } // a ticket of the closed part: it will never be served
        // ---- 1b. after the change-over the rays this warp is still searching are handed over to the GROUP form with their
        // search state (best candidate, runner-up, traversal stack): a LANE warp with a few long rays left costs the issue slots
        // of a full one. The ray gets a new record in the second part of the queue that points at the saved state.
        const bool handOver = closed && Q.resume != nullptr;
        if (handOver) {
            const bool mig = st == WS_RUN && state == TRAV_CONTINUE && T.sp <= WAVE_RESUME_STACK;
            const unsigned migMask = __ballot_sync(0xffffffffu, mig);
            if (migMask != 0u) {
                int rbase = 0, qbase = 0;
                if (lane == 0) {
                    rbase = atomicAdd(Q.ctl + WCTL_RESUME, __popc(migMask));
                    qbase = atomicAdd(Q.ctl + WCTL_TAIL2, __popc(migMask));
                }
                rbase = __shfl_sync(0xffffffffu, rbase, 0);
                qbase = __shfl_sync(0xffffffffu, qbase, 0);
                if (mig) {
                    const int r = rbase + __popc(migMask & ltMask), ntk = closeAt + qbase + __popc(migMask & ltMask);
                    const bool room = r < Q.resumeCap; // (always: a lane hands over at most once; without room the ray starts over)
                    float4* dst = Q.resume + (size_t)WAVE_RESUME_F4 * (room ? r : 0);
                    if (room) st128(dst, make_float4(T.t, i2f(T.hitTri), K.t2, __uint_as_float(T.node)));
                    for (int i = 0; room && i < T.sp; i += 2)
                        st128(dst + 1 + (i >> 1), make_float4(__uint_as_float(K.e[i].x), __uint_as_float(K.e[i].y),
                                                              i + 1 < T.sp ? __uint_as_float(K.e[i + 1].x) : 0.0f,
                                                              i + 1 < T.sp ? __uint_as_float(K.e[i + 1].y) : 0.0f));
                    waveRelease(Q); // the state is in L2 before the record that points at it can be seen
                    if (ntk < Q.cap) {
                        const float4* src = Q.rays + 3 * (size_t)tk;
                        const float4 a = ld128(src), b = ld128(src + 1), m = ld128(src + 2);
                        const float tag = __uint_as_float(Q.seq | WAVE_TAG2);
                        float4* q = Q.rays + 3 * (size_t)ntk;
                        st128(q, make_float4(a.x, a.y, a.z, tag));
                        st128(q + 1, make_float4(b.x, b.y, b.z, tag));
                        st128(q + 2, make_float4(m.x, m.y, i2f(room ? ((r + 1) | (T.sp << 24)) : 0), tag));
                        WAVE_LAT_NOW(ntk, 0);
                    }
                    st = WS_NONE;
                    tk = -1;
                    state = TRAV_DONE;
                }
            }
        }
        // ---- 2. lanes holding a ticket read their record (complete = the ray exists); a warp with nothing running looks cheaply first
        const bool look = runMask != 0u || wavePeekRay(Q, st == WS_WAIT, tk, Q.seq);
        if (look && st == WS_WAIT) {
            float4 a, b, c;
            if (waveLoadRay(Q, tk, Q.seq, a, b, c)) {
                maxDist = b.w;
                eps = c.z;
                any = (f2i(c.y) & CGRT_RAY_ANY) != 0;
                K.t2 = __int_as_float(0x7f800000);
                if (handOver) { // a ray of the first part that arrives after the change-over: passed on to the second part as it is
                    T.o = mk3(a);
                    T.d = mk3(b);
                    T.t = any ? b.w : a.w;                                              // the record's bound
                    T.node = (uint32_t)(any ? f2i(c.y) : ((f2i(c.y) << WAVE_SLOT_BITS) | f2i(c.x))); // the record's meta word
                    st = WS_PASS;
                } else {
                    state = fastBegin(S, T, mk3(a), mk3(b), a.w); // (the always-list is applied by the finish warps)
                    st = WS_RUN;
                    WAVE_LAT_NOW(tk, 1);
                    WAVE_LAT(tk, 6, 1u);
                }
            }
        }
        if (handOver) {
            const unsigned passMask = __ballot_sync(0xffffffffu, st == WS_PASS);
            if (passMask != 0u) {
                int qbase = 0;
                if (lane == 0) qbase = atomicAdd(Q.ctl + WCTL_TAIL2, __popc(passMask));
                qbase = __shfl_sync(0xffffffffu, qbase, 0);
                if (st == WS_PASS) {
                    waveStoreRay(Q, closeAt + qbase + __popc(passMask & ltMask), Q.seq | WAVE_TAG2, T.o, T.d, T.t, (int)T.node);
                    st = WS_NONE;
                    tk = -1;
                    state = TRAV_DONE;
                }
            }
        }
        if (__ballot_sync(0xffffffffu, st == WS_RUN) == 0u) {
            if (drained && __ballot_sync(0xffffffffu, st == WS_WAIT) == 0u) return false; // nothing held, nothing left: change form
            if (waveDone(Q)) return true;
            waveIdle(Q, t0, idlePolls);
            continue;
        }
        idlePolls = 0;
        // ---- 3. a burst of search steps; each step runs the node class the warp votes for. The burst ends early when enough
        // lanes have finished for a refill
#pragma unroll 1
        for (int it = 0; it < CGRT_WAVE_STEPS; it++) {
            const bool run = st == WS_RUN && state == TRAV_CONTINUE;
            const bool leaf = run && travIsLeaf(T.node);
            const int sAll = __popc(__ballot_sync(0xffffffffu, run));
            const int sLeaf = __popc(__ballot_sync(0xffffffffu, leaf));
            const int nDone = __popc(__ballot_sync(0xffffffffu, st == WS_RUN && state != TRAV_CONTINUE));
            if (sAll == 0 || (nDone >= CGRT_WAVE_REFILL && it > 0)) break;
            if (sAll - sLeaf >= sLeaf) {
                if (run && !leaf) state = fastStepWideDyn(S, T, K, any, maxDist);
            } else {
                if (leaf) state = fastStepLeafDyn(S, T, K, any, eps, maxDist);
            }
        }
    }
}

// ---- SEARCH warps, GROUP form: eight lanes per ray (the step of k_trace8 on tickets) ---------------------------------------
// (headIdx, baseIdx, tagBits): the part of the ray array this loop consumes - the whole queue in GROUP-only frames, the second
// part after a change-over
RT_DEV void waveGroupLoop(const DevScene& S, const WaveQ& Q, WaveShared& sh, unsigned long long t0, int headIdx, int baseIdx,
                          unsigned tagBits)
{
    const int lane = threadIdx.x & 31, g = lane >> 3, j = lane & 7;
    uint2* K = sh.gstack[threadIdx.x >> 3];
    const float slack = 1.000001f;
    // group-uniform ray state (every lane of the group holds the same values)
    V3 o = mk3(0.0f, 0.0f, 0.0f), d = o, inv = o;
    float t = 0.0f, t2 = 0.0f, eps = 0.0f, maxDist = 0.0f;
    int hitTri = -1, tk = -1, st = WS_NONE, state = TRAV_DONE, sp = 0;
    uint32_t node = 0u;
    bool any = false;
    int idlePolls = 0;
#ifdef CGRT_WAVE_LAT
    int nsteps = 0;
#endif
    while (true) {
        // ---- 1. finished groups hand in their result
        const bool fin = st == WS_RUN && state != TRAV_CONTINUE;
        if (__any_sync(0xffffffffu, fin)) {
            waveFinPush(Q, fin && j == 0, tk, state, t, hitTri, t2);
#ifdef CGRT_WAVE_LAT
            if (fin && j == 0) { WAVE_LAT_NOW(tk, 3); WAVE_LAT(tk, 2, (unsigned)nsteps); }
#endif
            if (fin) { st = WS_NONE; tk = -1; }
        }
        // ---- 2. every empty group takes a ticket, also one of a ray that does not exist yet
        const unsigned needy = __ballot_sync(0xffffffffu, st == WS_NONE && j == 0);
        if (needy != 0u) {
            const int base = waveClaim(Q, headIdx, __popc(needy));
            if (st == WS_NONE) {
                tk = baseIdx + base + __popc(needy & ((1u << (8 * g)) - 1u));
                st = WS_WAIT;
            }
        }
        // ---- 3. groups holding a ticket read their record (every lane of the group reads it - broadcast loads - and the group
        // starts when all eight have seen it complete). A poll costs the whole warp a round trip to L2: while other groups are
        // searching it happens once per burst of steps; a warp with nothing running looks cheaply first
        const bool anyRun = __ballot_sync(0xffffffffu, st == WS_RUN) != 0u;
        if (anyRun ? __any_sync(0xffffffffu, st == WS_WAIT) : wavePeekRay(Q, st == WS_WAIT, tk, tagBits)) {
            float4 a = make_float4(0.0f, 0.0f, 0.0f, 0.0f), b = a, c = a;
            const bool rdy = st == WS_WAIT && waveLoadRay(Q, tk, tagBits, a, b, c);
            const unsigned rm = __ballot_sync(0xffffffffu, rdy);
            const bool start = ((rm >> (8 * g)) & 0xFFu) == 0xFFu;
            if (start) {
                o = mk3(a);
                d = mk3(b);
                maxDist = b.w;
                eps = c.z;
                any = (f2i(c.y) & CGRT_RAY_ANY) != 0;
                FastTrav T0; // (every lane of the group evaluates the same start; the always-list is applied by the finish warps)
                state = fastBegin(S, T0, o, d, a.w);
                inv = T0.inv;
                t = T0.t;
                t2 = __int_as_float(0x7f800000);
                hitTri = T0.hitTri;
                sp = 0;
                node = T0.node;
                st = WS_RUN;
                const int rs = f2i(c.w);
#ifdef CGRT_WAVE_LAT
                nsteps = 0;
                if (j == 0) { WAVE_LAT_NOW(tk, 1); WAVE_LAT(tk, 6, rs != 0 ? 6u : 2u); }
#endif
                if (rs != 0) { // a search handed over by a LANE warp: continue from its state (it had passed fastBegin)
                    const float4* src = Q.resume + (size_t)WAVE_RESUME_F4 * ((rs & 0xffffff) - 1);
                    const float4 h = ld128(src);
                    t = h.x;
                    hitTri = f2i(h.y);
                    t2 = h.z;
                    node = __float_as_uint(h.w);
                    sp = rs >> 24;
                    state = TRAV_CONTINUE;
                    for (int i = 2 * j; i < sp; i += 16) {
                        const float4 e = ld128(src + 1 + (i >> 1));
                        K[i] = make_uint2(__float_as_uint(e.x), __float_as_uint(e.y));
                        if (i + 1 < sp) K[i + 1] = make_uint2(__float_as_uint(e.z), __float_as_uint(e.w));
                    }
                }
            }
            __syncwarp();
        }
        if (__ballot_sync(0xffffffffu, st == WS_RUN && state == TRAV_CONTINUE) == 0u) {
            if (__ballot_sync(0xffffffffu, st == WS_RUN) == 0u) {
                if (waveDone(Q)) return;
                waveIdle(Q, t0, idlePolls);
            }
            continue;
        }
        idlePolls = 0;
        // ---- 4. a burst of steps: the bookkeeping above (results, tickets, polls) costs as much as a step, so it runs once per
        // burst; the burst ends as soon as a group has finished its search (its result should not wait)
#pragma unroll 1
        for (int it = 0; it < CGRT_WAVE_GSTEPS; it++) {
            // one step of every active group. The per-lane tests run in divergent code WITHOUT collectives; the group results
            // are then combined with full-warp ballots / shuffles that all 32 lanes execute together.
            const bool active = st == WS_RUN && state == TRAV_CONTINUE;
            const bool isLeaf = (node & CGRT_TRI) != 0u;
#ifdef CGRT_WAVE_LAT
            if (active) nsteps++;
#endif
            const float bound = (any ? fminf(t, maxDist) : t) * slack;
            int pos = -1;                            // leaf: position of this lane's triangle
            float near = __int_as_float(0x7f800000); // leaf: distance of an acceptable triangle that does not beat the best
            bool p = false, amb = false;     // p: this lane's child box is hit / this lane's triangle is an acceptable candidate
            unsigned key = 0xffffffffu;      // ordering key of the lane's result (entry distance | child, or candidate distance)
            uint32_t id = 0u;
            float ti = 0.0f;
            if (active) {
                if (isLeaf) {
                    // leaf: lane j tests triangle j with the reference's accept arithmetic (cgrt_device.cuh fastStepLeafDyn)
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
            {
                const unsigned runG = __ballot_sync(0xffffffffu, st == WS_RUN && j == 0);
                const unsigned actG = __ballot_sync(0xffffffffu, st == WS_RUN && state == TRAV_CONTINUE && j == 0);
                if (actG == 0u || __popc(runG ^ actG) >= CGRT_WAVE_GFIN) break;
            }
        }
    }
}


// ---- the kernel -----------------------------------------------------------------------------------------------------------------
#ifndef CGRT_WAVE_MINBLOCKS
#define CGRT_WAVE_MINBLOCKS 8
#endif
// (the frame's parameters travel as a kernel argument: the kernel then depends on nothing but its own launch)
__global__ void __launch_bounds__(128, CGRT_WAVE_MINBLOCKS) k_wave(DevScene S, const FrameParams Pv,
                                                                  const float4* __restrict__ lights, WaveQ Q, RoundBuffers B,
                                                                  const int2* __restrict__ tileSeq, float* __restrict__ fb)
{
    __shared__ WaveShared sh;
    __shared__ FrameParams Psh;
    __shared__ int genCount;
    if (threadIdx.x == 0) {
        Psh = Pv;
        genCount = 0;
    }
    if (threadIdx.x < WAVE_NSTAT) sh.stat[threadIdx.x] = 0;
    __syncthreads();
    const FrameParams& P = Psh;
    const int lane = threadIdx.x & 31;
    const unsigned long long t0 = globalTimerNs();
    if (threadIdx.x == 0 && Q.trace != nullptr) atomicCAS((unsigned*)Q.ctl + WCTL_T0, 0u, (unsigned)t0 | 1u);

    // ---- phase A: primary rays (level 0). Rays that cannot enter the tree are black (trace(): miss, main.cpp:288-294)
    {
        int mine = 0;
        const int n = P.nSlots;
        for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
            const int slot = base + threadIdx.x;
            bool push = false;
            V3 o = mk3(0.0f, 0.0f, 0.0f), d = mk3(0.0f, 0.0f, 0.0f);
            if (slot < n) {
                int x, y, outIdx, local, v;
                B.pathDepth[slot] = 0;
                if (seqToPixel(P, tileSeq, slot, x, y, outIdx, local, v)) {
                    const ViewCamera C = viewCamera(P, lights, v);
                    o = C.o;
                    d = primaryDirection(P, C, x, y);
                    bool enter = S.nSpheres > 0; // a ray that does not enter the tree (bvh.cpp:831-844) can only hit spheres
                    if (!enter && S.nNodes > 0) {
                        const float4 q0 = __ldg(S.nodes + 0), q1 = __ldg(S.nodes + 1);
                        enter = startsInBox(o, mk3(q0), mk3(q1));
                        if (!enter) {
                            float tmp;
                            enter = slabTest(mk3(q0), mk3(q1), o, d, FLT_MAX, tmp);
                        }
                    }
                    push = enter;
                    if (!enter) storeRGB(fb, outIdx, mk3(0.0f, 0.0f, 0.0f));
                } else if (!P.screenLayout) {
                    storeRGB(fb, local, mk3(0.0f, 0.0f, 0.0f)); // padding pixels of edge tiles in the tile-major buffer
                }
            }
            const unsigned pm = __ballot_sync(0xffffffffu, push);
            if (pm != 0u) {
                int tbase = 0;
                if (lane == 0) tbase = atomicAdd(Q.ctl + WCTL_TAIL, __popc(pm));
                tbase = __shfl_sync(0xffffffffu, tbase, 0);
                if (push) {
                    waveStoreRay(Q, tbase + __popc(pm & ((1u << lane) - 1u)), Q.seq, o, d, FLT_MAX, slot); // level 0
                    mine++;
                }
            }
        }
        // the CTA's rays and its "phase A done" bit enter the counter together (rays may be finished by other CTAs before that:
        // the sum is exact whenever every CTA has reported, which is the only state the completion test accepts)
        if (mine) atomicAdd(&genCount, mine);
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) wavePending(Q, (long long)genCount + ((long long)1 << 32));
    }

    // ---- phase B: one role per SM (see the header): finish warps on every Q.finEvery-th SM, search warps on the others
    if (smId() % (unsigned)Q.finEvery == 0u) {
        if ((threadIdx.x & 31) == 0) atomicAdd(Q.ctl + WCTL_FINCOUNT, 1);
        waveFinishLoop(S, P, lights, Q, B, tileSeq, fb, sh, t0);
    } else if (Q.mode == 2) {
        waveGroupLoop(S, Q, sh, t0, WCTL_HEAD, 0, Q.seq);
    } else if (!waveLaneLoop(S, Q, t0)) {
        const int closeAt = (int)ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_CLOSEAT) - 1; // (non-zero: the LANE loop has seen it)
        waveGroupLoop(S, Q, sh, t0, WCTL_HEAD2, closeAt, Q.seq | WAVE_TAG2);
    }

    // Finish warps register before they process anything and release their writes when they leave their loop; phase C waits
    // until every registered finish warp has left (one thread per CTA looks, on a line of its own)
    if (threadIdx.x == 0) {
        int polls = 0;
        while (ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_FINCOUNT) != ldRelaxedGpu((const unsigned*)Q.ctl + WCTL_FINEXIT)) {
            __nanosleep(200);
            if ((++polls & 1023) == 0 && globalTimerNs() - t0 > Q.timeoutNs) {
                atomicExch(Q.ctl + WCTL_ERR, 1);
                break;
            }
        }
    }
    __syncthreads();
    // ---- phase C: shading(), shade() per pixel slot (the hit records / lit flags of other CTAs were released before the done
    // flag was raised; they are read through L2)
    {
        const int nL = P.nLights;
        for (int base = blockIdx.x * blockDim.x; base < P.nSlots; base += gridDim.x * blockDim.x) {
            const int slot = base + threadIdx.x;
            const int depth = slot < P.nSlots ? __ldcg(B.pathDepth + slot) : 0;
            bool wrote = false;
            int x = 0, y = 0;
            if (depth > 0) { // (else the pixel is already final: black)
                V3 direct[CGRT_MAX_LEVELS], ksv[CGRT_MAX_LEVELS];
                for (int k = 0; k < depth; k++) {
                    const int rec = slot * B.levels + k;
                    const float4* r = B.hitRec + 3 * (size_t)rec;
                    direct[k] = directColour<true>(S, lights, nL, __ldcg(r), __ldcg(r + 1), __ldcg(r + 2), B.lit + (size_t)rec * nL, ksv[k]);
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
    // ---- statistics of the frame (cgrt_render_stats)
    __syncthreads();
    if (threadIdx.x < WAVE_NSTAT) {
        const int v = sh.stat[threadIdx.x];
        if (v) {
            const int i = threadIdx.x;
            int* dst = nullptr;
            if (i == WAVE_STAT_PATHS) dst = B.counts + CGRT_CNT_PATHS;
            else if (i >= WAVE_STAT_HIT && i < WAVE_STAT_HIT + CGRT_MAX_LEVELS) dst = B.counts + CGRT_CNT_HIT + (i - WAVE_STAT_HIT);
            else if (i >= WAVE_STAT_BOUNCE && i <= WAVE_STAT_BOUNCE + CGRT_MAX_LEVELS) dst = B.counts + CGRT_CNT_BOUNCE + (i - WAVE_STAT_BOUNCE);
            else if (i == WAVE_STAT_REPLAYC) dst = B.counts + CGRT_CNT_REPLAY_PATHS;
            else if (i == WAVE_STAT_REPLAYS) dst = B.counts + CGRT_CNT_REPLAY_SHADOW;
            if (dst) atomicAdd(dst, v);
        }
    }
}
