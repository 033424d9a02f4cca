// mrs_step_group_body.cuh -- the body of the group kernels (N <= 32).
// Compiled into the kernel without the external wrench (EXT = false) and into its overload with it (EXT = true):
// the same text, so the kernel without is what it was before the wrench existed (the body as a shared
// __forceinline__ function lost the __launch_bounds__ range facts ptxas schedules by, and changed its SASS).
// Included only inside those kernel definitions in mrs_step.cuh; no include guard.
    MrsConfig c_bk;
    Derived d_bk;
    if constexpr (BAKED) baked_fill(c_bk, d_bk, c_in, d_in);
    const MrsConfig& c = BAKED ? c_bk : c_in;
    const Derived& d = BAKED ? d_bk : d_in;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr bool kFull = GT != 0;
    constexpr bool kStage = MRS_PREFETCH && kFull;
    // shared memory, one contiguous region per warp so that every address is one per-warp base plus an
    // immediate: [32 positions] (the pair tile, 512 B) [prefetch stage]
    constexpr int kWarpBytes = group_warp_smem_bytes<MODE, GT>();
    __shared__ int sh_counter, sh_hi, sh_range, sh_lo, sh_pull;
    __shared__ unsigned sh_epoch;
    __shared__ unsigned sh_events[7];       // CTA-level status word + the six statistics counters
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    unsigned char* wbase = smem_raw + wib * kWarpBytes;
    float4* wpos = reinterpret_cast<float4*>(wbase);
#ifdef MRS_EXP_OLDSMEM
    float* stage = reinterpret_cast<float*>(wbase + 1024);
#else
    float* stage = reinterpret_cast<float*>(wbase + 512);
#endif
    const int G = GT ? GT : a.G;
    const int N = GT ? GT : c.N;
    const int E = c.E;
    const int gpw = 32 / G;
    const int ai = lane & (G - 1);
    const int gb = lane - ai;
    const unsigned S = (unsigned)E * (unsigned)N;
    const int wtotal = gridDim.x * WPB;
    const MrsPhysicsParams& ph = c.phys;
    const bool pair_contact = ph.agent_contact && N > 1;

    // Work distribution (see the comment above the kernel) over the chunks [a.chunk_lo, a.nchunks).
    // kLocal: the CTA owns the contiguous share [cta_lo, cta_hi) and its warps draw chunk indices from
    // a shared-memory counter; a warp always knows its next chunk (the stage prefetch needs it) and
    // draws the one after next at the top of an iteration, so the atomic's latency is never waited for.
    constexpr bool kLocal = WPB > 4;
    constexpr bool kHand = kLocal && MRS_PREFETCH && GT != 0 && !MANY;
    const int T = MANY ? a.T : 1;
    const int gw = blockIdx.x * WPB + wib;
    if (threadIdx.x < 7) sh_events[threadIdx.x] = 0u;
    if (threadIdx.x == 7) sh_pull = 0;
    const int role = kHand ? a.role : 0;
    if (role == 2) {
        asm volatile("griddepcontrol.launch_dependents;");
        if (threadIdx.x == 0) {
            // my range: entry blockIdx of the previous launch.  And a bound on the launches in flight: a CTA that
            // takes the contact path can run many times longer than a step, and the launches behind it would
            // pile up (each with one CTA spinning for the straggler's range) until they lap the eight queues --
            // so a launch also waits until the launch three positions back has published ALL its ranges (its
            // last entry exists).  Then at most the queues of positions t-2 .. t+1 are live.
            const unsigned long long* q = b.sync + kSyncQueue + ((a.seq - 1) & (kSyncQueues - 1)) * kSyncQueueLen + blockIdx.x;
            const unsigned long long* q3 = b.sync + kSyncQueue + ((a.seq - 3) & (kSyncQueues - 1)) * kSyncQueueLen + (gridDim.x - 1);
#ifdef MRS_EXP_NOBOUND
            const bool bound = false;
#else
            const bool bound = a.seq >= 3;
#endif
            unsigned long long e = ld_acquire_gpu_u64(q), e3 = bound ? ld_acquire_gpu_u64(q3) : 0ull, t0 = 0;
            unsigned epoch = (unsigned)ld_acquire_gpu_u64(b.sync);
            auto pending = [&]() {
                const unsigned long long tag = (unsigned long long)epoch << 16;
                return (e >> 16) != (tag | (unsigned)a.seq) || (bound && (e3 >> 16) != (tag | (unsigned)(a.seq - 2)));
            };
            while (pending()) {
                if (t0 == 0) t0 = global_ns();
                else if (global_ns() - t0 > 2000000000ull) {       // 2 s: the chain is broken -- fall back, flag it
                    if (b.status) atomicOr(b.status, MRS_STATUS_SYNC_TIMEOUT);
                    asm volatile("griddepcontrol.wait;" ::: "memory");
                    e = blockIdx.x;
                    break;
                }
                e = ld_acquire_gpu_u64(q);
                if (bound) e3 = ld_acquire_gpu_u64(q3);
                epoch = (unsigned)ld_acquire_gpu_u64(b.sync);
            }
            // the queue four positions ahead was last used four positions back: that launch is complete now
            if (blockIdx.x == 0) atomicExch(b.sync + kSyncCount + ((a.seq + 4) & (kSyncQueues - 1)), 0ull);
            sh_range = (int)(e & 0xffffull);
            sh_epoch = epoch;               // (shared memory: the tag of this CTA's own entry, needed at the very end)
        }
    } else {
        if (role == 0) asm volatile("griddepcontrol.launch_dependents;");
        asm volatile("griddepcontrol.wait;" ::: "memory");
        if (threadIdx.x == 0) sh_range = blockIdx.x;
        if (role == 1) {
            // everything before this launch is complete: start a new chain, then let the first link in
            if (blockIdx.x == 0 && threadIdx.x == 0) {
#pragma unroll
                for (int q = 0; q < kSyncQueues; ++q) atomicExch(b.sync + kSyncCount + q, 0ull);
                atomicAdd(b.sync, 1ull);
                __threadfence();
            }
            __syncthreads();
            asm volatile("griddepcontrol.launch_dependents;");
        }
    }
    if (threadIdx.x == 0) {
        const int nwork = a.nchunks - a.chunk_lo;
        const int r = sh_range;
        sh_counter = sh_lo = a.chunk_lo + (int)(((long long)r * nwork) / gridDim.x);
        sh_hi = a.chunk_lo + (int)(((long long)(r + 1) * nwork) / gridDim.x);
    }
    // chunks parked for the contact path: first step they need it and the warp that parked them (all ones = not
    // parked), one slot per chunk of this CTA (SM-filling shape: index = chunk - first chunk of the CTA's range;
    // small shape: warp * rounds + round).  A warp processes what it parked itself: no CTA barrier in between.
    unsigned* parked = reinterpret_cast<unsigned*>(smem_raw + WPB * kWarpBytes);      // step | parking warp << 16
    for (int i = threadIdx.x; i < a.slow_slots; i += WPB * 32) parked[i] = 0xffffffffu;
    __syncthreads();
    // one elected lane draws a chunk index (-1 when the share is used up); the others get it by shuffle later.
    // elect.sync keeps ptxas from wrapping the single-lane atomic in its warp-aggregation sequence (vote, popc,
    // ltmask, shuffle + a divergent block: 17 instructions; this form is 6).
    auto draw = [&]() -> int {
        int v = 0;
        asm volatile("{\n .reg .pred p;\n elect.sync _|p, 0xffffffff;\n @p atom.shared.add.u32 %0, [%1], 1;\n}"
                     : "+r"(v) : "r"((unsigned)__cvta_generic_to_shared(&sh_counter)) : "memory");
        return v;           // valid in lane 0 (the elected lane of a full warp)
    };
    const int chunk_hi = sh_hi;
    auto claim = [&](int v) -> int { return (v < chunk_hi) ? v : -1; };
    // chunk = 32 consecutive agent slots (kFull).  The stage is filled in 16-byte pieces, piece q at float
    // offset 4 q, lane l moves pieces l, l + 32, ...:  [0, 96) state planes 0-11 (plane q >> 3, sub-piece
    // q & 7: a lane's plane advances by 4 per round, so its element index is lane part + round part +
    // chunk part), then the chunk's actions (32 * ACTION_DIM contiguous floats: one whole round for
    // ACTION_DIM 4), then plane 12, then 8 pieces per PID plane.
    constexpr int kNC = mode_nctrl<MODE>();
    constexpr int kA = ModeTraits<MODE>::A;
    constexpr int kActBeg = 96, kActEnd = kActBeg + 8 * kA;       // piece ranges
    constexpr int kP12Beg = kActEnd, kP12End = kP12Beg + 8;
    constexpr int kCtlBeg = kP12End, kCtlEnd = kCtlBeg + 8 * kNC;
    constexpr int kPieces = kCtlEnd;
    static_assert(kPieces * 4 == mode_stage_floats<MODE>(), "stage layout");
    const unsigned lane_el = (unsigned)(lane >> 3) * S + (unsigned)(lane & 7) * 4u;   // plane (l>>3), sub-piece (l&7)
    auto prefetch = [&](int chunk) {
        const unsigned s0 = (unsigned)chunk * 32u;
#pragma unroll
        for (int i = 0; i < (kPieces + 31) / 32; ++i) {
            const int q = lane + 32 * i;
            const int lo = 32 * i, hi = 32 * i + 31;       // compile-time after unrolling: the tests below fold
            if (hi < kActBeg) {
                cp_async16(stage + 4 * q, b.state + (lane_el + s0 + (unsigned)(4 * i) * S));
            } else {
                if (lo < kActEnd && hi >= kActBeg && (lo >= kActBeg || q >= kActBeg) && (hi < kActEnd || q < kActEnd))
                    cp_async16(stage + 4 * q, a.actions + (s0 * (unsigned)kA + (unsigned)(q - kActBeg) * 4u));
                if (lo < kP12End && hi >= kP12Beg && (lo >= kP12Beg || q >= kP12Beg) && (hi < kP12End || q < kP12End))
                    cp_async16(stage + 4 * q, b.state + (12u * S + s0 + (unsigned)(q - kP12Beg) * 4u));
                if (kNC > 0 && lo < kCtlEnd && hi >= kCtlBeg && (lo >= kCtlBeg || q >= kCtlBeg) && (hi < kCtlEnd || q < kCtlEnd)) {
                    const int cq = q - kCtlBeg;
                    cp_async16(stage + 4 * q, b.ctrl + ((unsigned)mode_ctrl_plane<MODE>(cq >> 3) * S + s0 + (unsigned)(cq & 7) * 4u));
                }
            }
        }
        cp_async_commit();
    };
#ifdef MRS_TRACE
    // debug build (tools/trace_c5.py): per-warp timeline (globaltimer ns) into bufs.scratch seen as
    // u64[warps][8], plus per-step aggregates [min start, max wait release, max end, min end]
    unsigned long long* trace = reinterpret_cast<unsigned long long*>(b.scratch) + (size_t)gw * 8;
    unsigned long long* agg = reinterpret_cast<unsigned long long*>(b.scratch) + (size_t)8192 * 8 + (size_t)a.slot_x * 4;
    int trace_i = 0;
    auto stamp = [&]() {
        unsigned long long tns;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tns));
        if (lane == 0 && trace_i < 8) trace[trace_i] = tns;
        // aggregates: one atomic per CTA (per-warp atomics on one address -- 8 k per launch -- stretched the
        // kernel boundary by ~6 us and showed up as a gap that the production build does not have)
        if (threadIdx.x == 0 && trace_i == 0) atomicMin(agg + 0, tns);
        if (threadIdx.x == 0 && trace_i == 1) atomicMax(agg + 1, tns);
        ++trace_i;
    };
    auto stamp_end = [&]() {            // called after the CTA's final barrier: the CTA's end
        unsigned long long tns;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tns));
        if (threadIdx.x == 0) { atomicMax(agg + 2, tns); atomicMin(agg + 3, tns); }
    };
    stamp();
#endif
#ifdef MRS_TRACE
    stamp();
#endif
    int chunk, chunk_next;
    if (kLocal) {
        chunk = claim(__shfl_sync(kFull32, draw(), 0));
        chunk_next = chunk >= 0 ? claim(__shfl_sync(kFull32, draw(), 0)) : -1;
    } else {
        chunk = a.chunk_lo + gw;
        chunk_next = chunk + wtotal;
        if (chunk >= a.nchunks) chunk = -1;
        if (chunk_next >= a.nchunks) chunk_next = -1;
    }
    if (kStage && chunk >= 0) prefetch(chunk);
    // A chunk that needs the contact path is PARKED (its slot in `parked` gets the step) and processed after this
    // loop: the hot loop keeps its shape -- one vote, and a branch around the stores -- whatever the contact path
    // costs (inside the loop it cost ~90 extra instructions per chunk: its loop-invariant set-up was hoisted here).
    const int rounds_static = kLocal ? 0 : (a.nchunks - a.chunk_lo + wtotal - 1) / wtotal;
    int round_i = 0, my_parked = 0;
    while (chunk >= 0) {
        const int ticket = (kLocal && chunk_next >= 0) ? draw() : -1;   // the chunk after next; warp-uniform condition
        // kFull: the chunk is 32 consecutive valid slots; else lanes >= N of a group (and envs >= E) idle
        const int e = chunk * gpw + (lane / G);
        const bool valid = kFull ? true : ((e < E) && (ai < N));
        const unsigned s = kFull ? (unsigned)chunk * 32u + (unsigned)lane
                                 : (valid ? (unsigned)e * (unsigned)N + (unsigned)ai : 0u);
        Agent st;
        Ctrl k;
        float4 act0 = make_float4(0.f, 0.f, 0.f, 0.f);
        ExtWrench xw{};
        if constexpr (EXT) {
            if (valid) xw = load_wrench(b.wrench, S, s);
        }
        if constexpr (kStage) {
            cp_async_wait_all();
            __syncwarp();           // pieces were fetched by other lanes
            st.px = stage[0 * 32 + lane]; st.py = stage[1 * 32 + lane]; st.pz = stage[2 * 32 + lane];
            st.qx = stage[3 * 32 + lane]; st.qy = stage[4 * 32 + lane]; st.qz = stage[5 * 32 + lane];
            st.qw = stage[6 * 32 + lane];
            st.vx = stage[7 * 32 + lane]; st.vy = stage[8 * 32 + lane]; st.vz = stage[9 * 32 + lane];
            st.wx = stage[10 * 32 + lane]; st.wy = stage[11 * 32 + lane]; st.wz = stage[4 * kP12Beg + lane];
            const float* cs = stage + 4 * kCtlBeg + lane;
            if constexpr (ModeTraits<MODE>::io) {
#pragma unroll
                for (int i = 0; i < 3; ++i) k.io[i] = cs[i * 32];
            }
            if constexpr (ModeTraits<MODE>::ip) {
#pragma unroll
                for (int i = 0; i < 3; ++i) k.ip[i] = cs[(3 + i) * 32];
            }
            if constexpr (ModeTraits<MODE>::vel) {
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    k.iv[i] = cs[(3 + i) * 32]; k.lve[i] = cs[(6 + i) * 32];
                    k.dve[i] = cs[(9 + i) * 32]; k.ltv[i] = cs[(12 + i) * 32];
                }
            }
            const float* as = stage + 4 * kActBeg + kA * lane;
            if constexpr (kA == 4) act0 = *reinterpret_cast<const float4*>(as);
            if constexpr (kA == 3) act0 = make_float4(as[0], as[1], as[2], 0.f);
            __syncwarp();           // everyone has read its column before the stage is refilled
            if (chunk_next >= 0) prefetch(chunk_next);
        } else if (valid) {
            load_agent(b.state, S, s, st);
            load_ctrl<MODE>(b.ctrl, S, s, k);
        } else {
            dummy_agent(st);
#pragma unroll
            for (int i = 0; i < 3; ++i) k.io[i] = k.ip[i] = k.iv[i] = k.lve[i] = k.dve[i] = k.ltv[i] = 0.f;
        }
        float* Xs = a.X0;       // tape slots of step t (they move down one slot per step)
        float* As = a.A0;
        // the action of step t + 1 is loaded while step t is computed (mrs_step_many: a load at the top of
        // every step had its whole latency exposed, 20 % of that kernel's stall samples); act0 holds the
        // action of the coming step
        if (!kStage) {
            float tmp[4] = {0.f, 0.f, 0.f, 0.f};
            if (valid) (void)load_action<MODE>(a.actions, (size_t)s, tmp);
            act0 = make_float4(tmp[0], tmp[1], tmp[2], tmp[3]);
        }
        bool state_stored = false;      // the contact path of a single-step launch stores the state itself
        for (int t = 0; t < T; ++t, Xs -= a.xstride, As -= a.astride) {
            // per-step event word: the registers behind it live only as long as the step needs them
            unsigned status = 0;
            unsigned n_agent_rows = 0, n_ground = 0;
            float rpm[4];
            float act[4] = {act0.x, act0.y, act0.z, act0.w};
            if (kA > 0 && valid && (isnan(act0.x) || isnan(act0.y) || isnan(act0.z) || (kA == 4 && isnan(act0.w))))
                status |= MRS_STATUS_NAN_ACTION;
            if (MANY && t + 1 < T && valid) {
                float tmp[4];
                (void)load_action<MODE>(a.actions, (size_t)(t + 1) * S + s, tmp);
                act0 = make_float4(tmp[0], tmp[1], tmp[2], tmp[3]);
            }

#ifdef MRS_EXP_COPYONLY      // experiment (profiles/README.md): memory movement of a step only, no physics
            st.px += act[0] * 1e-12f;
            if (false) {
#else
            {
#endif
            // ---- pair pass 1: downwash + contact proximity on the pre-step positions.  Multi-step launches run it
            // BEFORE the controller (the contact hand-off below must see the PID state of the step's start: it lives
            // in registers only); single-step launches after it, where its shared-memory latency hides behind the
            // controller arithmetic (the contact path re-reads the untouched PID planes from global memory).
            float dw = 0.f;
            bool near = false;
            auto pair_pass1 = [&]() {
            // ---- pair pass 1: downwash + contact proximity on the pre-step positions
            __syncwarp();
            wpos[lane] = make_float4(st.px, st.py, st.pz, 0.f);
            __syncwarp();
#ifndef MRS_PAIR_ONCE
#define MRS_PAIR_ONCE 1
#endif
            if constexpr (MRS_PAIR_ONCE && GT != 0) {
                // Every unordered pair is evaluated ONCE: in round k lane a handles the pair (a, a + k mod N), so
                // rounds 1 .. N/2 - 1 cover each pair exactly once and round N/2 covers its pairs from both ends.
                // The downwash acts on whichever of the two flies lower (dz > 0 seen from below), so one evaluation
                // with |dz| serves both; the partner's share and the squared distance travel by shuffle.
                if (MODE != MRS_NO_ACTION || pair_contact) {
                    float dmin = 3.0e38f;
#pragma unroll
                    for (int k = 1; k <= GT / 2; ++k) {
#ifdef MRS_EXP_P1FENCE
                        asm volatile("" ::: "memory");      // keep the rounds' shared-memory loads apart
#endif
                        const float4 pj = wpos[gb + ((ai + k) & (GT - 1))];
                        const float rx = pj.x - st.px, ry = pj.y - st.py, rz = pj.z - st.pz;
                        const float dxy2 = rx * rx + ry * ry;
                        const float d2 = dxy2 + rz * rz;
                        float f = 0.f;
                        if (MODE != MRS_NO_ACTION) f = downwash_pair(c.quad, d, dxy2, fabsf(rz));   // 0 when dz == 0
                        dw += (rz > 0.f) ? f : 0.f;
                        dmin = fminf(dmin, d2);
                        if (k < GT / 2) {
                            const int src = gb + ((ai - k) & (GT - 1));       // the lane whose round-k partner I am
                            const float got = __shfl_sync(kFull32, (rz < 0.f) ? f : 0.f, src);
                            const float gd2 = __shfl_sync(kFull32, d2, src);
                            if (MODE != MRS_NO_ACTION) dw += got;
                            dmin = fminf(dmin, gd2);
                        }
                    }
                    near = dmin < d.lim2;
                }
            } else
            if (MODE != MRS_NO_ACTION || pair_contact) {
#pragma unroll 8
                for (int r = 1; r < G; ++r) {
                    const int j = ai ^ r;
                    if (GT || j < N) {
                        const float4 pj = wpos[gb + j];
                        const float rx = pj.x - st.px, ry = pj.y - st.py, rz = pj.z - st.pz;
                        const float dxy2 = rx * rx + ry * ry;
                        if (MODE != MRS_NO_ACTION) dw += downwash_pair(c.quad, d, dxy2, rz);
                        near = near || (dxy2 + rz * rz < d.lim2);
                    }
                }
            }
            };
            // ---- contact (rare): a warp with an agent near the ground or near another agent -- or with a NaN action,
            // which makes that agent step without rotor forces -- hands the whole chunk to the contact path
            // (chunk_step_contact) at the top of the next iteration: the step is redone there from the state in
            // global memory with the sequential-impulse solver.  The fast path carries no contact code.
            auto hand_off = [&]() -> bool {
#ifdef MRS_EXP_NODETECT
                return false;
#endif
                if (!__any_sync(kFull32, valid && ((ph.ground_contact && st.pz < d.gnd_skip_z) || (pair_contact && near) ||
                                                   status != 0u)))
                    return false;
                if (MANY && valid) {         // the registers hold the newest state: make it visible to the contact path
                    store_agent(b.state, S, s, st);
                    store_ctrl<MODE>(b.ctrl, S, s, k);
                }
                if (lane == 0) parked[kLocal ? chunk - sh_lo : wib * rounds_static + round_i] = (unsigned)t | ((unsigned)wib << 16);
                ++my_parked;
                state_stored = true;         // steps t .. T-1 of this chunk belong to the contact path
                return true;
            };
            if constexpr (MANY) {
                pair_pass1();
                if (hand_off()) break;
            }
            float R[9];
            quat_to_mat(st, R);
            action_to_rpm<MODE>(c, c_in.quad, d, st, R, act, k, rpm);
            if constexpr (!MANY) {
                pair_pass1();
                (void)hand_off();            // single step: no break -- the stores below are skipped (state_stored)
            }
            if (b.rpm && MODE != MRS_NO_ACTION && valid && !state_stored) {       // optional Quadcopter.speeds mirror
#pragma unroll
                for (int i = 0; i < 4; ++i) *plane_ptr(b.rpm + s, S, i) = rpm[i];
            }
            apply_wrench<MODE != MRS_NO_ACTION, EXT>(c, d, st, R, rpm, dw, xw);
            integrate(c, d, st);
            if (!agent_finite(st)) status |= MRS_STATUS_NONFINITE;

            }
            // ---- observation: newest X slice and newest A slice into their tape slots
            // (X rows staged through shared memory and written as whole 16-byte pieces were measured: neutral
            // at C5, 18.4 vs 18.1 us -- unlike the A rows below, the float2 stores are not the limiter)
            if (!state_stored) {
            if (a.X0 && valid) write_X(Xs, c.state_layout, s, st);
            if (a.A0) {
                float* Arow = As + (size_t)s * N;
                if (d.comm_inf) {
                    // COMM_RANGE = inf: ones - eye (MRS.py:119-121), written with the same lane-pair row sharing
                    // as below (whole-sector STG.128) where the width is a compile-time constant
                    if constexpr (GT != 0) {
                        const int h = lane & 1;
                        float* Arow0 = As + (size_t)(s & ~1u) * GT;
                        const int d0 = (ai & ~1) - 4 * h;
#pragma unroll
                        for (int qq = 0; qq < GT / 8; ++qq) {
                            const int col = 8 * qq + 4 * h;
                            float v0[4], v1[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                v0[u] = (8 * qq + u == d0) ? 0.f : 1.f;
                                v1[u] = (8 * qq + u == d0 + 1) ? 0.f : 1.f;
                            }
                            MRS_TAPE_ST(reinterpret_cast<float4*>(Arow0 + col), make_float4(v0[0], v0[1], v0[2], v0[3]));
                            MRS_TAPE_ST(reinterpret_cast<float4*>(Arow0 + GT + col), make_float4(v1[0], v1[1], v1[2], v1[3]));
                        }
                    } else if (valid) {
                        for (int j = 0; j < N; ++j) Arow[j] = (j == ai) ? 0.f : 1.f;
                    }
                } else {
                    __syncwarp();
                    wpos[lane] = make_float4(st.px, st.py, st.pz, 0.f);
                    __syncwarp();
                    if constexpr (GT != 0) {
                        // Lane pair (2k, 2k+1) shares the two rows 2k, 2k+1 of A: the even lane computes the
                        // even column quads of BOTH rows, the odd lane the odd quads.  One STG.128 of the pair
                        // then covers 32 contiguous bytes, i.e. whole 32-byte sectors (a lane writing its own
                        // row alone sends every sector twice, half filled), and every column position read
                        // from shared memory serves two rows.
                        const int h = lane & 1;
                        const float4 r0 = wpos[lane & ~1], r1 = wpos[lane | 1];
                        float* Arow0 = As + (size_t)(s & ~1u) * GT;
                        const int d0 = (ai & ~1) - 4 * h;          // column of row 0's diagonal relative to quad h
#pragma unroll
                        for (int qq = 0; qq < GT / 8; ++qq) {       // this lane's quads: h, h + 2, ...
                            const int col = 8 * qq + 4 * h;
                            float4 pj[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) pj[u] = wpos[gb + col + u];
                            float v0[4], v1[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const float h0 = adjacency_pair(r0.x, r0.y, r0.z, pj[u].x, pj[u].y, pj[u].z, d.s_max);
                                const float h1 = adjacency_pair(r1.x, r1.y, r1.z, pj[u].x, pj[u].y, pj[u].z, d.s_max);
                                v0[u] = (8 * qq + u == d0) ? 0.f : h0;
                                v1[u] = (8 * qq + u == d0 + 1) ? 0.f : h1;
                            }
                            MRS_TAPE_ST(reinterpret_cast<float4*>(Arow0 + col), make_float4(v0[0], v0[1], v0[2], v0[3]));
                            MRS_TAPE_ST(reinterpret_cast<float4*>(Arow0 + GT + col), make_float4(v1[0], v1[1], v1[2], v1[3]));
                        }
                    } else if (valid) {
                        if ((N & 3) == 0) {
#pragma unroll 2
                            for (int j = 0; j < N; j += 4) {
                                // loads and arithmetic unconditional, the diagonal is a select afterwards: a
                                // conditional around the shared-memory load compiles to one divergent
                                // BSSY/BRA/BSYNC block per element (no overlap between the pairs)
                                float4 pj[4];
#pragma unroll
                                for (int u = 0; u < 4; ++u) pj[u] = wpos[gb + j + u];
                                float v[4];
#pragma unroll
                                for (int u = 0; u < 4; ++u) {
                                    const float hit = adjacency_pair(st.px, st.py, st.pz, pj[u].x, pj[u].y, pj[u].z, d.s_max);
                                    v[u] = (j + u == ai) ? 0.f : hit;
                                }
                                MRS_TAPE_ST(reinterpret_cast<float4*>(Arow + j), make_float4(v[0], v[1], v[2], v[3]));
                            }
                        } else {
                            for (int j = 0; j < N; ++j) {
                                const float4 pj = wpos[gb + j];
                                const float hit = adjacency_pair(st.px, st.py, st.pz, pj.x, pj.y, pj.z, d.s_max);
                                Arow[j] = (j == ai) ? 0.f : hit;
                            }
                        }
                    }
                }
            }
            // status / statistics: warp-reduce, then CTA-level shared-memory counters; the global atomics
            // happen once per CTA at the end.  (A swarm resting on the ground reports a ground contact per
            // agent per step: with one global atomic per warp-chunk that was 10 k same-address L2 atomics
            // per launch at C5 and cost ~15 % of the step.)
            }
            if (!valid || state_stored) { status = 0; n_agent_rows = 0; n_ground = 0; }
            if (__reduce_or_sync(kFull32, status | n_agent_rows | n_ground)) {      // rare in free flight
                const unsigned any_status = __reduce_or_sync(kFull32, status);
                const unsigned sum_rows = __reduce_add_sync(kFull32, n_agent_rows);
                const unsigned sum_gnd = __reduce_add_sync(kFull32, n_ground);
                // per agent (the status of a lane without an agent, or of a handed-off chunk, is 0 here)
                const unsigned sum_bad = __reduce_add_sync(kFull32, (status & MRS_STATUS_NONFINITE) ? 1u : 0u);
                const unsigned sum_nan = __reduce_add_sync(kFull32, (status & MRS_STATUS_NAN_ACTION) ? 1u : 0u);
                if (lane == 0) {
                    if (any_status) atomicOr(&sh_events[0], any_status);
                    if (sum_rows) atomicAdd(&sh_events[1], sum_rows);
                    if (sum_gnd) atomicAdd(&sh_events[2], sum_gnd);
                    if (sum_bad) atomicAdd(&sh_events[3], sum_bad);
                    if (sum_nan) atomicAdd(&sh_events[4], sum_nan);
                }
            }
        }

        if (valid && !state_stored) {
            float* p0 = b.state + s;
            *plane_ptr(p0, S, 0) = st.px; *plane_ptr(p0, S, 1) = st.py; *plane_ptr(p0, S, 2) = st.pz;
            *plane_ptr(p0, S, 3) = st.qx; *plane_ptr(p0, S, 4) = st.qy; *plane_ptr(p0, S, 5) = st.qz;
            *plane_ptr(p0, S, 6) = st.qw;
            *plane_ptr(p0, S, 7) = st.vx; *plane_ptr(p0, S, 8) = st.vy; *plane_ptr(p0, S, 9) = st.vz;
            *plane_ptr(p0, S, 10) = st.wx; *plane_ptr(p0, S, 11) = st.wy; *plane_ptr(p0, S, 12) = st.wz;
            store_ctrl<MODE>(b.ctrl, S, s, k);
        }
#ifdef MRS_TRACE
        stamp();
#endif
        chunk = chunk_next;
        ++round_i;
        if (kLocal) {
            chunk_next = (chunk >= 0) ? claim(__shfl_sync(kFull32, ticket, 0)) : -1;
        } else {
            chunk_next = (chunk >= 0 && chunk + wtotal < a.nchunks) ? chunk + wtotal : -1;
        }
    }
#ifndef MRS_EXP_NOCALL
    // ---- the parked chunks: contact path.  Shared out over the CTA's warps through a counter (a chunk's solve takes
    // anything from one sweep to solver_iters, so the warp that parked a chunk is not the one that has to redo it);
    // in free flight this is one CTA-wide vote.
    if (__syncthreads_or(my_parked)) {
        const int n_slots = kLocal ? sh_hi - sh_lo : WPB * rounds_static;
        for (;;) {
            int i = 0;
            if (lane == 0) i = atomicAdd(&sh_pull, 1);
            i = __shfl_sync(kFull32, i, 0);
            if (i >= n_slots) break;
            const unsigned e = parked[i];
            if (e == 0xffffffffu) continue;
            const int w = (int)(e >> 16);
            const int pc = kLocal ? sh_lo + i : a.chunk_lo + blockIdx.x * WPB + w + (i - w * rounds_static) * wtotal;
            chunk_step_contact<MODE, GT, EXT>(&c_in, &d_in, &b, &a, GT ? GT : a.G, pc, (int)(e & 0xffffu), T, kFull32, wpos, sh_events);
        }
    }
#endif
    __syncthreads();
    if (threadIdx.x == 0) {
        if (sh_events[0] && b.status) atomicOr(b.status, sh_events[0]);
        if (b.stats) {
            if (sh_events[1]) atomicAdd(b.stats + MRS_STAT_AGENT_CONTACTS, (unsigned long long)sh_events[1]);
            if (sh_events[2]) atomicAdd(b.stats + MRS_STAT_GROUND_CONTACTS, (unsigned long long)sh_events[2]);
            if (sh_events[3]) atomicAdd(b.stats + MRS_STAT_NONFINITE, (unsigned long long)sh_events[3]);
            if (sh_events[4]) atomicAdd(b.stats + MRS_STAT_NAN_ACTIONS, (unsigned long long)sh_events[4]);
            if (sh_events[5]) atomicAdd(b.stats + MRS_STAT_CONTACT_CHUNKS, (unsigned long long)sh_events[5]);
            if (sh_events[6]) atomicAdd(b.stats + MRS_STAT_SOLVER_SWEEPS, (unsigned long long)sh_events[6]);
        }
        if (role != 0) {
            // publish the finished range (the CTA barrier above ordered every thread's state stores before this fence)
            __threadfence();
            const unsigned epoch = (role == 1) ? (unsigned)ld_acquire_gpu_u64(b.sync) : sh_epoch;
            const int q = a.seq & (kSyncQueues - 1);
            const unsigned long long j = atomicAdd(b.sync + kSyncCount + q, 1ull);
            st_release_gpu_u64(b.sync + kSyncQueue + q * kSyncQueueLen + (int)(j & (kSyncQueueLen - 1)),
                               ((unsigned long long)epoch << 32) | ((unsigned long long)(a.seq + 1) << 16) | (unsigned)sh_range);
        }
    }
#ifdef MRS_TRACE
    stamp_end();
#endif
