// mrs_step.cuh -- the step kernels of the B200-native mrs-gym step path and their launch logic, templated on
// the action mode (instantiated per mode by mrs_step_mode.cu).
//
// Two execution shapes, chosen per call from N (agents per env):
//
//  * N <= 32  "group" path: one lane per agent, an env is a group of G = pow2ceil(N) lanes of one
//    warp (N=8: 4 envs per warp).  Everything of MRS.step that touches the simulator is ONE kernel:
//    action -> cascaded PID / mixer -> rotor wrench + ground effect + drag + downwash ->
//    Bullet velocity update -> sphere / ground contact -> position + quaternion integration ->
//    newest X slice + newest A slice.  The three intra-env pair passes (downwash on pre-step
//    positions, contact on unconstrained velocities, adjacency on post-step positions) go through a
//    per-warp shared-memory tile read with 128-bit LDS.  With T > 1 (mrs_step_many) the state stays
//    in registers across steps, only actions stream in and X/A stream out.
//
//  * N > 32   "tiled" path: an env spans many CTAs, so the step is three kernels with the pair
//    passes tiled n-body style through shared memory:  pre (forces -> v*, w*; copies pre-step
//    positions to scratch), post (contact, integration, X), adjacency (row tile x column tile,
//    coalesced 128-bit stores; this is a pure streaming store at N=4096).
//
// Reference behaviour: /root/reference/mrsgym/MRS.py:240-277 and callees (see mrs_device.cuh);
// Bullet step restated in oracle/bullet_model.py.  No CPU fallback exists in this library.
#pragma once
#include "mrs_common.cuh"
#include "mrs_contact_env.cuh"

namespace mrs {

// ------------------------------------------------------------------------------ group path
// GT > 0: compile-time group width with N == GT (8, 16, 32: pair loops unrolled) and FULL chunks only:
//         every chunk is 32 consecutive valid agent slots, so the kernel carries no bounds logic at
//         all; a ragged last chunk (E not a multiple of 32/N) is a second, one-chunk launch of the
//         GT == 0 kernel (dispatch_step).
// GT == 0: run-time width a.G >= N (any N <= 32), lanes >= N of a group idle.
// WPB = warps per CTA.  WPB = 4: many small CTAs, chunks handed out grid-stride (small jobs).
// WPB = 4 * minb (one CTA owns a whole SM): the CTA takes a contiguous share of the chunks and its
// warps pull them from a shared-memory counter.  Per-warp timestamps at C5 (tools/trace_c5.py)
// showed that with a static split the warps of one launch finish between 12 and 21 us after the
// start -- the hardware warp scheduler is not fair -- and the kernel lasts as long as its slowest
// warp; the SM-local dynamic hand-out keeps all warps of an SM busy until its share is done
// (first / last warp end 14.7 / 20.2 us).  A device-wide atomic counter was tried first: 12k
// same-address L2 atomics per launch serialise and cost +40 %.
//
// BAKED: the model constants (cf2x.urdf, QuadControl gains, Bullet defaults, DT, GRAVITY and what the
// host derives from them) are compile-time values taken from the generated mrs_baked.cuh instead of
// kernel parameters.  sm_100a has no constant-bank operands on its FP instructions: every parameter a
// chunk uses costs an LDC/LDCU issue slot (~10 % of the generic kernel's instructions), immediates cost
// nothing and fold.  The host picks the baked kernel only when the caller's MrsConfig carries exactly
// those values (config_is_baked: bitwise compare); anything else runs the generic kernel.

// plane `pl` of an SoA buffer given the pointer to the agent's slot in plane 0: one IMAD.WIDE.U32
__device__ __forceinline__ float* plane_ptr(float* p0, unsigned S, int pl) {
    return reinterpret_cast<float*>(reinterpret_cast<char*>(p0) + (unsigned long long)S * (unsigned)(pl * 4));
}
__device__ __forceinline__ const float* plane_ptr(const float* p0, unsigned S, int pl) {
    return reinterpret_cast<const float*>(reinterpret_cast<const char*>(p0) + (unsigned long long)S * (unsigned)(pl * 4));
}

// ------------------------------------------------------------------------------ contact path of the group kernels
// One step of one warp-chunk, global memory to global memory, WITH the contact solver
// (bullet_model.solve_contacts): the group kernels call it for a chunk in which some agent is near the ground or
// near another agent, and carry no contact code themselves.  A real function, called from ONE place after the hot
// chunk loop (the parked-chunk pass): inlined anywhere in the kernel -- even after the loop -- its mere presence
// changed the register allocation and instruction scheduling of the hot loop (+1.3 us per C5 step, measured with
// the path compiled in but never taken), and inside the loop its loop-invariant set-up was hoisted to the top of the
// kernel (~290 instructions and a stack frame per warp).
// Same arithmetic as the fast path for everything but the contact rows.  GT = the compile-time group width of the
// full-chunk kernels (8 / 16 / 32 = N), 0 = run-time width.
// In-warp solve: every lane owns one agent, its ground rows and -- per tournament round -- the pair rows with its
// round partner; the partner's velocity travels by shuffle, both lanes of a pair evaluate the same rows from their
// own side and get equal and opposite changes.
template <int MODE, int GT>
static __device__ __noinline__ void chunk_step_contact(const MrsConfig* cptr, const Derived* dptr, const MrsBuffers* bptr,
                                                       const StepArgs* aptr, int G_in, int chunk, int t0, int T, unsigned lane_mask,
                                                       float4* wpos, unsigned* sh_events) {
    const MrsConfig& c = *cptr;
    const Derived& d = *dptr;
    const MrsBuffers& b = *bptr;
    const StepArgs& a = *aptr;
    const int lane = threadIdx.x & 31;
    const int G = GT ? GT : G_in;                       // full-chunk kernels: group width = N = GT at compile time
    const int N = GT ? GT : c.N, E = c.E;
    const int gpw = 32 / G, ai = lane & (G - 1), gb = lane - ai;
    const unsigned S = (unsigned)E * (unsigned)N;
    const int e = chunk * gpw + (lane / G);
    const bool valid = (e < E) && (ai < N);
    const bool mine = valid && ((lane_mask >> lane) & 1u);     // lanes whose env this call handles (it stores nothing else)
    const unsigned s = valid ? (unsigned)e * (unsigned)N + (unsigned)ai : 0u;
    const MrsPhysicsParams& ph = c.phys;
    const ContactParams cp = make_contact_params(ph, d);
    constexpr int kA = ModeTraits<MODE>::A;
    Agent st;
    Ctrl k;
    if (valid) {
        load_agent_cg(b.state, S, s, st);
        load_ctrl_cg<MODE>(b.ctrl, S, s, k);
    } else {
        dummy_agent(st);
#pragma unroll
        for (int i = 0; i < 3; ++i) k.io[i] = k.ip[i] = k.iv[i] = k.lve[i] = k.dve[i] = k.ltv[i] = 0.f;
    }
    if (lane == 0) atomicAdd(&sh_events[5], (unsigned)(T - t0));       // warp-chunk steps on the contact path
  for (int t = t0; t < T; ++t) {
    unsigned status = 0, n_agent_rows = 0, n_ground = 0, n_sweeps = 0;
    float act[4] = {0.f, 0.f, 0.f, 0.f};
    if (valid && kA > 0 && load_action<MODE>(a.actions, (size_t)t * S + s, act)) status |= MRS_STATUS_NAN_ACTION;
    float R[9], rpm[4];
    quat_to_mat(st, R);
    // NaN action (the reference raises before stepping, MRS.py:247-248; device-resident actions cannot): the agent
    // gets no rotor forces in this step, like MRS.step(None) (MRS.py:243,252), its PID state stays as it is
    const bool nan_act = status != 0u;
    if (nan_act) {
        rpm[0] = rpm[1] = rpm[2] = rpm[3] = 0.f;
    } else {
        action_to_rpm<MODE>(c, c.quad, d, st, R, act, k, rpm);
    }
    if (b.rpm && MODE != MRS_NO_ACTION && mine) {
#pragma unroll
        for (int i = 0; i < 4; ++i) b.rpm[(size_t)i * S + s] = rpm[i];
    }
    // pair pass 1: downwash on the pre-step positions
    __syncwarp();
    wpos[lane] = make_float4(st.px, st.py, st.pz, 0.f);
    __syncwarp();
    // ... and the rounds of the tournament in which some pair of this warp is in range (positions do not change
    // during the solve): every lane marks the rounds of its own pairs, the warp ORs them
    float dw = 0.f;
    unsigned my_rounds = 0u;
#pragma unroll
    for (int r = 1; r < (GT ? GT : G); ++r) {
        const int j = ai ^ r;
        if (j < N) {
            const float4 pj = wpos[gb + j];
            const float rx = pj.x - st.px, ry = pj.y - st.py, rz = pj.z - st.pz;
            const float dxy2 = rx * rx + ry * ry;
            if (MODE != MRS_NO_ACTION) dw += downwash_pair(c.quad, d, dxy2, rz);
            if (dxy2 + rz * rz < cp.lim2) my_rounds |= 1u << tour_round_small(min(ai, j), max(ai, j), N);
        }
    }
    if (nan_act) dw = 0.f;
    apply_wrench<MODE != MRS_NO_ACTION>(c, d, st, R, rpm, dw);
    // ---- contact solve
    const bool gcand = cp.ground_contact && valid && st.pz < cp.gnd_skip_z;
    GroundRows g;
    g.act = 0u;
    if (gcand) ground_setup(cp, st.pz, R, g);
    const unsigned ract = __reduce_or_sync(kFull32, (cp.agent_contact && valid) ? my_rounds : 0u);
    if (__any_sync(kFull32, g.act != 0u) || ract) {
        float lam_g[4] = {0.f, 0.f, 0.f, 0.f}, fl[2] = {0.f, 0.f};
        // pair impulses, three per round.  N = 8: seven rounds, walked by an unrolled loop so that the impulses stay in
        // registers and the partner of a round is a compile-time function of the lane; wider groups index the
        // array by the round (local memory) and walk only the occupied rounds
        constexpr bool kStaticRounds = false;   // measured at N = 8: the unrolled walk makes the sweep loop 1170 instructions
                                                // (instruction-fetch stalls), 165 vs 150 us per step on the collapsed C5 swarm
        constexpr int kRoundsMax = GT ? GT - 1 : 31;
        float lam_p[3 * kRoundsMax];
        if constexpr (kStaticRounds) {
#pragma unroll
            for (int i = 0; i < 3 * kRoundsMax; ++i) lam_p[i] = 0.f;
        } else {
            for (unsigned m = ract; m; m &= m - 1u) {
                const int r = __ffs(m) - 1;
                lam_p[3 * r] = lam_p[3 * r + 1] = lam_p[3 * r + 2] = 0.f;
            }
        }
        float v[3] = {st.vx, st.vy, st.vz};
        float wb[3] = {R[0] * st.wx + R[3] * st.wy + R[6] * st.wz, R[1] * st.wx + R[4] * st.wy + R[7] * st.wz,
                       R[2] * st.wx + R[5] * st.wy + R[8] * st.wz};
        // An env stops sweeping when ITS rows have converged (like the oracle), whatever the other envs of the warp
        // do: its result does not depend on which envs it shares a warp with (shard invariance).
        bool alive = valid;
        float worst;
        auto do_round = [&](int r, float* lam3) {
            const int j = valid ? tour_partner(r, ai, N) : ai;
            const float vj[3] = {__shfl_sync(kFull32, v[0], gb + j), __shfl_sync(kFull32, v[1], gb + j),
                                 __shfl_sync(kFull32, v[2], gb + j)};
            if (alive && j != ai) {
                const float4 pj = wpos[gb + j];
                float dv[3];
                bool on;
                const float wr = pair_rows(cp, st.px - pj.x, st.py - pj.y, st.pz - pj.z, v, vj, lam3, dv, on);
                v[0] += dv[0]; v[1] += dv[1]; v[2] += dv[2];
                worst = fmaxf(worst, wr);
            }
        };
        for (int it = 0; it < cp.solver_iters; ++it) {
            worst = 0.f;
            if (alive && g.act) worst = ground_sweep(cp, g, lam_g, fl, v, wb);
            if constexpr (kStaticRounds) {
#pragma unroll
                for (int r = 0; r < kRoundsMax; ++r)
                    if ((ract >> r) & 1u) do_round(r, lam_p + 3 * r);
            } else {
                for (unsigned m = ract; m; m &= m - 1u) {
                    const int r = __ffs(m) - 1;
                    do_round(r, lam_p + 3 * r);
                }
            }
            if (alive) ++n_sweeps;
            for (int o = G >> 1; o > 0; o >>= 1) worst = fmaxf(worst, __shfl_xor_sync(kFull32, worst, o));
            alive = alive && !(worst < cp.solver_tol);
            if (!__any_sync(kFull32, alive)) break;
        }
        st.vx = v[0]; st.vy = v[1]; st.vz = v[2];
        st.wx = R[0] * wb[0] + R[1] * wb[1] + R[2] * wb[2];
        st.wy = R[3] * wb[0] + R[4] * wb[1] + R[5] * wb[2];
        st.wz = R[6] * wb[0] + R[7] * wb[1] + R[8] * wb[2];
        if ((lam_g[0] + lam_g[1]) + (lam_g[2] + lam_g[3]) > 0.f) ++n_ground;
        if constexpr (kStaticRounds) {
#pragma unroll
            for (int r = 0; r < kRoundsMax; ++r)
                if (((ract >> r) & 1u) && lam_p[3 * r] > 0.f) ++n_agent_rows;
        } else {
            for (unsigned m = ract; m; m &= m - 1u)
                if (lam_p[3 * (__ffs(m) - 1)] > 0.f) ++n_agent_rows;
        }
    }
    integrate(c, d, st);
    if (!agent_finite(st)) status |= MRS_STATUS_NONFINITE;
    // ---- observation + state
    if (a.X0 && mine) write_X(a.X0 - (long long)t * a.xstride, c.state_layout, s, st);
    if (a.A0) {
        float* Arow = a.A0 - (long long)t * a.astride + (size_t)s * N;
        __syncwarp();
        wpos[lane] = make_float4(st.px, st.py, st.pz, 0.f);
        __syncwarp();
        if (mine) {
            for (int j = 0; j < N; ++j) {
                const float4 pj = wpos[gb + j];
                const float hit = d.comm_inf ? 1.f : adjacency_pair(st.px, st.py, st.pz, pj.x, pj.y, pj.z, d.s_max);
                MRS_TAPE_ST(Arow + j, (j == ai) ? 0.f : hit);
            }
        }
        __syncwarp();
    }
    if (!mine) { status = 0; n_agent_rows = 0; n_ground = 0; n_sweeps = 0; }
    {
        const unsigned any_status = __reduce_or_sync(kFull32, status);
        const unsigned sum_rows = __reduce_add_sync(kFull32, n_agent_rows);
        const unsigned sum_gnd = __reduce_add_sync(kFull32, n_ground);
        const unsigned max_sw = __reduce_max_sync(kFull32, n_sweeps);
        if (lane == 0) {
            if (any_status) atomicOr(&sh_events[0], any_status);
            if (sum_rows) atomicAdd(&sh_events[1], sum_rows);
            if (sum_gnd) atomicAdd(&sh_events[2], sum_gnd);
            if (any_status & MRS_STATUS_NONFINITE) atomicAdd(&sh_events[3], 1u);
            if (any_status & MRS_STATUS_NAN_ACTION) atomicAdd(&sh_events[4], 1u);
            if (max_sw) atomicAdd(&sh_events[6], max_sw);
        }
    }
  }
    if (mine) {
        store_agent(b.state, S, s, st);
        store_ctrl<MODE>(b.ctrl, S, s, k);
    }
}

// dynamic shared memory of one warp of the group kernel: pair tile (+ prefetch stage for full chunks)
template <int MODE, int GT> __host__ __device__ constexpr int group_warp_smem_bytes() {
#ifdef MRS_EXP_OLDSMEM
    return 1024 + ((MRS_PREFETCH && GT != 0) ? mode_stage_floats<MODE>() * 4 : 0);
#else
    return 512 + ((MRS_PREFETCH && GT != 0) ? mode_stage_floats<MODE>() * 4 : 0);
#endif
}

//
// MANY: T > 1 steps per launch (mrs_step_many: the state stays in registers across steps); the single-step
// kernels carry no step loop, no action double-buffering and no tape strides.
//
// Hand-over between consecutive single-step launches (kHand: SM-filling CTAs over full chunks, a.role != 0; host
// side: mrs_rollout).  Envs are independent, so chunk range r of step t+1 depends on range r of step t ONLY.
// With a grid-wide dependency every step pays the slowest SM of the previous one plus the grid boundary
// (tools/trace_c5.py: first CTA done after 14.4 us, last after 16.6 us, next grid released 0.8 us later).
// Instead a CTA that finishes range r publishes r in a queue (bufs.sync) and CTA i of the NEXT launch -- the block
// scheduler starts CTAs in index order on whichever SM has just become free -- takes the i-th finished range:
// ranges flow from launch to launch in completion order and an SM never waits for another SM.
//   sync[0]               epoch: bumped by the head of every chain
//   sync[8 + q]           ranges published so far by the launch that owns queue q = position & 7
//   sync[16 + 1024 q + i] i-th range published by that launch: epoch << 32 | (position + 1) << 16 | range
// role 1 (head, position 0): waits for the whole previous grid (griddepcontrol.wait), resets the counters, bumps
//   the epoch, takes range = blockIdx, publishes.
// role 2 (link, position t): does NOT wait for the previous grid; CTA i waits for entry i of launch t - 1; its
//   it also waits for the LAST entry of launch t - 3 (bounds the launches in flight behind a slow CTA), and its
//   first CTA clears the counter of queue (t + 4) & 7 -- last used by launch t - 4, next by launch t + 4.
// All state / PID / action reads of these kernels are cp.async.cg (L2); the publishing thread fences after the
// CTA barrier that follows the state stores.  A link that waits longer than 2 s falls back to the grid-wide wait
// and raises MRS_STATUS_SYNC_TIMEOUT.
constexpr int kSyncCount = 8, kSyncQueue = 16, kSyncQueueLen = 1024, kSyncQueues = 8;
#ifndef MRS_DEFAULT_CPS
#define MRS_DEFAULT_CPS 4          // CTAs per SM of the single-step SM-filling shape (each with 1 / CPS of the SM's warps)
#endif
static_assert(kSyncQueue + kSyncQueues * kSyncQueueLen <= MRS_SYNC_WORDS, "sync buffer layout");

template <int MODE, int GT, int WPB, bool BAKED, bool MANY>
__global__ void __launch_bounds__(WPB * 32, WPB == 4 ? ModeTraits<MODE>::minb : (4 * ModeTraits<MODE>::minb) / WPB)
#ifdef MRS_EXP_NOGC
step_group_kernel(const __grid_constant__ MrsConfig c_in, const __grid_constant__ Derived d_in, const MrsBuffers b,
                  const StepArgs a) {
#else
step_group_kernel(const __grid_constant__ MrsConfig c_in, const __grid_constant__ Derived d_in,
                  const __grid_constant__ MrsBuffers b, const __grid_constant__ StepArgs a) {
#endif
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
            apply_wrench<MODE != MRS_NO_ACTION>(c, d, st, R, rpm, dw);
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
                if (lane == 0) {
                    if (any_status) atomicOr(&sh_events[0], any_status);
                    if (sum_rows) atomicAdd(&sh_events[1], sum_rows);
                    if (sum_gnd) atomicAdd(&sh_events[2], sum_gnd);
                    if (any_status & MRS_STATUS_NONFINITE) atomicAdd(&sh_events[3], 1u);
                    if (any_status & MRS_STATUS_NAN_ACTION) atomicAdd(&sh_events[4], 1u);
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
            chunk_step_contact<MODE, GT>(&c_in, &d_in, &b, &a, GT ? GT : a.G, pc, (int)(e & 0xffffu), T, kFull32, wpos, sh_events);
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
}

// ------------------------------------------------------------------------------ wide path (N > 32)
// An env no longer fits a warp, so the pair passes are spread over LPA lanes PER AGENT (LPA = 8 for
// N <= 128, else 32): every lane walks the partners j = l, l + LPA, ... of its agent straight from
// the L1/L2-resident position planes, the partial sums are combined with a fixed-order xor-shuffle
// tree (deterministic), and the group's lane 0 runs the per-agent part.  One env of 4096 agents
// therefore fills the GPU with 4096 warps instead of 32 CTAs.
// scratch planes: 0-2 unconstrained velocity, 3-5 pre-step position, 6 contact-proximity flag.
template <int LPA>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = LPA / 2; o > 0; o >>= 1) v += __shfl_xor_sync(kFull32, v, o);
    return v;
}

// per-agent part of the wide pre pass: controller -> rotor wrench + aero (dw = downwash sum) ->
// unconstrained velocities; stashes v*, the pre-step position and the proximity flag in scratch
template <int MODE>
__device__ __forceinline__ void agent_pre(const MrsConfig& c, const Derived& d, const MrsBuffers& b,
                                          const float* __restrict__ actions, unsigned S, unsigned s, float dw, bool near) {
    Agent st;
    Ctrl k;
    load_agent(b.state, S, s, st);
    load_ctrl<MODE>(b.ctrl, S, s, k);
    const float pix = st.px, piy = st.py, piz = st.pz;
    float act[4];
    unsigned status = 0;
    if (load_action<MODE>(actions, s, act)) status |= MRS_STATUS_NAN_ACTION;
    float R[9], rpm[4];
    quat_to_mat(st, R);
    if (status) {            // NaN action: no rotor forces in this step, PID state untouched (see chunk_step_contact)
        rpm[0] = rpm[1] = rpm[2] = rpm[3] = 0.f;
        dw = 0.f;
    } else {
        action_to_rpm<MODE>(c, c.quad, d, st, R, act, k, rpm);
    }
    apply_wrench<MODE != MRS_NO_ACTION>(c, d, st, R, rpm, dw);
    float* sc = b.scratch;
    sc[0 * (size_t)S + s] = st.vx; sc[1 * (size_t)S + s] = st.vy; sc[2 * (size_t)S + s] = st.vz;
    sc[3 * (size_t)S + s] = pix; sc[4 * (size_t)S + s] = piy; sc[5 * (size_t)S + s] = piz;
    sc[6 * (size_t)S + s] = near ? 1.f : 0.f;
    b.state[10 * (size_t)S + s] = st.wx; b.state[11 * (size_t)S + s] = st.wy; b.state[12 * (size_t)S + s] = st.wz;
    store_ctrl<MODE>(b.ctrl, S, s, k);
    if (b.rpm && MODE != MRS_NO_ACTION) {
#pragma unroll
        for (int i = 0; i < 4; ++i) b.rpm[i * (size_t)S + s] = rpm[i];
    }
    if (status && b.status) {
        atomicOr(b.status, status);
        if (b.stats) atomicAdd(b.stats + MRS_STAT_NAN_ACTIONS, 1ull);
    }
}

template <int MODE, int LPA>
__global__ void __launch_bounds__(kBlock)
step_pre_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b,
                const float* __restrict__ actions) {
    pdl_enter();
    const int N = c.N;
    const unsigned S = (unsigned)c.E * (unsigned)N;
    const unsigned gid = (blockIdx.x * kBlock + threadIdx.x) / LPA;      // agent slot of this lane group
    const int l = threadIdx.x & (LPA - 1);
    const bool valid = gid < S;
    const unsigned s = valid ? gid : 0u;
    const unsigned env0 = (s / (unsigned)N) * (unsigned)N;
    const int ai = (int)(s - env0);
    const float* __restrict__ px = b.state + 0 * (size_t)S + env0;
    const float* __restrict__ py = b.state + 1 * (size_t)S + env0;
    const float* __restrict__ pz = b.state + 2 * (size_t)S + env0;
    const float pix = px[ai], piy = py[ai], piz = pz[ai];
    float dw = 0.f;
    bool near = false;
    const bool pair_contact = c.phys.agent_contact && N > 1;
    if (MODE != MRS_NO_ACTION || pair_contact) {
        // Uniform trip count for the whole warp (the vote below needs every lane).  The SFU part of the
        // downwash is skipped for a whole warp when none of its 32 pairs can contribute: partner not
        // above (rz <= 0), dxy >= 10, or exp(-0.5 (dxy/beta)^2) underflowing float32 (0.5 q^2 > 104).
        // Consecutive partners share a height layer in a lattice-like swarm, so the vote is mostly uniform.
        // four partners per lane and iteration: independent loads in flight, one vote per four pairs
        for (int j0 = 0; j0 < N; j0 += 4 * LPA) {
            float dxy2[4], rz[4];
            bool live[4], any_live = false;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = j0 + u * LPA + l;
                const bool in = j < N;
                const int jj = in ? j : ai;
                const float rx = px[jj] - pix, ry = py[jj] - piy;
                rz[u] = pz[jj] - piz;
                dxy2[u] = rx * rx + ry * ry;
                const bool other = in && j != ai;
                const float beta = c.quad.dw2 * rz[u] + c.quad.dw3;
                live[u] = MODE != MRS_NO_ACTION && other && rz[u] > 0.f && dxy2[u] < 100.f &&
                          !(dxy2[u] > 208.f * beta * beta);
                any_live = any_live || live[u];
                near = near || (other && dxy2[u] + rz[u] * rz[u] < d.lim2);
            }
            if (MODE != MRS_NO_ACTION && __any_sync(kFull32, any_live)) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float f = downwash_pair(c.quad, d, dxy2[u], rz[u]);
                    dw += live[u] ? f : 0.f;
                }
            }
        }
    }
    static_assert(LPA <= 32, "N > 128 uses pair_tile_kernel");
    dw = group_sum<LPA>(dw);
    const unsigned gmask = (LPA == 32) ? kFull32 : (((1u << (LPA & 31)) - 1u) << ((threadIdx.x & 31) & ~(LPA - 1)));
    near = (__ballot_sync(kFull32, near) & gmask) != 0u;
    if (l != 0 || !valid) return;
    agent_pre<MODE>(c, d, b, actions, S, s, dw, near && pair_contact);
}

// ------------------------------------------------------------------------------ pre pass, 32 < N <= 128, many agents
// One THREAD per agent.  A CTA covers 128 consecutive agent slots (they may span several envs); the positions
// of all envs it touches go to shared memory once (<= 128 + 2 (N - 1) slots) and every thread walks the N
// partners of its own env there with the pair loop of pair_tile_kernel (17 instructions per pair without the
// downwash term, warp vote around it, `0 < d2 < lim2` on the float bits so that the agent itself needs no
// special case), then runs the per-agent part itself.  With 8 lanes per agent (step_pre_kernel) seven of the
// eight lanes idle through the ~500 instructions of the per-agent part and a pair costs 45 instructions;
// this shape needs a quarter of the lane-instructions once there are enough agents to fill the GPU.
constexpr int kMidTile = kBlock + 2 * (128 - 1);

template <int MODE>
__global__ void __launch_bounds__(kBlock)
step_mid_pre_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b,
                    const float* __restrict__ actions) {
    __shared__ float4 tile[kMidTile];
    pdl_enter();
    const int N = c.N;
    const unsigned S = (unsigned)c.E * (unsigned)N;
    const unsigned s0 = blockIdx.x * (unsigned)kBlock;
    const unsigned sl = min(s0 + (unsigned)kBlock, S) - 1u;            // last slot of this CTA
    const unsigned e_first = s0 / (unsigned)N, e_last = sl / (unsigned)N;
    const unsigned t0 = e_first * (unsigned)N;                          // first slot in the tile
    const unsigned count = (e_last + 1u) * (unsigned)N - t0;
    for (unsigned idx = threadIdx.x; idx < count; idx += kBlock)
        tile[idx] = make_float4(b.state[t0 + idx], b.state[(size_t)S + t0 + idx], b.state[2 * (size_t)S + t0 + idx], 0.f);
    __syncthreads();
    const unsigned s = s0 + threadIdx.x;
    const bool valid = s < S;
    const unsigned sv = valid ? s : sl;
    const unsigned base = (sv / (unsigned)N) * (unsigned)N - t0;       // my env's first entry in the tile
    const float4 me = tile[sv - t0];
    const bool pair_contact = c.phys.agent_contact && N > 1;
    const unsigned lim_m1 = __float_as_uint(d.lim2) - 1u;
    float dw = 0.f;
    bool near = false;
    for (int j0 = 0; j0 < N; j0 += 4) {
        float dxy2[4], rz[4];
        bool live[4], any_live = false;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = min(j0 + u, N - 1);                           // the tail repeats the last partner ...
            const bool in = j0 + u < N;                                 // ... without counting it
            const float4 pj = tile[base + j];
            const float rx = pj.x - me.x, ry = pj.y - me.y;
            rz[u] = pj.z - me.z;
            dxy2[u] = rx * rx + ry * ry;
            const float d2 = dxy2[u] + rz[u] * rz[u];
            near = near || (in && __float_as_uint(d2) - 1u < lim_m1);
            const float beta = c.quad.dw2 * rz[u] + c.quad.dw3;
            live[u] = MODE != MRS_NO_ACTION && in && rz[u] > 0.f && dxy2[u] < 100.f && !(dxy2[u] > 208.f * beta * beta);
            any_live = any_live || live[u];
        }
        if (MODE != MRS_NO_ACTION && __any_sync(kFull32, any_live)) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float f = downwash_pair(c.quad, d, dxy2[u], rz[u]);
                dw += live[u] ? f : 0.f;
            }
        }
    }
    if (valid) agent_pre<MODE>(c, d, b, actions, S, s, dw, near && pair_contact);
}

// ------------------------------------------------------------------------------ 32 < N <= 128, many envs: the whole step in one launch
// One CTA per env, one thread per agent (blockDim = N rounded up to a warp).  The same arithmetic as the three-kernel
// path above (pair loop of step_mid_pre_kernel, agent_pre, contact_env_body, step_post_kernel, adjacency rows), in the
// same order (results equal to the bit for all modes but set_control, whose mixer ptxas contracts differently in
// the two kernels: float32 rounding there) -- but the unconstrained velocities stay in registers, the
// scratch planes are touched only by an env that has a pair in contact range (CTA-wide vote), and the env's slice of
// A is written by the CTA that has just moved its agents (row-contiguous 16-byte stores) instead of a fourth kernel
// on a side stream.  At 1024 envs x 64 agents: one launch per step instead of four.
template <int MODE>
__global__ void __launch_bounds__(kBlock, 4)
step_env_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b,
                const float* __restrict__ actions, int slot_x, float* __restrict__ A_slice) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ float4 tile[kBlock];
    pdl_enter();
    const int N = c.N, tid = threadIdx.x;
    const unsigned S = (unsigned)c.E * (unsigned)N;
    const unsigned env0 = blockIdx.x * (unsigned)N;
    const bool valid = tid < N;
    const unsigned s = env0 + (unsigned)(valid ? tid : N - 1);
    const MrsPhysicsParams& ph = c.phys;
    Agent st;
    Ctrl k;
    load_agent(b.state, S, s, st);
    load_ctrl<MODE>(b.ctrl, S, s, k);
    tile[tid] = make_float4(st.px, st.py, st.pz, 0.f);
    __syncthreads();
    // ---- pair pass (step_mid_pre_kernel's loop)
    const float4 me = tile[valid ? tid : N - 1];
    const bool pair_contact = ph.agent_contact && N > 1;
    const unsigned lim_m1 = __float_as_uint(d.lim2) - 1u;
    float dw = 0.f;
    bool near = false;
    for (int j0 = 0; j0 < N; j0 += 4) {
        float dxy2[4], rz[4];
        bool live[4], any_live = false;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = min(j0 + u, N - 1);
            const bool in = j0 + u < N;
            const float4 pj = tile[j];
            const float rx = pj.x - me.x, ry = pj.y - me.y;
            rz[u] = pj.z - me.z;
            dxy2[u] = rx * rx + ry * ry;
            const float d2 = dxy2[u] + rz[u] * rz[u];
            near = near || (in && __float_as_uint(d2) - 1u < lim_m1);
            const float beta = c.quad.dw2 * rz[u] + c.quad.dw3;
            live[u] = MODE != MRS_NO_ACTION && in && rz[u] > 0.f && dxy2[u] < 100.f && !(dxy2[u] > 208.f * beta * beta);
            any_live = any_live || live[u];
        }
        if (MODE != MRS_NO_ACTION && __any_sync(kFull32, any_live)) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float f = downwash_pair(c.quad, d, dxy2[u], rz[u]);
                dw += live[u] ? f : 0.f;
            }
        }
    }
    near = near && pair_contact && valid;
    // ---- per-agent part (agent_pre): controller -> rotor wrench + aero -> unconstrained velocities, in registers
    const float pix = st.px, piy = st.py, piz = st.pz;
    float act[4];
    unsigned status = 0;
    if (valid && load_action<MODE>(actions, s, act)) status |= MRS_STATUS_NAN_ACTION;
    float R[9], rpm[4];
    quat_to_mat(st, R);
    if (status) {
        rpm[0] = rpm[1] = rpm[2] = rpm[3] = 0.f;
        dw = 0.f;
    } else {
        action_to_rpm<MODE>(c, c.quad, d, st, R, act, k, rpm);
    }
    apply_wrench<MODE != MRS_NO_ACTION>(c, d, st, R, rpm, dw);
    if (valid) {
        store_ctrl<MODE>(b.ctrl, S, s, k);
        if (b.rpm && MODE != MRS_NO_ACTION) {
#pragma unroll
            for (int i = 0; i < 4; ++i) b.rpm[i * (size_t)S + s] = rpm[i];
        }
    }
    // ---- joint contact solve, only for an env that has a pair in range
    if (__syncthreads_or(near)) {
        float* sc = b.scratch;
        if (valid) {
            sc[0 * (size_t)S + s] = st.vx; sc[1 * (size_t)S + s] = st.vy; sc[2 * (size_t)S + s] = st.vz;
            sc[3 * (size_t)S + s] = pix; sc[4 * (size_t)S + s] = piy; sc[5 * (size_t)S + s] = piz;
            sc[6 * (size_t)S + s] = near ? 1.f : 0.f;
            b.state[10 * (size_t)S + s] = st.wx; b.state[11 * (size_t)S + s] = st.wy; b.state[12 * (size_t)S + s] = st.wz;
        }
        __syncthreads();
        contact_env_body(c, d, b, blockIdx.x, smem_raw);
        __syncthreads();
        if (near) {
            st.vx = sc[0 * (size_t)S + s]; st.vy = sc[1 * (size_t)S + s]; st.vz = sc[2 * (size_t)S + s];
            st.wx = b.state[10 * (size_t)S + s]; st.wy = b.state[11 * (size_t)S + s]; st.wz = b.state[12 * (size_t)S + s];
        }
    }
    // ---- post (step_post_kernel): ground-only solve for agents that touch nothing else, integration, state, X
    unsigned gnd = 0, bad = 0;
    if (valid) {
        if (ph.ground_contact && !near && st.pz < d.gnd_skip_z) {
            if (ground_solve(make_contact_params(ph, d), st, R)) gnd = 1;
        }
        integrate(c, d, st);
        store_agent(b.state, S, s, st);
        if (b.X_tape && c.state_layout != MRS_X_NONE)
            write_X(b.X_tape + (size_t)slot_x * S * state_dim(c.state_layout), c.state_layout, s, st);
        bad = agent_finite(st) ? 0u : 1u;
    }
    {
        const unsigned w_gnd = __reduce_add_sync(kFull32, gnd);
        const unsigned w_bad = __reduce_add_sync(kFull32, bad);
        const unsigned w_nan = __reduce_add_sync(kFull32, status ? 1u : 0u);
        if ((tid & 31) == 0) {
            if ((w_bad || w_nan) && b.status)
                atomicOr(b.status, (w_bad ? MRS_STATUS_NONFINITE : 0u) | (w_nan ? MRS_STATUS_NAN_ACTION : 0u));
            if (b.stats) {
                if (w_gnd) atomicAdd(b.stats + MRS_STAT_GROUND_CONTACTS, (unsigned long long)w_gnd);
                if (w_bad) atomicAdd(b.stats + MRS_STAT_NONFINITE, (unsigned long long)w_bad);
                if (w_nan) atomicAdd(b.stats + MRS_STAT_NAN_ACTIONS, (unsigned long long)w_nan);
            }
        }
    }
    // ---- the env's slice of A from the new positions
    if (A_slice) {
        __syncthreads();
        if (valid) tile[tid] = make_float4(st.px, st.py, st.pz, 0.f);
        __syncthreads();
        float* out = A_slice + (size_t)env0 * N;
        if ((N & 3) == 0) {
            const int qpr = N >> 2;                     // quads per row
            for (int q = tid; q < N * qpr; q += blockDim.x) {
                const int i = q / qpr, j = (q - i * qpr) * 4;
                const float4 pi = tile[i];
                float v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float4 pj = tile[j + u];
                    v[u] = (j + u == i) ? 0.f : (d.comm_inf ? 1.f : adjacency_pair(pi.x, pi.y, pi.z, pj.x, pj.y, pj.z, d.s_max));
                }
                __stcs(reinterpret_cast<float4*>(out + (size_t)i * N + j), make_float4(v[0], v[1], v[2], v[3]));
            }
        } else {
            for (int q = tid; q < N * N; q += blockDim.x) {
                const int i = q / N, j = q - i * N;
                const float4 pi = tile[i], pj = tile[j];
                out[q] = (j == i) ? 0.f : (d.comm_inf ? 1.f : adjacency_pair(pi.x, pi.y, pi.z, pj.x, pj.y, pj.z, d.s_max));
            }
        }
    }
}

// ------------------------------------------------------------------------------ pair pass for N > 128
// n-body tiling.  A CTA owns 128 agents of one env (one per thread, own position in registers) and one
// of `nsplit` slices of the partner range; partner positions go through shared memory in tiles of 128
// and every thread reads the SAME partner (broadcast LDS.128), so a pair costs no global load, no index
// arithmetic and no shuffle: ~16 instructions without the downwash term, which is skipped per warp when
// none of its 32 agents can feel this partner (not above, dxy >= 10 m, or exp(-0.5 (dxy/beta)^2)
// underflowing float32).  Partial sums of slice js go to scratch plane kPairPlane0 + js, the proximity
// flag to plane kPairPlane0 + nsplit + js; agent_pre_kernel adds them in slice order (deterministic).
// (The first version gave every agent a whole CTA that walked the partners from the L1-resident position
// planes: 45 instructions per pair, 29.9 us at N = 4096.)

template <int MODE>
__global__ void __launch_bounds__(kBlock)
pair_tile_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b, int jw,
                 int nsplit) {
    __shared__ float4 tile[kBlock];
    pdl_enter();
    const int N = c.N;
    const unsigned S = (unsigned)c.E * (unsigned)N;
    const int itiles = (N + kBlock - 1) / kBlock;
    const unsigned per_env = (unsigned)(itiles * nsplit);
    const unsigned env = blockIdx.x / per_env, rem = blockIdx.x - env * per_env;
    const int it = (int)(rem / (unsigned)nsplit), js = (int)(rem - (unsigned)it * (unsigned)nsplit);
    const unsigned env0 = env * (unsigned)N;
    const int i = it * kBlock + threadIdx.x;
    const bool valid = i < N;
    const float* __restrict__ px = b.state + 0 * (size_t)S + env0;
    const float* __restrict__ py = b.state + 1 * (size_t)S + env0;
    const float* __restrict__ pz = b.state + 2 * (size_t)S + env0;
    // an idle lane sits far below everything: no partner is above-and-near, none is close
    const float pix = valid ? px[i] : 0.f, piy = valid ? py[i] : 0.f, piz = valid ? pz[i] : 3.0e18f;
    const bool pair_contact = c.phys.agent_contact && N > 1;
    // 0 < d2 < lim2 as ONE unsigned compare of the float bits (d2 >= 0 or NaN): (bits - 1) < (bits(lim2) - 1);
    // d2 == 0 is the agent itself (or a coincident partner, which the contact row ignores anyway)
    const unsigned lim_m1 = __float_as_uint(d.lim2) - 1u;
    float dw = 0.f;
    bool near = false;
    // Tile culling: a tile whose highest partner lies more than the contact range below the lowest agent of
    // this warp can neither blow on any of them (dz <= 0) nor touch them: skipped as a whole (exact, not a
    // cut-off).  It pays when the index order follows height; the C4 bench lattice has z as its fastest
    // index, so no tile is skipped there and the test costs ~1 %.
    __shared__ float tile_zmax[kBlock / 32];
    float wz_min = valid ? piz : 3.0e38f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wz_min = fminf(wz_min, __shfl_xor_sync(kFull32, wz_min, o));
    const float z_skip = wz_min - sqrtf(d.lim2);
    const int jbeg = js * jw, jend = min(jbeg + jw, N);
    for (int j0 = jbeg; j0 < jend; j0 += kBlock) {
        const int jj = j0 + threadIdx.x;
        const float4 mine = (jj < jend) ? make_float4(px[jj], py[jj], pz[jj], 0.f) : make_float4(3.0e18f, 0.f, -3.0e18f, 0.f);
        float zm = mine.z;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) zm = fmaxf(zm, __shfl_xor_sync(kFull32, zm, o));
        __syncthreads();
        tile[threadIdx.x] = mine;
        if ((threadIdx.x & 31) == 0) tile_zmax[threadIdx.x >> 5] = zm;
        __syncthreads();
        const float tz = fmaxf(fmaxf(tile_zmax[0], tile_zmax[1]), fmaxf(tile_zmax[2], tile_zmax[3]));
        if (tz < z_skip) continue;          // warp-uniform
#pragma unroll 2
        for (int jl = 0; jl < kBlock; jl += 4) {
            float dxy2[4], rz[4];
            bool live[4], any_live = false;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float4 pj = tile[jl + u];
                const float rx = pj.x - pix, ry = pj.y - piy;
                rz[u] = pj.z - piz;
                dxy2[u] = rx * rx + ry * ry;
                const float d2 = dxy2[u] + rz[u] * rz[u];
                near = near || (__float_as_uint(d2) - 1u < lim_m1);
                const float beta = c.quad.dw2 * rz[u] + c.quad.dw3;
                live[u] = MODE != MRS_NO_ACTION && rz[u] > 0.f && dxy2[u] < 100.f && !(dxy2[u] > 208.f * beta * beta);
                any_live = any_live || live[u];
            }
            if (MODE != MRS_NO_ACTION && __any_sync(kFull32, any_live)) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float f = downwash_pair(c.quad, d, dxy2[u], rz[u]);
                    dw += live[u] ? f : 0.f;
                }
            }
        }
    }
    if (!valid) return;
    const unsigned s = env0 + (unsigned)i;
    b.scratch[(size_t)(kPairPlane0 + js) * S + s] = dw;
    b.scratch[(size_t)(kPairPlane0 + nsplit + js) * S + s] = (near && pair_contact) ? 1.f : 0.f;
}

// thread-per-agent half of the wide pre pass for N >= 1024 (dw and the proximity flag come from scratch)
template <int MODE>
__global__ void __launch_bounds__(kBlock)
agent_pre_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b,
                 const float* __restrict__ actions, int nsplit) {
    pdl_enter();
    const unsigned S = (unsigned)c.E * (unsigned)c.N;
    const unsigned s = blockIdx.x * kBlock + threadIdx.x;
    if (s >= S) return;
    float dw = 0.f, fl = 0.f;
    for (int j0 = 0; j0 < nsplit; j0 += 8) {       // fixed order: the sum does not depend on the launch shape
        float pd[8], pf[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {              // independent loads in flight
            const bool in = j0 + u < nsplit;
            pd[u] = in ? b.scratch[(size_t)(kPairPlane0 + j0 + u) * S + s] : 0.f;
            pf[u] = in ? b.scratch[(size_t)(kPairPlane0 + nsplit + j0 + u) * S + s] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) { dw += pd[u]; fl += pf[u]; }
    }
    agent_pre<MODE>(c, d, b, actions, S, s, dw, fl != 0.f);
}

// ------------------------------------------------------------------------------ launch
template <int MODE, int GT, int WPB, bool BAKED, bool MANY>
static int launch_group_wpb(const MrsConfig& c, const Derived& d, const MrsBuffers& b, const StepArgs& a_in, long long blocks,
                            bool pdl, cudaStream_t st) {
    StepArgs a = a_in;
    // the parked-chunk list of a CTA (contact path): 4 bytes per chunk the CTA can own
    const long long nwork = a.nchunks - a.chunk_lo;
    a.slow_slots = (WPB > 4) ? (int)((nwork + blocks - 1) / blocks) + 1
                             : WPB * (int)((nwork + blocks * WPB - 1) / (blocks * WPB));
    const size_t smem = (size_t)WPB * group_warp_smem_bytes<MODE, GT>() + (((size_t)a.slow_slots * 4 + 15) & ~(size_t)15);
    if (smem > 200 * 1024) return MRS_ERR_UNSUPPORTED;
    static size_t configured[64] = {};        // per device: the attribute belongs to the function ON a device
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return MRS_ERR_CUDA;
    if (smem > 48 * 1024 && smem > configured[dev]) {
        if (cudaFuncSetAttribute(step_group_kernel<MODE, GT, WPB, BAKED, MANY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
            cudaSuccess)
            return MRS_ERR_CUDA;
        configured[dev] = smem;
    }
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)blocks);
    lc.blockDim = dim3(WPB * 32);
    lc.dynamicSmemBytes = smem;
    lc.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = attr;
    lc.numAttrs = pdl ? 1 : 0;
    if (cudaLaunchKernelEx(&lc, step_group_kernel<MODE, GT, WPB, BAKED, MANY>, c, d, b, a) != cudaSuccess) {
        (void)cudaGetLastError();
        return MRS_ERR_CUDA;
    }
    return last_error();
}

template <int MODE, int GT, int WPB>
static int launch_group_variant(const MrsConfig& c, const Derived& d, const MrsBuffers& b, const StepArgs& a, long long blocks,
                                bool pdl, bool baked, cudaStream_t st) {
    if (a.T > 1)
        return baked ? launch_group_wpb<MODE, GT, WPB, true, true>(c, d, b, a, blocks, pdl, st)
                     : launch_group_wpb<MODE, GT, WPB, false, true>(c, d, b, a, blocks, pdl, st);
    return baked ? launch_group_wpb<MODE, GT, WPB, true, false>(c, d, b, a, blocks, pdl, st)
                 : launch_group_wpb<MODE, GT, WPB, false, false>(c, d, b, a, blocks, pdl, st);
}

template <int MODE, int GT>
static int launch_group(const MrsConfig& c, const Derived& d, const MrsBuffers& b, StepArgs a, cudaStream_t st) {
    constexpr int kBig = 4 * ModeTraits<MODE>::minb;            // warps of a CTA that owns a whole SM
    const int sms = sm_count();
    if (sms <= 0) return MRS_ERR_CUDA;
    static const int use_pdl = env_int("MRS_B200_PDL", 1);
    static const int use_big = env_int("MRS_B200_BIGCTA", 1);
    static const int use_hand = env_int("MRS_B200_HANDOVER", 1);
    // large jobs (every warp of the GPU gets more than two chunks): one SM-sized CTA per SM with the
    // shared-memory hand-out.  Programmatic dependent launch pays off for full waves (measured
    // -2.3 % at C5); partial waves are faster with plain stream order (C3: +11 % with PDL).
    static const int use_baked = env_int("MRS_B200_BAKED", 1);
    const bool baked = use_baked && config_is_baked(c, d);
    const int nwork = a.nchunks - a.chunk_lo;
    if (use_big && nwork > 2 * sms * kBig) {
        // One launch per step: kCps CTAs per SM (each with 1 / kCps of the SM's warps) and the range hand-over
        // between the launches of a chain (mrs_rollout; needs the sync words, PDL, full chunks).  Measured at C5
        // (us per step, 200-step graphs): 1 / 2 / 4 CTAs per SM with a grid-wide dependency 16.7 / 16.6 / 16.8,
        // with the hand-over 17.2 / 14.7 / 14.3 -- an SM-sized CTA leaves its SM idle through its own hand-over
        // latency, four small ones hide it behind each other.  Multi-step launches keep one CTA per SM (4.5e10 vs
        // 3.9e10 agent-steps/s with four).
        if (a.T > 1) {
            a.role = 0;
            return launch_group_variant<MODE, GT, kBig>(c, d, b, a, sms, use_pdl != 0, baked, st);
        }
        static const int cps = env_int("MRS_B200_CPS", MRS_DEFAULT_CPS);          // dev builds: 1, 2 or 4
        if (!(use_hand && use_pdl && b.sync && GT != 0 && sms * cps <= kSyncQueueLen)) a.role = 0;
#ifdef MRS_CPS_VARIANTS
        if (cps == 1) return launch_group_variant<MODE, GT, kBig>(c, d, b, a, sms, use_pdl != 0, baked, st);
        if (cps == 2) return launch_group_variant<MODE, GT, kBig / 2>(c, d, b, a, 2 * sms, use_pdl != 0, baked, st);
#endif
        return launch_group_variant<MODE, GT, kBig / MRS_DEFAULT_CPS>(c, d, b, a, MRS_DEFAULT_CPS * sms, use_pdl != 0, baked, st);
    }
    a.role = 0;
    const long long need = ((long long)nwork + 3) / 4;
    const long long cap = (long long)sms * ModeTraits<MODE>::minb;
    const long long blocks = need < cap ? need : cap;
    const bool pdl = use_pdl && need >= cap;
    return launch_group_variant<MODE, GT, 4>(c, d, b, a, blocks, pdl, baked, st);
}

template <int MODE, int LPA>
static int launch_wide_lpa(const MrsConfig& c, const Derived& d, const MrsBuffers& b, const StepArgs& a, cudaStream_t st) {
    const size_t S = (size_t)c.E * c.N;
    constexpr int A = ModeTraits<MODE>::A;
    const unsigned blocks = (unsigned)((S * LPA + kBlock - 1) / kBlock);
    SideLane* L = (b.A_tape && a.T > 1) ? side_lane() : nullptr;
    int jw = 0, nsplit = 0;
    if (LPA > 32) pair_split(c.E, c.N, &jw, &nsplit);
    for (int t = 0; t < a.T; ++t) {
        const float* act_t = a.actions ? a.actions + (size_t)t * S * A : nullptr;
        if constexpr (LPA > 32) {
            const int itiles = (c.N + kBlock - 1) / kBlock;
            if (int rc = launch_pdl(true, pair_tile_kernel<MODE>, dim3((unsigned)((long long)itiles * nsplit * c.E)), kBlock, 0, st, c, d,
                                    b, jw, nsplit))
                return rc;
            if (int rc = launch_pdl(true, agent_pre_kernel<MODE>, dim3((unsigned)((S + kBlock - 1) / kBlock)), kBlock, 0, st, c, d, b,
                                    act_t, nsplit))
                return rc;
        } else {
            if (int rc = launch_pdl(false, step_pre_kernel<MODE, LPA>, dim3(blocks), kBlock, 0, st, c, d, b, act_t)) return rc;
        }
        if (int rc = launch_contact_env(c, d, b, LPA > 32, st)) return rc;
        if (L && t > 0 && cudaStreamWaitEvent(st, L->adj_done, 0) != cudaSuccess) return MRS_ERR_CUDA;
        if (int rc = launch_step_post(c, d, b, a.slot_x - t, LPA > 32, st)) return rc;
        if (b.A_tape) {
            cudaStream_t as = st;
            if (L) {
                if (cudaEventRecord(L->posted, st) != cudaSuccess) return MRS_ERR_CUDA;
                if (cudaStreamWaitEvent(L->s, L->posted, 0) != cudaSuccess) return MRS_ERR_CUDA;
                as = L->s;
            }
            const int rc = launch_adjacency(b.state, S, 1, b.A_tape + (size_t)(a.slot_a - t) * S * c.N, c.E, c.N, d.s_max,
                                            d.comm_inf, as);
            if (rc) return rc;
            if (L && cudaEventRecord(L->adj_done, L->s) != cudaSuccess) return MRS_ERR_CUDA;
        }
    }
    if (L && cudaStreamWaitEvent(st, L->adj_done, 0) != cudaSuccess) return MRS_ERR_CUDA;
    return last_error();
}

// 32 < N <= 128 with enough agents to fill the GPU: one thread per agent in both passes
template <int MODE>
static int launch_mid(const MrsConfig& c, const Derived& d, const MrsBuffers& b, const StepArgs& a, cudaStream_t st) {
    const size_t S = (size_t)c.E * c.N;
    constexpr int A = ModeTraits<MODE>::A;
    const unsigned blocks = (unsigned)((S + kBlock - 1) / kBlock);
    SideLane* L = (b.A_tape && a.T > 1) ? side_lane() : nullptr;
    for (int t = 0; t < a.T; ++t) {
        const float* act_t = a.actions ? a.actions + (size_t)t * S * A : nullptr;
        if (int rc = launch_pdl(false, step_mid_pre_kernel<MODE>, dim3(blocks), kBlock, 0, st, c, d, b, act_t)) return rc;
        if (int rc = launch_contact_env(c, d, b, false, st)) return rc;
        if (L && t > 0 && cudaStreamWaitEvent(st, L->adj_done, 0) != cudaSuccess) return MRS_ERR_CUDA;
        if (int rc = launch_step_post(c, d, b, a.slot_x - t, false, st)) return rc;
        if (b.A_tape) {
            cudaStream_t as = st;
            if (L) {
                if (cudaEventRecord(L->posted, st) != cudaSuccess) return MRS_ERR_CUDA;
                if (cudaStreamWaitEvent(L->s, L->posted, 0) != cudaSuccess) return MRS_ERR_CUDA;
                as = L->s;
            }
            const int rc = launch_adjacency(b.state, S, 1, b.A_tape + (size_t)(a.slot_a - t) * S * c.N, c.E, c.N, d.s_max,
                                            d.comm_inf, as);
            if (rc) return rc;
            if (L && cudaEventRecord(L->adj_done, L->s) != cudaSuccess) return MRS_ERR_CUDA;
        }
    }
    if (L && cudaStreamWaitEvent(st, L->adj_done, 0) != cudaSuccess) return MRS_ERR_CUDA;
    return last_error();
}

// 32 < N <= 128, many envs: one fused launch per step (step_env_kernel)
template <int MODE>
static int launch_env_fused(const MrsConfig& c, const Derived& d, const MrsBuffers& b, const StepArgs& a, cudaStream_t st) {
    const size_t S = (size_t)c.E * c.N;
    constexpr int A = ModeTraits<MODE>::A;
    const unsigned threads = (unsigned)((c.N + 31) / 32 * 32);
    const size_t smem = contact_env_smem((int)threads, c.N);
    for (int t = 0; t < a.T; ++t) {
        const float* act_t = a.actions ? a.actions + (size_t)t * S * A : nullptr;
        float* A_slice = b.A_tape ? b.A_tape + (size_t)(a.slot_a - t) * S * c.N : nullptr;
        if (int rc = launch_pdl(true, step_env_kernel<MODE>, dim3((unsigned)c.E), threads, smem, st, c, d, b, act_t, a.slot_x - t,
                                A_slice))
            return rc;
    }
    return last_error();
}

template <int MODE>
static int launch_tiled(const MrsConfig& c, const Derived& d, const MrsBuffers& b, const StepArgs& a, cudaStream_t st) {
    if (!b.scratch) return MRS_ERR_ARG;
    if ((unsigned long long)c.E * c.N * 32ull >= 0x7fffffffull * (unsigned long long)kBlock) return MRS_ERR_UNSUPPORTED;
    // lanes-per-agent kernels fill the GPU with few agents (latency); thread-per-agent kernels do a quarter of
    // the work once there are enough of them
    static const long long mid_min = env_int("MRS_B200_MID_MIN_AGENTS", 32768);
    const int fused_mid = env_int("MRS_B200_FUSED_MID", 1);       // 0: the three-kernel path (A/B runs, parity test)
    if (c.N <= 128 && (long long)c.E * c.N >= mid_min)
        return fused_mid ? launch_env_fused<MODE>(c, d, b, a, st) : launch_mid<MODE>(c, d, b, a, st);
    if (c.N <= 128) return launch_wide_lpa<MODE, 8>(c, d, b, a, st);
    return launch_wide_lpa<MODE, 128>(c, d, b, a, st);     // n-body tiles (pair_tile_kernel) + agent_pre_kernel
}

static int pow2ceil(int n) {
    int g = 1;
    while (g < n) g <<= 1;
    return g;
}

template <int MODE>
int dispatch_step(const MrsConfig& c, const MrsBuffers& b, StepArgs a, cudaStream_t st) {
    const Derived d = make_derived(c);
    if (c.N <= 32) {
        a.G = pow2ceil(c.N);
        const size_t S = (size_t)c.E * c.N;
        a.xstride = (long long)(S * (size_t)state_dim(c.state_layout));
        a.astride = (long long)(S * (size_t)c.N);
        a.X0 = (b.X_tape && c.state_layout != MRS_X_NONE) ? b.X_tape + (size_t)a.slot_x * (size_t)a.xstride : nullptr;
        a.A0 = b.A_tape ? b.A_tape + (size_t)a.slot_a * (size_t)a.astride : nullptr;
        const int gpw = 32 / a.G;
        const int nchunks = (c.E + gpw - 1) / gpw;
        a.chunk_lo = 0;
        a.nchunks = nchunks;
        if (c.N != 8 && c.N != 16 && c.N != 32) return launch_group<MODE, 0>(c, d, b, a, st);
        // power-of-two swarms: unrolled pair loops over FULL chunks (32 valid slots); a ragged last chunk
        // (E not a multiple of 32/N) goes to the run-time-width kernel as a one-chunk launch
        const int nfull = c.E / gpw;
        int rc = MRS_OK;
        if (nfull > 0) {
            a.nchunks = nfull;
            switch (c.N) {
                case 8:  rc = launch_group<MODE, 8>(c, d, b, a, st); break;
                case 16: rc = launch_group<MODE, 16>(c, d, b, a, st); break;
                default: rc = launch_group<MODE, 32>(c, d, b, a, st); break;
            }
        }
        if (rc == MRS_OK && nfull < nchunks) {
            a.chunk_lo = nfull;
            a.nchunks = nchunks;
            a.role = 0;
            rc = launch_group<MODE, 0>(c, d, b, a, st);
        }
        return rc;
    }
    return launch_tiled<MODE>(c, d, b, a, st);
}

}  // namespace mrs
