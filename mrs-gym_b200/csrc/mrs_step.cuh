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
// EXT: b.wrench holds the external wrench (MrsBuffers.wrench), loaded once per call and applied in every step.
template <int MODE, int GT, bool EXT = false>
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
    ExtWrench xw{};
    if constexpr (EXT) {
        if (valid) xw = load_wrench(b.wrench, S, s);
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
    apply_wrench<MODE != MRS_NO_ACTION, EXT>(c, d, st, R, rpm, dw, xw);     // a NaN action keeps the external wrench
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
        // non-finite agents and NaN actions count per agent, like the N > 32 kernels
        const unsigned sum_bad = __reduce_add_sync(kFull32, (status & MRS_STATUS_NONFINITE) ? 1u : 0u);
        const unsigned sum_nan = __reduce_add_sync(kFull32, (status & MRS_STATUS_NAN_ACTION) ? 1u : 0u);
        if (lane == 0) {
            if (any_status) atomicOr(&sh_events[0], any_status);
            if (sum_rows) atomicAdd(&sh_events[1], sum_rows);
            if (sum_gnd) atomicAdd(&sh_events[2], sum_gnd);
            if (sum_bad) atomicAdd(&sh_events[3], sum_bad);
            if (sum_nan) atomicAdd(&sh_events[4], sum_nan);
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


// EXT (the overload with a sixth template argument): the external wrench b.wrench (MrsBuffers.wrench) is bound.
// Every lane loads its agent's six components once per chunk (a multi-step launch keeps them in registers for
// all T steps) and the contact path loads them again; only step_group_kernel<MODE, 0, 4, false, MANY, true>
// is built with it.
template <int MODE, int GT, int WPB, bool BAKED, bool MANY>
__global__ void __launch_bounds__(WPB * 32, WPB == 4 ? ModeTraits<MODE>::minb : (4 * ModeTraits<MODE>::minb) / WPB)
#ifdef MRS_EXP_NOGC
step_group_kernel(const __grid_constant__ MrsConfig c_in, const __grid_constant__ Derived d_in, const MrsBuffers b,
                  const StepArgs a) {
#else
step_group_kernel(const __grid_constant__ MrsConfig c_in, const __grid_constant__ Derived d_in,
                  const __grid_constant__ MrsBuffers b, const __grid_constant__ StepArgs a) {
#endif
    constexpr bool EXT = false;
#include "mrs_step_group_body.cuh"
}

// the same with the external wrench (b.wrench != NULL): run-time width, small CTAs, generic constants only
template <int MODE, int GT, int WPB, bool BAKED, bool MANY, bool EXT>
__global__ void __launch_bounds__(WPB * 32, ModeTraits<MODE>::minb)
step_group_kernel(const __grid_constant__ MrsConfig c_in, const __grid_constant__ Derived d_in,
                  const __grid_constant__ MrsBuffers b, const __grid_constant__ StepArgs a) {
    static_assert(EXT && GT == 0 && WPB == 4 && !BAKED, "wrench kernels: run-time width, small CTAs, generic");
#include "mrs_step_group_body.cuh"
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
// unconstrained velocities; stashes v*, the pre-step position and the proximity flag in scratch.  EXT: plus the
// external wrench b.wrench (MrsBuffers.wrench), which a NaN-action agent keeps
template <int MODE, bool EXT = false>
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
    ExtWrench xw{};
    if constexpr (EXT) xw = load_wrench(b.wrench, S, s);
    apply_wrench<MODE != MRS_NO_ACTION, EXT>(c, d, st, R, rpm, dw, xw);
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
    if (status) {
        if (b.status) atomicOr(b.status, status);
        if (b.stats) atomicAdd(b.stats + MRS_STAT_NAN_ACTIONS, 1ull);
    }
}


template <int MODE, int LPA>
__global__ void __launch_bounds__(kBlock)
step_pre_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b,
                const float* __restrict__ actions) {
    constexpr bool EXT = false;
#include "mrs_step_pre_body.cuh"
}

template <int MODE, int LPA, bool EXT>      // with the external wrench (b.wrench != NULL)
__global__ void __launch_bounds__(kBlock)
step_pre_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b,
                const float* __restrict__ actions) {
    static_assert(EXT, "wrench kernel");
#include "mrs_step_pre_body.cuh"
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
    constexpr bool EXT = false;
#include "mrs_step_mid_pre_body.cuh"
}

template <int MODE, bool EXT>               // with the external wrench (b.wrench != NULL)
__global__ void __launch_bounds__(kBlock)
step_mid_pre_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b,
                    const float* __restrict__ actions) {
    static_assert(EXT, "wrench kernel");
#include "mrs_step_mid_pre_body.cuh"
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
    constexpr bool EXT = false;
#include "mrs_step_env_body.cuh"
}

template <int MODE, bool EXT>               // with the external wrench (b.wrench != NULL)
__global__ void __launch_bounds__(kBlock, 4)
step_env_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b,
                const float* __restrict__ actions, int slot_x, float* __restrict__ A_slice) {
    static_assert(EXT, "wrench kernel");
#include "mrs_step_env_body.cuh"
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
    constexpr bool EXT = false;
#include "mrs_step_agent_pre_body.cuh"
}

template <int MODE, bool EXT>               // with the external wrench (b.wrench != NULL)
__global__ void __launch_bounds__(kBlock)
agent_pre_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b,
                 const float* __restrict__ actions, int nsplit) {
    static_assert(EXT, "wrench kernel");
#include "mrs_step_agent_pre_body.cuh"
}

// ------------------------------------------------------------------------------ launch
// The kernels with the external wrench overload those without (one more template argument, EXT = true), so that
// the kernels without keep their names; a typed pointer picks one of the two.
template <int MODE, int GT, int WPB, bool BAKED, bool MANY, bool EXT>
static auto group_kernel() {
    void (*k)(MrsConfig, Derived, MrsBuffers, StepArgs) = nullptr;
    if constexpr (EXT) k = step_group_kernel<MODE, GT, WPB, BAKED, MANY, true>;
    else k = step_group_kernel<MODE, GT, WPB, BAKED, MANY>;
    return k;
}
template <int MODE, int LPA, bool EXT>
static auto pre_kernel() {
    void (*k)(MrsConfig, Derived, MrsBuffers, const float*) = nullptr;
    if constexpr (EXT) k = step_pre_kernel<MODE, LPA, true>;
    else k = step_pre_kernel<MODE, LPA>;
    return k;
}
template <int MODE, bool EXT>
static auto mid_pre_kernel() {
    void (*k)(MrsConfig, Derived, MrsBuffers, const float*) = nullptr;
    if constexpr (EXT) k = step_mid_pre_kernel<MODE, true>;
    else k = step_mid_pre_kernel<MODE>;
    return k;
}
template <int MODE, bool EXT>
static auto agent_kernel() {
    void (*k)(MrsConfig, Derived, MrsBuffers, const float*, int) = nullptr;
    if constexpr (EXT) k = agent_pre_kernel<MODE, true>;
    else k = agent_pre_kernel<MODE>;
    return k;
}
template <int MODE, bool EXT>
static auto env_kernel() {
    void (*k)(MrsConfig, Derived, MrsBuffers, const float*, int, float*) = nullptr;
    if constexpr (EXT) k = step_env_kernel<MODE, true>;
    else k = step_env_kernel<MODE>;
    return k;
}

template <int MODE, int GT, int WPB, bool BAKED, bool MANY, bool EXT = false>
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
        if (cudaFuncSetAttribute(group_kernel<MODE, GT, WPB, BAKED, MANY, EXT>(), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
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
    if (cudaLaunchKernelEx(&lc, group_kernel<MODE, GT, WPB, BAKED, MANY, EXT>(), c, d, b, a) != cudaSuccess) {
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

// external wrench bound (b.wrench != NULL), any N <= 32 and E: the run-time-width kernels with EXT on the small-CTA
// shape of launch_group -- generic constants, no chained hand-over
template <int MODE>
static int launch_group_ext(const MrsConfig& c, const Derived& d, const MrsBuffers& b, StepArgs a, cudaStream_t st) {
    const int sms = sm_count();
    if (sms <= 0) return MRS_ERR_CUDA;
    static const int use_pdl = env_int("MRS_B200_PDL", 1);
    a.role = 0;
    const long long need = ((long long)(a.nchunks - a.chunk_lo) + 3) / 4;
    const long long cap = (long long)sms * ModeTraits<MODE>::minb;
    const long long blocks = need < cap ? need : cap;
    const bool pdl = use_pdl && need >= cap;
    if (a.T > 1) return launch_group_wpb<MODE, 0, 4, false, true, true>(c, d, b, a, blocks, pdl, st);
    return launch_group_wpb<MODE, 0, 4, false, false, true>(c, d, b, a, blocks, pdl, st);
}

template <int MODE, int LPA, bool EXT>
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
            if (int rc = launch_pdl(true, agent_kernel<MODE, EXT>(), dim3((unsigned)((S + kBlock - 1) / kBlock)), kBlock, 0, st, c, d, b,
                                    act_t, nsplit))
                return rc;
        } else {
            if (int rc = launch_pdl(false, pre_kernel<MODE, LPA, EXT>(), dim3(blocks), kBlock, 0, st, c, d, b, act_t)) return rc;
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
template <int MODE, bool EXT>
static int launch_mid(const MrsConfig& c, const Derived& d, const MrsBuffers& b, const StepArgs& a, cudaStream_t st) {
    const size_t S = (size_t)c.E * c.N;
    constexpr int A = ModeTraits<MODE>::A;
    const unsigned blocks = (unsigned)((S + kBlock - 1) / kBlock);
    SideLane* L = (b.A_tape && a.T > 1) ? side_lane() : nullptr;
    for (int t = 0; t < a.T; ++t) {
        const float* act_t = a.actions ? a.actions + (size_t)t * S * A : nullptr;
        if (int rc = launch_pdl(false, mid_pre_kernel<MODE, EXT>(), dim3(blocks), kBlock, 0, st, c, d, b, act_t)) return rc;
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
template <int MODE, bool EXT>
static int launch_env_fused(const MrsConfig& c, const Derived& d, const MrsBuffers& b, const StepArgs& a, cudaStream_t st) {
    const size_t S = (size_t)c.E * c.N;
    constexpr int A = ModeTraits<MODE>::A;
    const unsigned threads = (unsigned)((c.N + 31) / 32 * 32);
    const size_t smem = contact_env_smem((int)threads, c.N);
    for (int t = 0; t < a.T; ++t) {
        const float* act_t = a.actions ? a.actions + (size_t)t * S * A : nullptr;
        float* A_slice = b.A_tape ? b.A_tape + (size_t)(a.slot_a - t) * S * c.N : nullptr;
        if (int rc = launch_pdl(true, env_kernel<MODE, EXT>(), dim3((unsigned)c.E), threads, smem, st, c, d, b, act_t, a.slot_x - t,
                                A_slice))
            return rc;
    }
    return last_error();
}

// EXT: the external wrench is bound (b.wrench != NULL): the pre / fused kernels with EXT, the rest unchanged
template <int MODE, bool EXT>
static int launch_tiled(const MrsConfig& c, const Derived& d, const MrsBuffers& b, const StepArgs& a, cudaStream_t st) {
    if (!b.scratch) return MRS_ERR_ARG;
    if ((unsigned long long)c.E * c.N * 32ull >= 0x7fffffffull * (unsigned long long)kBlock) return MRS_ERR_UNSUPPORTED;
    // lanes-per-agent kernels fill the GPU with few agents (latency); thread-per-agent kernels do a quarter of
    // the work once there are enough of them
    static const long long mid_min = env_int("MRS_B200_MID_MIN_AGENTS", 32768);
    const int fused_mid = env_int("MRS_B200_FUSED_MID", 1);       // 0: the three-kernel path (A/B runs, parity test)
    if (c.N <= 128 && (long long)c.E * c.N >= mid_min)
        return fused_mid ? launch_env_fused<MODE, EXT>(c, d, b, a, st) : launch_mid<MODE, EXT>(c, d, b, a, st);
    if (c.N <= 128) return launch_wide_lpa<MODE, 8, EXT>(c, d, b, a, st);
    return launch_wide_lpa<MODE, 128, EXT>(c, d, b, a, st);     // n-body tiles (pair_tile_kernel) + agent_pre_kernel
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
        if (b.wrench) return launch_group_ext<MODE>(c, d, b, a, st);
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
    return b.wrench ? launch_tiled<MODE, true>(c, d, b, a, st) : launch_tiled<MODE, false>(c, d, b, a, st);
}

}  // namespace mrs
