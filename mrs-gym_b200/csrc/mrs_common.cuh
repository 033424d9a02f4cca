// mrs_common.cuh -- shared by every translation unit of libmrs_b200.so: step arguments, SoA state access,
// cp.async helpers, host-side derivation of the per-call constants, and the declarations that tie the per-mode
// step units (mrs_step_mode.cu, one object per ACTION_TYPE) to the ABI unit (mrs_kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "mrs_b200.h"
#include "mrs_device.cuh"
#include "mrs_baked.cuh"

namespace mrs {

constexpr int kBlock = 128;
constexpr unsigned kFull32 = 0xffffffffu;

struct StepArgs {
    const float* actions;  // [T][E][N][A]
    int T;
    int slot_x, slot_a;    // step t writes X tape slot slot_x - t and A tape slot slot_a - t
    // group path: the same as pointers, resolved once on the host (NULL = that tape is not written):
    // step t writes X to X0 - t * xstride and A to A0 - t * astride (strides in floats)
    float* X0;
    float* A0;
    long long xstride, astride;
    int G;                 // group width (power of two >= N), group path only
    int role;              // range hand-over between chained single-step launches: 0 none, 1 head, 2 link (mrs_step.cuh)
    int seq;               // position of the launch in its chain (0 = head)
    int slow_slots;        // entries of a CTA's parked-chunk list (filled in by launch_group_wpb)
    int chunk_lo, nchunks; // this launch walks the warp-sized work items [chunk_lo, nchunks), group path only
};

// ------------------------------------------------------------------------------ state planes
// the six external wrench components of agent slot s (MrsBuffers.wrench, [6][S]): read-only for the whole launch
__device__ __forceinline__ ExtWrench load_wrench(const float* __restrict__ w, unsigned S, unsigned s) {
    ExtWrench x;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        x.f[k] = __ldg(w + (size_t)k * S + s);
        x.t[k] = __ldg(w + (size_t)(3 + k) * S + s);
    }
    return x;
}


__device__ __forceinline__ void load_agent(const float* __restrict__ st, unsigned S, unsigned s, Agent& a) {
    a.px = st[0 * S + s]; a.py = st[1 * S + s]; a.pz = st[2 * S + s];
    a.qx = st[3 * S + s]; a.qy = st[4 * S + s]; a.qz = st[5 * S + s]; a.qw = st[6 * S + s];
    a.vx = st[7 * S + s]; a.vy = st[8 * S + s]; a.vz = st[9 * S + s];
    a.wx = st[10 * S + s]; a.wy = st[11 * S + s]; a.wz = st[12 * S + s];
}

// the same through L2 (ld.global.cg): the contact path reads state another SM may have written moments ago
__device__ __forceinline__ void load_agent_cg(const float* st, unsigned S, unsigned s, Agent& a) {
    a.px = __ldcg(st + 0 * (size_t)S + s); a.py = __ldcg(st + 1 * (size_t)S + s); a.pz = __ldcg(st + 2 * (size_t)S + s);
    a.qx = __ldcg(st + 3 * (size_t)S + s); a.qy = __ldcg(st + 4 * (size_t)S + s); a.qz = __ldcg(st + 5 * (size_t)S + s);
    a.qw = __ldcg(st + 6 * (size_t)S + s);
    a.vx = __ldcg(st + 7 * (size_t)S + s); a.vy = __ldcg(st + 8 * (size_t)S + s); a.vz = __ldcg(st + 9 * (size_t)S + s);
    a.wx = __ldcg(st + 10 * (size_t)S + s); a.wy = __ldcg(st + 11 * (size_t)S + s); a.wz = __ldcg(st + 12 * (size_t)S + s);
}

__device__ __forceinline__ void store_agent(float* __restrict__ st, unsigned S, unsigned s, const Agent& a) {
    st[0 * S + s] = a.px; st[1 * S + s] = a.py; st[2 * S + s] = a.pz;
    st[3 * S + s] = a.qx; st[4 * S + s] = a.qy; st[5 * S + s] = a.qz; st[6 * S + s] = a.qw;
    st[7 * S + s] = a.vx; st[8 * S + s] = a.vy; st[9 * S + s] = a.vz;
    st[10 * S + s] = a.wx; st[11 * S + s] = a.wy; st[12 * S + s] = a.wz;
}

__device__ __forceinline__ void dummy_agent(Agent& a) {
    a.px = a.py = 0.f; a.pz = 1.0e3f;
    a.qx = a.qy = a.qz = 0.f; a.qw = 1.f;
    a.vx = a.vy = a.vz = 0.f;
    a.wx = a.wy = a.wz = 0.f;
}

template <int MODE>
__device__ __forceinline__ void load_ctrl(const float* __restrict__ ct, unsigned S, unsigned s, Ctrl& k) {
    using MT = ModeTraits<MODE>;
    if constexpr (MT::io) {
#pragma unroll
        for (int i = 0; i < 3; ++i) k.io[i] = ct[(0 + i) * S + s];
    }
    if constexpr (MT::ip) {
#pragma unroll
        for (int i = 0; i < 3; ++i) k.ip[i] = ct[(3 + i) * S + s];
    }
    if constexpr (MT::vel) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            k.iv[i] = ct[(6 + i) * S + s];
            k.lve[i] = ct[(9 + i) * S + s];
            k.dve[i] = ct[(12 + i) * S + s];
            k.ltv[i] = ct[(15 + i) * S + s];
        }
    }
}

template <int MODE>
__device__ __forceinline__ void load_ctrl_cg(const float* ct, unsigned S, unsigned s, Ctrl& k) {
    using MT = ModeTraits<MODE>;
    if constexpr (MT::io) {
#pragma unroll
        for (int i = 0; i < 3; ++i) k.io[i] = __ldcg(ct + (size_t)(0 + i) * S + s);
    }
    if constexpr (MT::ip) {
#pragma unroll
        for (int i = 0; i < 3; ++i) k.ip[i] = __ldcg(ct + (size_t)(3 + i) * S + s);
    }
    if constexpr (MT::vel) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            k.iv[i] = __ldcg(ct + (size_t)(6 + i) * S + s);
            k.lve[i] = __ldcg(ct + (size_t)(9 + i) * S + s);
            k.dve[i] = __ldcg(ct + (size_t)(12 + i) * S + s);
            k.ltv[i] = __ldcg(ct + (size_t)(15 + i) * S + s);
        }
    }
}

template <int MODE>
__device__ __forceinline__ void store_ctrl(float* __restrict__ ct, unsigned S, unsigned s, const Ctrl& k) {
    using MT = ModeTraits<MODE>;
    if constexpr (MT::io) {
#pragma unroll
        for (int i = 0; i < 3; ++i) ct[(0 + i) * S + s] = k.io[i];
    }
    if constexpr (MT::ip) {
#pragma unroll
        for (int i = 0; i < 3; ++i) ct[(3 + i) * S + s] = k.ip[i];
    }
    if constexpr (MT::vel) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            ct[(6 + i) * S + s] = k.iv[i];
            ct[(9 + i) * S + s] = k.lve[i];
            ct[(12 + i) * S + s] = k.dve[i];
            ct[(15 + i) * S + s] = k.ltv[i];
        }
    }
}

template <int MODE>
__device__ __forceinline__ bool load_action(const float* __restrict__ actions, size_t idx, float* act) {
    constexpr int A = ModeTraits<MODE>::A;
    if constexpr (A == 4) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(actions) + idx);
        act[0] = v.x; act[1] = v.y; act[2] = v.z; act[3] = v.w;
        return isnan(v.x) || isnan(v.y) || isnan(v.z) || isnan(v.w);
    } else if constexpr (A == 3) {
        const float* p = actions + idx * 3;
        act[0] = __ldg(p); act[1] = __ldg(p + 1); act[2] = __ldg(p + 2); act[3] = 0.f;
        return isnan(act[0]) || isnan(act[1]) || isnan(act[2]);
    } else {
        act[0] = act[1] = act[2] = act[3] = 0.f;
        return false;
    }
}

// tape stores are write-once streams (nobody on the device re-reads a slot soon): streaming hint
#ifndef MRS_TAPE_STREAMING
#define MRS_TAPE_STREAMING 1
#endif
#if MRS_TAPE_STREAMING
#define MRS_TAPE_ST(ptr, val) __stcs((ptr), (val))
#else
#define MRS_TAPE_ST(ptr, val) (*(ptr) = (val))
#endif

// newest X slice of one agent (Environment.get_X with the built-in state_fn layouts)
__device__ __forceinline__ void write_X(float* __restrict__ Xs, int layout, unsigned s, const Agent& a) {
    if (layout == MRS_X_POS_VEL) {
        float2* p = reinterpret_cast<float2*>(Xs + (size_t)s * 6);
        MRS_TAPE_ST(p + 0, make_float2(a.px, a.py));
        MRS_TAPE_ST(p + 1, make_float2(a.pz, a.vx));
        MRS_TAPE_ST(p + 2, make_float2(a.vy, a.vz));
    } else if (layout == MRS_X_FULL) {
        float* p = Xs + (size_t)s * 13;
        p[0] = a.px; p[1] = a.py; p[2] = a.pz;
        p[3] = a.qx; p[4] = a.qy; p[5] = a.qz; p[6] = a.qw;
        p[7] = a.vx; p[8] = a.vy; p[9] = a.vz;
        p[10] = a.wx; p[11] = a.wy; p[12] = a.wz;
    }
}

// ------------------------------------------------------------------------------ async staging
// The group kernel walks several warp-chunks per warp.  While chunk c is being computed, the 13
// state planes (+ the first action) of chunk c+1 are already in flight to a per-warp shared-memory
// stage through cp.async (LDGSTS): the load latency of a chunk is hidden behind the arithmetic of
// the previous one without holding a second register copy of the state.  Stage layout per warp
// (floats): 13 state planes x 32 | the mode's PID planes x 32 | 32 actions x ACTION_DIM; everything is
// moved as 16-byte pieces (a plane's share of a chunk is 128 contiguous bytes = 8 pieces).
#ifndef MRS_PREFETCH
#define MRS_PREFETCH 1
#endif

__device__ __forceinline__ void cp_async4(float* smem, const float* gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async16(float* smem, const float* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// acquire / release accesses and the nanosecond clock of the launch-to-launch range hand-over
__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// ------------------------------------------------------------------------------ host side
inline int sm_count() {
    static int g_sm_count = 0;
    if (g_sm_count == 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
        g_sm_count = n;
    }
    return g_sm_count;
}

inline int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

// Programmatic dependent launch for the multi-kernel paths (N > 32: pre / contact / post): a kernel lets its
// successor start launching at once and waits for its predecessor's completion + flush before it touches memory, so
// launch latency and the prologue overlap the predecessor's tail.  Every kernel launched through launch_pdl calls
// pdl_enter() first; without the launch attribute both instructions are no-ops.  Measured: C4 (one env x 4096
// agents, four kernels per step) 37.2 -> 31.0 us per step; 1024 envs x 64 agents (thread-per-agent path, adjacency
// of the previous step on a side stream) 29.4 -> 32.0 us, so only the N > 128 path asks for it.
__device__ __forceinline__ void pdl_enter() {
    asm volatile("griddepcontrol.launch_dependents;\n\tgriddepcontrol.wait;" ::: "memory");
}

template <typename... KArgs, typename... Args>
inline int launch_pdl(bool pdl, void (*kernel)(KArgs...), dim3 grid, unsigned block, size_t smem, cudaStream_t st, Args... args) {
    static const int use_pdl = env_int("MRS_B200_PDL", 1);
    cudaLaunchConfig_t lc = {};
    lc.gridDim = grid;
    lc.blockDim = dim3(block);
    lc.dynamicSmemBytes = smem;
    lc.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = attr;
    lc.numAttrs = (pdl && use_pdl) ? 1 : 0;
    if (cudaLaunchKernelEx(&lc, kernel, KArgs(args)...) != cudaSuccess) {
        (void)cudaGetLastError();
        return MRS_ERR_CUDA;
    }
    return MRS_OK;
}

// largest float s with sqrt_rn(s) <= r  (see adjacency_pair)
inline float adjacency_threshold(float r) {
    if (!(r >= 0.f)) return -1.f;          // negative or NaN range: nothing is adjacent
    if (isinf(r)) return INFINITY;
    float s = r * r;
    if (isinf(s)) return 3.402823466e+38f;  // every finite squared distance qualifies
    while (sqrtf(s) > r) s = nextafterf(s, -INFINITY);
    for (;;) {
        const float up = nextafterf(s, INFINITY);
        if (isinf(up) || sqrtf(up) > r) break;
        s = up;
    }
    return s;
}

inline int check_cfg(const MrsConfig* cfg) {
    if (!cfg) return MRS_ERR_ARG;
    if (cfg->E <= 0 || cfg->N <= 0 || cfg->K < 0) return MRS_ERR_ARG;
    if (cfg->action_type < 0 || cfg->action_type > MRS_NO_ACTION) return MRS_ERR_ARG;
    if (cfg->state_layout < 0 || cfg->state_layout > MRS_X_FULL) return MRS_ERR_ARG;
    return MRS_OK;
}

inline int last_error() { return cudaGetLastError() == cudaSuccess ? MRS_OK : MRS_ERR_CUDA; }

inline Derived make_derived(const MrsConfig& c) {
    Derived d;
    const MrsQuadParams& q = c.quad;
    const MrsPhysicsParams& p = c.phys;
    d.inv_mass = (float)(1.0 / (double)p.mass);
    for (int i = 0; i < 3; ++i) d.inv_I[i] = (float)(1.0 / (double)p.inertia[i]);
    const double pr4 = (double)q.prop_radius / 4.0;
    d.gnd_c = (float)((double)q.kf * (double)q.gnd_eff_coeff * pr4 * pr4);
    d.dw_c = (float)((double)q.dw1 * pr4 * pr4);
    d.rpm2rad = (float)(2.0 * 3.14159265358979323846 / 60.0);
    d.q_x2 = (float)(0.25 * (double)c.dt * (double)c.dt);
    d.cap_w2 = (float)(((double)p.ang_motion_threshold / (double)c.dt) * ((double)p.ang_motion_threshold / (double)c.dt));
    const double cap_ang = 0.5 * 1.57079632679489661923 / (double)c.dt;      // Bullet: 0.5 * SIMD_HALF_PI / dt
    d.cap_k = (float)(sin(0.5 * cap_ang * (double)c.dt) / cap_ang);
    d.cap_c = (float)cos(0.5 * cap_ang * (double)c.dt);
    const float lim = 2.f * p.contact_radius + p.contact_margin;
    d.lim2 = lim * lim;
    // no rim point of the collision cylinder reaches lower than sqrt(r^2 + h^2) below the CoM
    d.gnd_skip_z = p.ground_z + p.contact_margin + sqrtf(p.col_radius * p.col_radius + p.col_halfheight * p.col_halfheight) +
                   p.col_margin + 1e-3f;
    d.inv_dt = (float)(1.0 / (double)c.dt);
    d.erp_dt = (float)((double)p.erp2 / (double)c.dt);
    d.comm_inf = isinf(c.comm_range) && c.comm_range > 0.f;
    d.s_max = adjacency_threshold(c.comm_range);
    d.inv_ctrl_dt = (float)(1.0 / (double)q.ctrl_dt);
    d.inv_4kf = (float)(1.0 / (4.0 * (double)q.kf));
    d.inv_pwm_a = (float)(1.0 / (double)q.pwm2rpm_a);
    d.inv_qmass = (float)(1.0 / (double)q.mass);
    return d;
}

// true iff the caller's configuration carries exactly the constants mrs_baked.cuh was generated from
inline bool config_is_baked(const MrsConfig& c, const Derived& d) {
    MrsConfig cc = c;
    Derived dd = d;
    baked_constants(cc, dd);
    return memcmp(&cc, &c, sizeof(MrsConfig)) == 0 && memcmp(&dd, &d, sizeof(Derived)) == 0;
}

constexpr int kPairPlane0 = MRS_SCRATCH_PLANES;      // first partial-sum plane of the tiled pair pass
constexpr int kPairMaxSplit = MRS_SCRATCH_PAIR_SPLITS;

// partner slices of pair_tile_kernel: ~8 CTAs per SM of a B200, at most kPairMaxSplit partial planes, whole
// tiles per slice.  A pure function of (E, N): mrs_scratch_planes sizes the caller's scratch from it.
inline void pair_split(int E, int N, int* jw, int* nsplit) {
    const long long itiles = (N + kBlock - 1) / kBlock;
    const long long want = 8LL * 148;
    long long ns = (want + itiles * E - 1) / (itiles * E);
    if (ns > kPairMaxSplit) ns = kPairMaxSplit;
    if (ns > itiles) ns = itiles;                                                    // at least one tile per slice
    if (ns < 1) ns = 1;
    int w = (int)((N + ns - 1) / ns);
    w = (w + kBlock - 1) / kBlock * kBlock;
    *jw = w;
    *nsplit = (N + w - 1) / w;
}


// defined in mrs_kernels.cu
int launch_adjacency(const float* pos, size_t cs, size_t as, float* A, int E, int N, float s_max, int comm_inf,
                     cudaStream_t st);
// wide path (N > 32): joint contact solve per env (one CTA per env) and the per-agent post pass
int launch_contact_env(const MrsConfig& c, const Derived& d, const MrsBuffers& b, bool pdl, cudaStream_t st);
int launch_step_post(const MrsConfig& c, const Derived& d, const MrsBuffers& b, int slot, bool pdl, cudaStream_t st);
struct SideLane {
    cudaStream_t s = nullptr;
    cudaEvent_t posted = nullptr, adj_done = nullptr;
    bool ok = false;
};
SideLane* side_lane();

// One env.step (T steps) of action mode MODE: defined in mrs_step.cuh, instantiated once per mode in its own
// object file (mrs_step_mode.cu, -DMRS_INSTANTIATE_MODE=k) so that the modes compile in parallel.
template <int MODE>
int dispatch_step(const MrsConfig& c, const MrsBuffers& b, StepArgs a, cudaStream_t st);

}  // namespace mrs
