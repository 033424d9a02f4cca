// mrs_kernels.cu -- ABI unit of libmrs_b200.so: the C entry points (include/mrs_b200.h), the kernels that
// do not depend on the action mode (adjacency, observe, set_state, spawn, sensors, tape maintenance) and the
// dispatch to the per-mode step units (mrs_step.cuh, one object per mode from mrs_step_mode.cu).
//
// Reference behaviour: /root/reference/mrsgym/MRS.py:240-277 and callees (see mrs_device.cuh);
// Bullet step restated in oracle/bullet_model.py.  No CPU fallback exists in this library.
#include <mutex>

#include "mrs_common.cuh"
#include "mrs_contact_env.cuh"

namespace mrs {

// ------------------------------------------------------------------------------ adjacency
// Flat version, any N and any position layout: one thread per output element.
// pos component c of agent (e, i) = pos[c * cs + (e * N + i) * as].
__global__ void __launch_bounds__(256)
adjacency_flat_kernel(const float* __restrict__ pos, size_t cs, size_t as, float* __restrict__ A, int E, int N,
                      float s_max, int comm_inf) {
    const size_t total = (size_t)E * N * N;
    for (size_t kx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; kx < total; kx += (size_t)gridDim.x * blockDim.x) {
        const int j = (int)(kx % N);
        const size_t row = kx / N;
        const int i = (int)(row % N);
        const size_t e = row / N;
        float v;
        if (i == j) v = 0.f;
        else if (comm_inf) v = 1.f;
        else {
            const size_t si = (e * N + i) * as, sj = (e * N + j) * as;
            v = adjacency_pair(pos[si], pos[cs + si], pos[2 * cs + si], pos[sj], pos[cs + sj], pos[2 * cs + sj], s_max);
        }
        A[kx] = v;
    }
}

// Quad version for N < 128, N % 4 == 0 (swarms of 36 .. 124 agents, many envs): one thread per row and column
// quad, lanes along the columns, so a warp's STG.128 writes whole rows (N = 64: two rows = 512 contiguous
// bytes).  The positions of the few envs a CTA touches are staged in shared memory once: no per-element
// div / mod, no scattered position loads (the flat kernel needs 6 loads and ~25 instructions per element).
constexpr int kQuadTile = 3 * 128;
__global__ void __launch_bounds__(kBlock)
adjacency_quad_kernel(const float* __restrict__ pos, size_t cs, size_t as, float* __restrict__ A, int E, int N,
                      float s_max, int comm_inf) {
    __shared__ float4 tile[kQuadTile];
    const unsigned Q = (unsigned)N / 4u;
    const size_t nquads = (size_t)E * N * Q;
    const size_t g0 = (size_t)blockIdx.x * kBlock;
    const size_t gl = (g0 + kBlock < nquads ? g0 + kBlock : nquads) - 1;
    const size_t e_first = (g0 / Q) / (unsigned)N, e_last = (gl / Q) / (unsigned)N;      // envs of the CTA's rows
    const size_t t0 = e_first * (unsigned)N;
    const unsigned count = (unsigned)((e_last + 1) * (unsigned)N - t0);                   // <= 3 N
    for (unsigned idx = threadIdx.x; idx < count; idx += kBlock) {
        const size_t sj = (t0 + idx) * as;
        tile[idx] = make_float4(pos[sj], pos[cs + sj], pos[2 * cs + sj], 0.f);
    }
    __syncthreads();
    const size_t g = g0 + threadIdx.x;
    if (g >= nquads) return;
    const size_t row = g / Q;                       // agent slot of the row
    const unsigned q = (unsigned)(g - row * Q);
    const unsigned env_base = (unsigned)((row / (unsigned)N) * (unsigned)N - t0);
    const unsigned i = (unsigned)(row - (row / (unsigned)N) * (unsigned)N);
    const float4 pi = tile[(unsigned)(row - t0)];
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const unsigned j = 4u * q + (unsigned)u;
        const float4 pj = tile[env_base + j];
        const float hit = comm_inf ? 1.f : adjacency_pair(pi.x, pi.y, pi.z, pj.x, pj.y, pj.z, s_max);
        v[u] = (j == i) ? 0.f : hit;
    }
    __stcs(reinterpret_cast<float4*>(A + row * (unsigned)N + 4u * q), make_float4(v[0], v[1], v[2], v[3]));
}

// Tiled version for N >= 128, N % 4 == 0.  CTA = kRowTile rows x 512 columns of one env; each
// lane keeps its 4 column positions in registers, row positions are broadcast from shared
// memory, each warp store is 512 contiguous bytes of one A row.
constexpr int kRowTile = 32;
__global__ void __launch_bounds__(kBlock)
adjacency_tiled_kernel(const float* __restrict__ pos, size_t cs, size_t as, float* __restrict__ A, int E, int N,
                       float s_max, int comm_inf) {
    __shared__ float4 rows[kRowTile];
    const int col_tiles = (N + 4 * kBlock - 1) / (4 * kBlock);
    const int ct = blockIdx.x % col_tiles;
    const int rt = blockIdx.x / col_tiles;
    const size_t e = blockIdx.y;
    const size_t env0 = e * N;
    const int i0 = rt * kRowTile;
    const int j = ct * 4 * kBlock + threadIdx.x * 4;
    if (threadIdx.x < kRowTile && i0 + threadIdx.x < N) {
        const size_t si = (env0 + i0 + threadIdx.x) * as;
        rows[threadIdx.x] = make_float4(pos[si], pos[cs + si], pos[2 * cs + si], 0.f);
    }
    float xj[4], yj[4], zj[4];
    const bool col_ok = j < N;
    if (col_ok) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const size_t sj = (env0 + j + u) * as;
            xj[u] = pos[sj]; yj[u] = pos[cs + sj]; zj[u] = pos[2 * cs + sj];
        }
    }
    __syncthreads();
    if (!col_ok) return;
    const int nrows = min(kRowTile, N - i0);
    float* out = A + (env0 + i0) * (size_t)N + j;
    for (int r = 0; r < nrows; ++r) {
        const float4 pi = rows[r];
        const int i = i0 + r;
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (j + u == i) v[u] = 0.f;
            else if (comm_inf) v[u] = 1.f;
            else v[u] = adjacency_pair(pi.x, pi.y, pi.z, xj[u], yj[u], zj[u], s_max);
        }
        __stcs(reinterpret_cast<float4*>(out + (size_t)r * N), make_float4(v[0], v[1], v[2], v[3]));
    }
}

// Compact adjacency for the wire: one bit per entry, ceil(N / 32) words per row (bit j of word w = A[i][32 w + j]).
// One thread per row; a row of N <= 32 floats is read with 128-bit loads when N % 4 == 0.
__global__ void __launch_bounds__(256)
pack_adjacency_kernel(const float* __restrict__ A, unsigned* __restrict__ bits, size_t rows, int N, int W) {
    const size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const float* row = A + r * (size_t)N;
    for (int w = 0; w < W; ++w) {
        unsigned m = 0u;
        const int j1 = min(32, N - 32 * w);
        if ((N & 3) == 0) {
            for (int j = 0; j < j1; j += 4) {
                const float4 v = __ldcs(reinterpret_cast<const float4*>(row + 32 * w + j));
                m |= (v.x != 0.f ? 1u : 0u) << j | (v.y != 0.f ? 2u : 0u) << j | (v.z != 0.f ? 4u : 0u) << j | (v.w != 0.f ? 8u : 0u) << j;
            }
        } else {
            for (int j = 0; j < j1; ++j) m |= (row[32 * w + j] != 0.f ? 1u : 0u) << j;
        }
        bits[r * (size_t)W + w] = m;
    }
}

static int launch_pack_adjacency(const float* A, unsigned* bits, int E, int N, cudaStream_t st) {
    const size_t rows = (size_t)E * N;
    const int W = (N + 31) / 32;
    pack_adjacency_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(A, bits, rows, N, W);
    return last_error();
}

// X of the current state (MRS.calc_Xk outside step)
__global__ void __launch_bounds__(256)
observe_x_kernel(const MrsBuffers b, unsigned S, int layout, int slot) {
    const unsigned s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    Agent st;
    load_agent(b.state, S, s, st);
    write_X(b.X_tape + (size_t)slot * S * (size_t)state_dim(layout), layout, s, st);
}

// ------------------------------------------------------------------------------ set_state
// Object.set_state (Object.py:42-65): euler 'xyz' (extrinsic) -> quaternion xyzw =
// qz(yaw) * qy(pitch) * qx(roll); NULL component = keep; masked per env.
__global__ void __launch_bounds__(256)
set_state_kernel(float* __restrict__ st, size_t S, int N, const float* __restrict__ pos, const float* __restrict__ ori,
                 const float* __restrict__ vel, const float* __restrict__ angvel, const unsigned char* __restrict__ mask) {
    const size_t s = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    if (mask && !mask[s / N]) return;
    if (pos) {
        st[0 * S + s] = pos[3 * s]; st[1 * S + s] = pos[3 * s + 1]; st[2 * S + s] = pos[3 * s + 2];
    }
    if (ori) {
        float sr, cr, sp, cp, sy, cy;
        sincosf(0.5f * ori[3 * s], &sr, &cr);
        sincosf(0.5f * ori[3 * s + 1], &sp, &cp);
        sincosf(0.5f * ori[3 * s + 2], &sy, &cy);
        st[3 * S + s] = sr * cp * cy - cr * sp * sy;
        st[4 * S + s] = cr * sp * cy + sr * cp * sy;
        st[5 * S + s] = cr * cp * sy - sr * sp * cy;
        st[6 * S + s] = cr * cp * cy + sr * sp * sy;
    }
    if (vel) {
        st[7 * S + s] = vel[3 * s]; st[8 * S + s] = vel[3 * s + 1]; st[9 * S + s] = vel[3 * s + 2];
    }
    if (angvel) {
        st[10 * S + s] = angvel[3 * s]; st[11 * S + s] = angvel[3 * s + 1]; st[12 * S + s] = angvel[3 * s + 2];
    }
}

// ------------------------------------------------------------------------------ spawn
// On-device MRS.generate_start_pos / generate_start_ori + reset (MRS.py:127-161,174-184) for the
// default spawn distribution (MRS.default_spawn_dist, MRS.py:69-78): z ~ U[z_lo, z_hi], xy ~ N(0,
// sigma) pulled onto the disc of radius xy_radius when outside it (Util.SphereTransform within=True),
// agents closer than 2*AGENT_RADIUS to another agent of their env are re-drawn until none collides
// (the higher-indexed agent of a colliding pair is re-drawn, so at least one of them stays).
// One warp per env (N <= 32), counter-based RNG (splitmix64 of seed / env / agent / draw), so a reset
// is reproducible from (seed, env) alone and independent of the launch shape.
struct SpawnArgs {
    unsigned long long seed;
    unsigned long long env_offset;      // global index of this shard's first env
    float z_lo, z_hi, xy_radius, xy_sigma;
    float yaw_lo, yaw_hi;
    int max_rounds;
};

__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
__device__ __forceinline__ float u01(unsigned long long h) { return ((h >> 40) + 0.5f) * (1.0f / 16777216.0f); }

// One start position from draw key `key`: Box-Muller xy pulled onto the disc, z uniform (mrs_spawn, mrs_autoreset).
__device__ __forceinline__ void spawn_draw(unsigned long long key, const SpawnArgs& sp, float& x, float& y, float& z) {
    const float u1 = u01(key), u2 = u01(splitmix64(key)), u3 = u01(splitmix64(key ^ 0x5851F42D4C957F2Dull));
    const float r = sp.xy_sigma * sqrtf(-2.f * logf(u1));          // Box-Muller
    float sn, cs;
    sincosf(6.28318530717958647692f * u2, &sn, &cs);
    x = r * cs; y = r * sn;
    const float mag = fmaxf(sqrtf(x * x + y * y), sp.xy_radius);     // SphereTransform(within=True)
    x = x / mag * sp.xy_radius; y = y / mag * sp.xy_radius;
    z = sp.z_lo + (sp.z_hi - sp.z_lo) * u3;
}

// Rejection rounds of one env on one warp (N <= 32, lane = agent): every flagged lane (all of them in round 0) draws
// with key_of(round), then a lane is flagged iff a lower lane lies closer than 2*AGENT_RADIUS.  Returns the rounds
// run; max_rounds means the env did not converge.
template <class KeyOf>
__device__ __forceinline__ int spawn_warp_rounds(const SpawnArgs& sp, int N, int lane, float lim2, KeyOf key_of,
                                                 float& x, float& y, float& z) {
    const bool valid = lane < N;
    bool redraw = true;
    int round = 0;
    for (; round < sp.max_rounds; ++round) {
        if (redraw && valid) spawn_draw(key_of(round), sp, x, y, z);
        bool hit = false;
        for (int j = 0; j < N; ++j) {
            const float xj = __shfl_sync(kFull32, x, j), yj = __shfl_sync(kFull32, y, j), zj = __shfl_sync(kFull32, z, j);
            const float dx = x - xj, dy = y - yj, dz = z - zj;
            hit = hit || (valid && j < lane && dx * dx + dy * dy + dz * dz < lim2);
        }
        redraw = hit;
        if (!__any_sync(kFull32, hit)) break;
    }
    return round;
}

// Attitude and rates of a fresh start: yaw only (roll = pitch = 0), velocities zero.  st: the agent's plane-0 entry.
__device__ __forceinline__ void spawn_write_rest(float* st, size_t S, float yaw) {
    float sy, cy;
    sincosf(0.5f * yaw, &sy, &cy);
    st[3 * S] = 0.f; st[4 * S] = 0.f; st[5 * S] = sy; st[6 * S] = cy;
#pragma unroll
    for (int p = 7; p < 13; ++p) st[p * S] = 0.f;
}

__global__ void __launch_bounds__(128)
spawn_kernel(const __grid_constant__ MrsConfig c, const MrsBuffers b, const SpawnArgs sp,
             const unsigned char* __restrict__ mask, unsigned* __restrict__ failed) {
    const int lane = threadIdx.x & 31;
    const int e = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (e >= c.E) return;
    if (mask && !mask[e]) return;
    const int N = c.N;
    const unsigned S = (unsigned)c.E * (unsigned)N;
    const float lim2 = 4.f * c.phys.agent_radius * c.phys.agent_radius;
    const unsigned long long ge = sp.env_offset + (unsigned long long)e;      // global env index: shards draw different envs
    float x = 0.f, y = 0.f, z = 0.f;
    const int round = spawn_warp_rounds(sp, N, lane, lim2, [&](int r) {
        return splitmix64(sp.seed ^ splitmix64((ge << 20) ^ ((unsigned long long)lane << 12) ^ (unsigned long long)r));
    }, x, y, z);
    if (round >= sp.max_rounds && lane == 0 && failed) atomicAdd(failed, 1u);
    if (lane >= N) return;
    const unsigned s = (unsigned)e * (unsigned)N + (unsigned)lane;
    float* st = b.state;
    st[0 * (size_t)S + s] = x; st[1 * (size_t)S + s] = y; st[2 * (size_t)S + s] = z;
    const unsigned long long ky = splitmix64(sp.seed ^ splitmix64(0xA5A5A5A5ull ^ ((sp.env_offset + (unsigned long long)e) << 20) ^ ((unsigned long long)lane << 12)));
    spawn_write_rest(st + s, S, sp.yaw_lo + (sp.yaw_hi - sp.yaw_lo) * u01(ky));
}

// Wide form (N > 32): one CTA per env, the same draws and the same rejection rule, stated per agent: in round r
// every agent flagged in round r - 1 (all of them in round 0) draws again, then agent i is flagged iff some j < i
// lies closer than 2*AGENT_RADIUS in this round's positions.  The positions live in the env's state planes (L2),
// the per-agent "drew this round" and "flagged" bits in ceil(N/32)-word masks in dynamic shared memory, so N is
// bounded only by that (~900K agents).
// After round 0 a pair of two agents that did not draw was tested in the previous round with the same positions
// and found apart (else the higher one would have drawn), so only pairs with a mover are tested: for every mover a,
// (a, k) for all k > a and, after round 0, for the non-movers k < a (mover pairs once).  A round costs
// movers x N pair tests; the flags are those of the full rule.
// The warp kernel's key packing aliases at agent >= 256 or round >= 4096, so this kernel packs (agent, round) into
// one 64-bit word under a per-env hash; round 0xFFFFFFFF (never drawn: max_rounds is an int) is the yaw's domain.
__device__ __forceinline__ unsigned long long spawn_wide_key(unsigned long long seed, unsigned long long env_hash,
                                                             unsigned agent, unsigned round) {
    return splitmix64(seed ^ splitmix64(env_hash ^ (((unsigned long long)agent << 32) | round)));
}

// The rejection rounds of one env on one CTA (see above); `spawn_bits` holds the two masks.  Returns the rounds run.
__device__ __forceinline__ int spawn_cta_rounds(const SpawnArgs& sp, int N, float lim2, unsigned long long env_hash,
                                                unsigned* spawn_bits, float* px, float* py, float* pz) {
    const int W = (N + 31) / 32;
    unsigned* moved = spawn_bits;          // agents that draw in this round
    unsigned* flag = spawn_bits + W;       // agents flagged by this round's test
    for (int w = threadIdx.x; w < W; w += blockDim.x) moved[w] = (w == W - 1 && (N & 31)) ? (1u << (N & 31)) - 1u : kFull32;
    __syncthreads();
    int round = 0;
    for (; round < sp.max_rounds; ++round) {
        for (int i = threadIdx.x; i < N; i += blockDim.x) {
            if (!((moved[i >> 5] >> (i & 31)) & 1u)) continue;
            spawn_draw(spawn_wide_key(sp.seed, env_hash, (unsigned)i, (unsigned)round), sp, px[i], py[i], pz[i]);
        }
        for (int w = threadIdx.x; w < W; w += blockDim.x) flag[w] = 0u;
        __syncthreads();                   // this round's positions and the cleared flags are visible to the CTA
        for (int w = 0; w < W; ++w) {
            for (unsigned bits = moved[w]; bits; bits &= bits - 1u) {
                const int a = 32 * w + __ffs(bits) - 1;
                const float xa = px[a], ya = py[a], za = pz[a];
                for (int k = a + 1 + threadIdx.x; k < N; k += blockDim.x) {
                    const float dx = xa - px[k], dy = ya - py[k], dz = za - pz[k];
                    if (dx * dx + dy * dy + dz * dz < lim2) atomicOr(&flag[k >> 5], 1u << (k & 31));
                }
                if (round == 0) continue;
                bool hit = false;
                for (int k = threadIdx.x; k < a; k += blockDim.x) {
                    if ((moved[k >> 5] >> (k & 31)) & 1u) continue;
                    const float dx = xa - px[k], dy = ya - py[k], dz = za - pz[k];
                    hit = hit || dx * dx + dy * dy + dz * dz < lim2;
                }
                if (hit) atomicOr(&flag[a >> 5], 1u << (a & 31));
            }
        }
        __syncthreads();
        int any = 0;
        for (int w = threadIdx.x; w < W; w += blockDim.x) {
            moved[w] = flag[w];
            any |= flag[w] != 0u;
        }
        if (!__syncthreads_or(any)) break;
    }
    return round;
}

__global__ void __launch_bounds__(1024)
spawn_wide_kernel(const __grid_constant__ MrsConfig c, const MrsBuffers b, const SpawnArgs sp,
                  const unsigned char* __restrict__ mask, unsigned* __restrict__ failed) {
    extern __shared__ unsigned spawn_bits[];
    const unsigned e = blockIdx.x;
    if (mask && !mask[e]) return;
    const int N = c.N;
    const size_t S = (size_t)c.E * (size_t)N;
    float* st = b.state + (size_t)e * N;
    const float lim2 = 4.f * c.phys.agent_radius * c.phys.agent_radius;
    const unsigned long long env_hash = splitmix64(sp.env_offset + (unsigned long long)e);
    const int round = spawn_cta_rounds(sp, N, lim2, env_hash, spawn_bits, st, st + S, st + 2 * S);
    if (round >= sp.max_rounds && threadIdx.x == 0 && failed) atomicAdd(failed, 1u);
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        const unsigned long long ky = spawn_wide_key(sp.seed, env_hash, (unsigned)i, 0xFFFFFFFFu);
        spawn_write_rest(st + i, S, sp.yaw_lo + (sp.yaw_hi - sp.yaw_lo) * u01(ky));
    }
}

// Raises `kernel`'s dynamic shared-memory limit to `smem` when that is above the default 48 KB (once per size and
// device; configured[dev] keeps the largest size set so far).
template <class Kernel>
static int ensure_dynamic_smem(Kernel kernel, size_t smem, size_t* configured) {
    int dev = 0, optin = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return MRS_ERR_CUDA;
    if (smem > configured[dev] && smem > 48 * 1024) {
        if (cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return MRS_ERR_CUDA;
        if (smem > (size_t)optin) return MRS_ERR_UNSUPPORTED;
        if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return MRS_ERR_CUDA;
        configured[dev] = smem;
    }
    return MRS_OK;
}

static int launch_spawn_wide(const MrsConfig& c, const MrsBuffers& b, const SpawnArgs& sp, const unsigned char* mask,
                             unsigned* failed, cudaStream_t st) {
    int threads = (c.N + 31) / 32 * 32;
    if (threads > 1024) threads = 1024;
    const size_t smem = 2 * (size_t)((c.N + 31) / 32) * sizeof(unsigned);
    // the two bit masks grow with N: raise the kernel's dynamic shared-memory limit to the largest size asked for
    static size_t configured[64] = {};
    const int rc = ensure_dynamic_smem(spawn_wide_kernel, smem, configured);
    if (rc) return rc;
    spawn_wide_kernel<<<(unsigned)c.E, (unsigned)threads, smem, st>>>(c, b, sp, mask, failed);
    return last_error();
}

// ------------------------------------------------------------------------------ auto-reset (mrs_autoreset)
// Episode bookkeeping of a closed loop plus the masked reset of the envs whose episode ended (header: the done rule
// and what a reset writes).  The draws are those of mrs_spawn -- spawn_draw and the same rejection rule -- under
// ONE key packing for every N: spawn_wide_key (agent, round) under a per-(env, episode) hash, so a reset depends on
// (seed, env_offset + e, episode) only.
struct AutoResetArgs {
    SpawnArgs sp;
    int episode_length, max_timesteps;
    int slot_x, slot_a;
    float s_max;
    int comm_inf;
};

__device__ __forceinline__ unsigned long long autoreset_env_hash(unsigned long long global_env, unsigned episode) {
    return splitmix64(splitmix64(global_env) ^ splitmix64(0xD1B54A32D192ED03ull ^ (unsigned long long)episode));
}

// the done rule: done_fn / MAX_TIMESTEPS see the count before the step's increment, episode_length the count after
__device__ __forceinline__ bool autoreset_done(const AutoResetArgs& a, const unsigned char* done_in, unsigned e, int n) {
    return (done_in && done_in[e]) || (a.max_timesteps >= 0 && n >= a.max_timesteps) ||
           (a.episode_length > 0 && n + 1 >= a.episode_length);
}

// X0 of agent slot s (position, yaw-only attitude, zero rates: what spawn_write_rest stored) into the K+1 X window
// slots.  Built from registers, not re-read from the state planes this kernel has just written.
__device__ __forceinline__ void autoreset_write_X(const MrsConfig& c, const MrsBuffers& b, const AutoResetArgs& a,
                                                  unsigned S, unsigned s, float x, float y, float z, float yaw) {
    if (!b.X_tape) return;
    Agent ag;
    ag.px = x; ag.py = y; ag.pz = z;
    float sy, cy;
    sincosf(0.5f * yaw, &sy, &cy);
    ag.qx = 0.f; ag.qy = 0.f; ag.qz = sy; ag.qw = cy;
    ag.vx = ag.vy = ag.vz = 0.f;
    ag.wx = ag.wy = ag.wz = 0.f;
    const size_t slot_elems = (size_t)S * (size_t)state_dim(c.state_layout);
    for (int k = 0; k <= c.K; ++k)
        write_X(b.X_tape + (size_t)((a.slot_x + k) % c.L) * slot_elems, c.state_layout, s, ag);
}

__device__ __forceinline__ float autoreset_adjacency(const AutoResetArgs& a, int i, int j, float xi, float yi, float zi,
                                                     float xj, float yj, float zj) {
    return (i == j) ? 0.f : (a.comm_inf ? 1.f : adjacency_pair(xi, yi, zi, xj, yj, zj, a.s_max));
}

// N <= 32: a warp per env, lane = agent, 4 envs per CTA
__global__ void __launch_bounds__(128)
autoreset_kernel(const __grid_constant__ MrsConfig c, const MrsBuffers b, const AutoResetArgs a,
                 const unsigned char* __restrict__ done_in, int* __restrict__ env_steps, unsigned* __restrict__ episode,
                 unsigned char* __restrict__ done_out, unsigned* __restrict__ failed) {
    const int lane = threadIdx.x & 31;
    const unsigned e = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (e >= (unsigned)c.E) return;
    const int n = env_steps[e];
    const bool done = autoreset_done(a, done_in, e, n);
    const unsigned ep = episode[e] + 1u;
    __syncwarp();
    if (!done) {
        if (lane == 0) { env_steps[e] = n + 1; done_out[e] = 0; }
        return;
    }
    const int N = c.N;
    const unsigned S = (unsigned)c.E * (unsigned)N;
    const float lim2 = 4.f * c.phys.agent_radius * c.phys.agent_radius;
    const unsigned long long env_hash = autoreset_env_hash(a.sp.env_offset + e, ep);
    float x = 0.f, y = 0.f, z = 0.f;
    const int round = spawn_warp_rounds(a.sp, N, lane, lim2, [&](int r) {
        return spawn_wide_key(a.sp.seed, env_hash, (unsigned)lane, (unsigned)r);
    }, x, y, z);
    if (lane == 0) {
        if (round >= a.sp.max_rounds && failed) atomicAdd(failed, 1u);
        episode[e] = ep; env_steps[e] = 0; done_out[e] = 1;
    }
    const unsigned s = e * (unsigned)N + (unsigned)lane;
    if (lane < N) {
        float* st = b.state + s;
        st[0] = x; st[(size_t)S] = y; st[2 * (size_t)S] = z;
        const float yaw = a.sp.yaw_lo + (a.sp.yaw_hi - a.sp.yaw_lo) * u01(spawn_wide_key(a.sp.seed, env_hash, (unsigned)lane, 0xFFFFFFFFu));
        spawn_write_rest(st, S, yaw);
        autoreset_write_X(c, b, a, S, s, x, y, z, yaw);
    }
    if (!b.A_tape) return;
    const unsigned NN = (unsigned)(N * N);
    const size_t slot_elems = (size_t)S * (size_t)N;
    float* A0 = b.A_tape + (size_t)a.slot_a * slot_elems + (size_t)e * NN;
    for (unsigned base = 0; base < NN; base += 32) {          // whole warp: the shuffles need every lane
        const unsigned idx = base + (unsigned)lane;
        const int i = idx < NN ? (int)(idx / (unsigned)N) : 0, j = idx < NN ? (int)(idx % (unsigned)N) : 0;
        const float xi = __shfl_sync(kFull32, x, i), yi = __shfl_sync(kFull32, y, i), zi = __shfl_sync(kFull32, z, i);
        const float xj = __shfl_sync(kFull32, x, j), yj = __shfl_sync(kFull32, y, j), zj = __shfl_sync(kFull32, z, j);
        if (idx < NN) A0[idx] = autoreset_adjacency(a, i, j, xi, yi, zi, xj, yj, zj);
    }
    for (int k = 1; k <= c.K; ++k) {
        float* Ak = b.A_tape + (size_t)((a.slot_a + k) % c.L) * slot_elems + (size_t)e * NN;
        for (unsigned idx = lane; idx < NN; idx += 32) Ak[idx] = 0.f;
    }
}

// N > 32: a CTA per env, the rounds of spawn_wide_kernel; dynamic shared memory = its two masks
__global__ void __launch_bounds__(1024)
autoreset_wide_kernel(const __grid_constant__ MrsConfig c, const MrsBuffers b, const AutoResetArgs a,
                      const unsigned char* __restrict__ done_in, int* __restrict__ env_steps, unsigned* __restrict__ episode,
                      unsigned char* __restrict__ done_out, unsigned* __restrict__ failed) {
    extern __shared__ unsigned spawn_bits[];
    const unsigned e = blockIdx.x;
    const int n = env_steps[e];
    const bool done = autoreset_done(a, done_in, e, n);
    const unsigned ep = episode[e] + 1u;
    __syncthreads();                       // every thread has read the counters before thread 0 rewrites them
    if (!done) {
        if (threadIdx.x == 0) { env_steps[e] = n + 1; done_out[e] = 0; }
        return;
    }
    const int N = c.N;
    const size_t S = (size_t)c.E * (size_t)N;
    float* st = b.state + (size_t)e * N;
    const float lim2 = 4.f * c.phys.agent_radius * c.phys.agent_radius;
    const unsigned long long env_hash = autoreset_env_hash(a.sp.env_offset + e, ep);
    const int round = spawn_cta_rounds(a.sp, N, lim2, env_hash, spawn_bits, st, st + S, st + 2 * S);
    if (threadIdx.x == 0) {
        if (round >= a.sp.max_rounds && failed) atomicAdd(failed, 1u);
        episode[e] = ep; env_steps[e] = 0; done_out[e] = 1;
    }
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        const float yaw = a.sp.yaw_lo + (a.sp.yaw_hi - a.sp.yaw_lo) * u01(spawn_wide_key(a.sp.seed, env_hash, (unsigned)i, 0xFFFFFFFFu));
        spawn_write_rest(st + i, S, yaw);
        autoreset_write_X(c, b, a, (unsigned)S, e * (unsigned)N + (unsigned)i, st[i], st[S + i], st[2 * S + i], yaw);
    }
    if (!b.A_tape) return;
    const size_t NN = (size_t)N * N;
    const size_t slot_elems = S * (size_t)N;
    float* A0 = b.A_tape + (size_t)a.slot_a * slot_elems + (size_t)e * NN;
    for (size_t idx = threadIdx.x; idx < NN; idx += blockDim.x) {     // positions: this CTA's writes, before the last barrier
        const int i = (int)(idx / (unsigned)N), j = (int)(idx % (unsigned)N);
        A0[idx] = autoreset_adjacency(a, i, j, st[i], st[S + i], st[2 * S + i], st[j], st[S + j], st[2 * S + j]);
    }
    for (int k = 1; k <= c.K; ++k) {
        float* Ak = b.A_tape + (size_t)((a.slot_a + k) % c.L) * slot_elems + (size_t)e * NN;
        for (size_t idx = threadIdx.x; idx < NN; idx += blockDim.x) Ak[idx] = 0.f;
    }
}

// ------------------------------------------------------------------------------ sensors (row f4)
// Analytic sensors of the 'simple' world (ground box top at ground_z, agents as CONTACT_RADIUS
// spheres -- the same contact geometry as the step; AGENT_RADIUS is only the spawn separation).  One thread per agent (proximity) or per
// (agent, ray) (raycast); partners are walked from the L1/L2-resident position planes.
// Object.collision / get_dist / get_contact_points / raycast (Object.py:100-174) on these primitives.
__global__ void __launch_bounds__(128)
proximity_kernel(const __grid_constant__ MrsConfig c, const MrsBuffers b, float thresh, float* __restrict__ gap_agent,
                 int* __restrict__ nearest, float* __restrict__ gap_ground, unsigned char* __restrict__ collision) {
    const unsigned S = (unsigned)c.E * (unsigned)c.N;
    const unsigned s = blockIdx.x * 128u + threadIdx.x;
    if (s >= S) return;
    const int N = c.N;
    const unsigned env0 = (s / (unsigned)N) * (unsigned)N;
    const int ai = (int)(s - env0);
    const float* px = b.state + env0;
    const float* py = b.state + (size_t)S + env0;
    const float* pz = b.state + 2 * (size_t)S + env0;
    const float x = px[ai], y = py[ai], z = pz[ai];
    float best = INFINITY;
    int arg = -1;
    for (int j = 0; j < N; ++j) {
        if (j == ai) continue;
        const float dx = x - px[j], dy = y - py[j], dz = z - pz[j];
        const float d2 = dx * dx + dy * dy + dz * dz;
        if (d2 < best) { best = d2; arg = j; }
    }
    const float ga = sqrtf(best) - 2.f * c.phys.contact_radius;
    // ground: same support extent of the collision cylinder as the contact row of the step
    const float qx = b.state[3 * (size_t)S + s], qy = b.state[4 * (size_t)S + s];
    const float R22 = 1.f - 2.f * (qx * qx + qy * qy);
    const float ext = c.phys.col_radius * sqrtf(fmaxf(1.f - R22 * R22, 0.f)) + c.phys.col_halfheight * fabsf(R22) +
                      c.phys.col_margin;
    const float gg = z - ext - c.phys.ground_z;
    if (gap_agent) gap_agent[s] = ga;
    if (nearest) nearest[s] = arg;
    if (gap_ground) gap_ground[s] = gg;
    if (collision) collision[s] = (ga < thresh || gg < thresh) ? 1 : 0;
}

// rays: [R][3] directions in the body frame (body != 0) or world frame, start = pos + R * offset;
// hit_dist [S][R] (inf = no hit within range), hit_id [S][R]: -1 none, N = ground, j = agent j
__global__ void __launch_bounds__(128)
raycast_kernel(const __grid_constant__ MrsConfig c, const MrsBuffers b, const float* __restrict__ dirs, int nrays, float ox,
               float oy, float oz, int body, float range, float* __restrict__ hit_dist, int* __restrict__ hit_id) {
    const unsigned S = (unsigned)c.E * (unsigned)c.N;
    const unsigned tid = blockIdx.x * 128u + threadIdx.x;
    if (tid >= S * (unsigned)nrays) return;
    const unsigned s = tid / (unsigned)nrays;
    const int r = (int)(tid - s * (unsigned)nrays);
    const int N = c.N;
    const unsigned env0 = (s / (unsigned)N) * (unsigned)N;
    const int ai = (int)(s - env0);
    Agent st;
    load_agent(b.state, S, s, st);
    float Rm[9];
    quat_to_mat(st, Rm);
    float dx = dirs[3 * r], dy = dirs[3 * r + 1], dz = dirs[3 * r + 2];
    float sx = ox, sy = oy, sz = oz;
    if (body) {
        const float tx = Rm[0] * dx + Rm[1] * dy + Rm[2] * dz, ty = Rm[3] * dx + Rm[4] * dy + Rm[5] * dz,
                    tz = Rm[6] * dx + Rm[7] * dy + Rm[8] * dz;
        dx = tx; dy = ty; dz = tz;
        const float ux = Rm[0] * ox + Rm[1] * oy + Rm[2] * oz, uy = Rm[3] * ox + Rm[4] * oy + Rm[5] * oz,
                    uz = Rm[6] * ox + Rm[7] * oy + Rm[8] * oz;
        sx = ux; sy = uy; sz = uz;
    }
    const float inv = rsqrtf(dx * dx + dy * dy + dz * dz);
    dx *= inv; dy *= inv; dz *= inv;
    sx += st.px; sy += st.py; sz += st.pz;
    float best = range;
    int id = -1;
    // ground: top face of the 30 x 30 x 1 box centred at the origin (plane.urdf:21-26)
    if (dz < 0.f && sz > c.phys.ground_z) {
        const float t = (c.phys.ground_z - sz) / dz;
        const float hx = sx + t * dx, hy = sy + t * dy;
        if (t < best && fabsf(hx) <= 15.f && fabsf(hy) <= 15.f) { best = t; id = N; }
    }
    const float* px = b.state + env0;
    const float* py = b.state + (size_t)S + env0;
    const float* pz = b.state + 2 * (size_t)S + env0;
    const float rad2 = c.phys.contact_radius * c.phys.contact_radius;
    for (int j = 0; j < N; ++j) {
        if (j == ai) continue;
        const float cx = px[j] - sx, cy = py[j] - sy, cz = pz[j] - sz;
        const float tc = cx * dx + cy * dy + cz * dz;                  // closest approach along the ray
        const float d2 = cx * cx + cy * cy + cz * cz - tc * tc;
        if (d2 > rad2) continue;
        const float t = tc - sqrtf(rad2 - d2);
        if (t >= 0.f && t < best) { best = t; id = j; }
    }
    hit_dist[tid] = (id >= 0) ? best : INFINITY;
    hit_id[tid] = id;
}

// tape maintenance: 128-bit grid-stride copy / zero fill (slot sizes are multiples of 4 floats
// whenever E*N is; scalar tail otherwise)
__global__ void __launch_bounds__(256)
tape_fill_kernel(float* __restrict__ dst, const float* __restrict__ src, size_t slot_elems, int count) {
    const size_t total = slot_elems * (size_t)count;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    if ((slot_elems & 3) == 0) {
        const size_t n4 = total >> 2, s4 = slot_elems >> 2;
        float4* d4 = reinterpret_cast<float4*>(dst);
        const float4* r4 = reinterpret_cast<const float4*>(src);
        for (size_t i = tid; i < n4; i += stride) d4[i] = src ? r4[i % s4] : make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
        for (size_t i = tid; i < total; i += stride) dst[i] = src ? src[i % slot_elems] : 0.f;
    }
}

// ------------------------------------------------------------------------------ wide path: contact + post
// contact_env_kernel: one CTA per env around contact_env_body (mrs_contact_env.cuh)
__global__ void __launch_bounds__(1024)
contact_env_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    pdl_enter();
    contact_env_body(c, d, b, blockIdx.x, smem_raw);
}

// post pass of the wide path, one thread per agent: ground-only contact solve (agents flagged for agent-agent
// contact were solved by contact_env_kernel), position / attitude integration, state store, newest X slice
__global__ void __launch_bounds__(kBlock)
step_post_kernel(const __grid_constant__ MrsConfig c, const __grid_constant__ Derived d, const MrsBuffers b, int slot) {
    pdl_enter();
    const unsigned S = (unsigned)c.E * (unsigned)c.N;
    const unsigned gid = blockIdx.x * kBlock + threadIdx.x;
    const bool valid = gid < S;
    const unsigned s = valid ? gid : 0u;
    const MrsPhysicsParams& ph = c.phys;
    const float* __restrict__ sc = b.scratch;
    unsigned gnd = 0, bad = 0;
    if (valid) {
        Agent st;
        st.px = sc[3 * (size_t)S + s]; st.py = sc[4 * (size_t)S + s]; st.pz = sc[5 * (size_t)S + s];
        st.vx = sc[0 * (size_t)S + s]; st.vy = sc[1 * (size_t)S + s]; st.vz = sc[2 * (size_t)S + s];
        const bool solved = sc[6 * (size_t)S + s] != 0.f;
        st.qx = b.state[3 * (size_t)S + s]; st.qy = b.state[4 * (size_t)S + s]; st.qz = b.state[5 * (size_t)S + s];
        st.qw = b.state[6 * (size_t)S + s];
        st.wx = b.state[10 * (size_t)S + s]; st.wy = b.state[11 * (size_t)S + s]; st.wz = b.state[12 * (size_t)S + s];
        if (ph.ground_contact && !solved && st.pz < d.gnd_skip_z) {
            float R[9];
            quat_to_mat(st, R);
            if (ground_solve(make_contact_params(ph, d), st, R)) gnd = 1;
        }
        integrate(c, d, st);
        store_agent(b.state, S, s, st);
        if (b.X_tape && c.state_layout != MRS_X_NONE)
            write_X(b.X_tape + (size_t)slot * S * state_dim(c.state_layout), c.state_layout, s, st);
        bad = agent_finite(st) ? 0u : 1u;
    }
    // statistics: one warp reduction, then at most two global atomics per warp (not per agent)
    const unsigned w_gnd = __reduce_add_sync(kFull32, gnd);
    const unsigned w_bad = __reduce_add_sync(kFull32, bad);
    if ((threadIdx.x & 31) == 0) {
        if (w_bad && b.status) atomicOr(b.status, MRS_STATUS_NONFINITE);
        if (b.stats) {
            if (w_gnd) atomicAdd(b.stats + MRS_STAT_GROUND_CONTACTS, (unsigned long long)w_gnd);
            if (w_bad) atomicAdd(b.stats + MRS_STAT_NONFINITE, (unsigned long long)w_bad);
        }
    }
}

// launches contact_env_kernel (one CTA per env) when agent-agent contact is enabled
int launch_contact_env(const MrsConfig& c, const Derived& d, const MrsBuffers& b, bool pdl, cudaStream_t st) {
    if (!c.phys.agent_contact || c.N < 2) return MRS_OK;
    int threads = (c.N + 31) / 32 * 32;
    if (threads > 1024) threads = 1024;
    const size_t smem = contact_env_smem(threads, c.N);
    // the round mask grows with N: raise the kernel's dynamic shared-memory limit to the largest size asked for
    static size_t configured[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return MRS_ERR_CUDA;
    if (smem > configured[dev]) {
        if (cudaFuncSetAttribute(contact_env_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return MRS_ERR_CUDA;
        configured[dev] = smem;
    }
    return launch_pdl(pdl, contact_env_kernel, dim3((unsigned)c.E), (unsigned)threads, smem, st, c, d, b);
}

int launch_step_post(const MrsConfig& c, const Derived& d, const MrsBuffers& b, int slot, bool pdl, cudaStream_t st) {
    const size_t S = (size_t)c.E * c.N;
    return launch_pdl(pdl, step_post_kernel, dim3((unsigned)((S + kBlock - 1) / kBlock)), kBlock, 0, st, c, d, b, slot);
}

// ------------------------------------------------------------------------------ host side
int launch_adjacency(const float* pos, size_t cs, size_t as, float* A, int E, int N, float s_max, int comm_inf,
                            cudaStream_t st) {
    if (N >= 128 && (N & 3) == 0) {
        const int col_tiles = (N + 4 * kBlock - 1) / (4 * kBlock);
        const int row_tiles = (N + kRowTile - 1) / kRowTile;
        dim3 grid((unsigned)(col_tiles * row_tiles), (unsigned)E);
        adjacency_tiled_kernel<<<grid, kBlock, 0, st>>>(pos, cs, as, A, E, N, s_max, comm_inf);
    } else if (N > 32 && (N & 3) == 0 && (size_t)E * N * (N / 4) < 0x7fffffffull * (size_t)kBlock) {
        const size_t nquads = (size_t)E * N * (N / 4);
        adjacency_quad_kernel<<<(unsigned)((nquads + kBlock - 1) / kBlock), kBlock, 0, st>>>(pos, cs, as, A, E, N, s_max,
                                                                                             comm_inf);
    } else {
        const size_t total = (size_t)E * N * N;
        const size_t blocks = (total + 255) / 256;
        const size_t cap = (size_t)(sm_count() > 0 ? sm_count() : 148) * 32;
        adjacency_flat_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(pos, cs, as, A, E, N, s_max,
                                                                                        comm_inf);
    }
    return last_error();
}

// Side stream of the wide path: the adjacency kernel of step t (a pure streaming store that only
// reads the new positions) runs next to the compute-bound pair kernel of step t+1; it has to be done
// before post(t+1) overwrites the positions.  Fork / join through events, so it is capturable.
// One lane per device, created once under a lock.  The lane's events are re-recorded by every call that uses it,
// so the calls that do (mrs_step_many / mrs_rollout with N > 32, mrs_rollout_host) must not run concurrently on one
// device from several host threads or caller streams (header: one host thread per GPU).
static SideLane g_side[64];
static std::mutex g_lane_mutex;
SideLane* side_lane() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lock(g_lane_mutex);
    SideLane& L = g_side[dev];
    if (!L.ok) {
        SideLane fresh;
        if (cudaStreamCreateWithFlags(&fresh.s, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
        if (cudaEventCreateWithFlags(&fresh.posted, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&fresh.adj_done, cudaEventDisableTiming) != cudaSuccess) {
            if (fresh.posted) cudaEventDestroy(fresh.posted);
            cudaStreamDestroy(fresh.s);
            (void)cudaGetLastError();
            return nullptr;
        }
        fresh.ok = true;
        L = fresh;
    }
    return &L;
}

#ifdef MRS_DEV_ONLY_MODE
extern template int dispatch_step<MRS_DEV_ONLY_MODE>(const MrsConfig&, const MrsBuffers&, StepArgs, cudaStream_t);
#else
extern template int dispatch_step<MRS_SET_TARGET_VEL>(const MrsConfig&, const MrsBuffers&, StepArgs, cudaStream_t);
extern template int dispatch_step<MRS_SET_TARGET_POS>(const MrsConfig&, const MrsBuffers&, StepArgs, cudaStream_t);
extern template int dispatch_step<MRS_SET_TARGET_ACCEL>(const MrsConfig&, const MrsBuffers&, StepArgs, cudaStream_t);
extern template int dispatch_step<MRS_SET_FORCE>(const MrsConfig&, const MrsBuffers&, StepArgs, cudaStream_t);
extern template int dispatch_step<MRS_SET_TARGET_ORI>(const MrsConfig&, const MrsBuffers&, StepArgs, cudaStream_t);
extern template int dispatch_step<MRS_SET_CONTROL>(const MrsConfig&, const MrsBuffers&, StepArgs, cudaStream_t);
extern template int dispatch_step<MRS_SET_SPEEDS>(const MrsConfig&, const MrsBuffers&, StepArgs, cudaStream_t);
extern template int dispatch_step<MRS_NO_ACTION>(const MrsConfig&, const MrsBuffers&, StepArgs, cudaStream_t);
#endif

static int step_impl(const MrsConfig* cfg, const MrsBuffers* bufs, const float* actions, int T, int slot_x, int slot_a,
                     void* stream, int role = 0, int seq = 0) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!bufs || !bufs->state || !bufs->ctrl) return MRS_ERR_ARG;
    if (T <= 0) return MRS_ERR_ARG;
    if (cfg->action_type != MRS_NO_ACTION && !actions) return MRS_ERR_ARG;
    if (bufs->X_tape && cfg->state_layout != MRS_X_NONE && (slot_x >= cfg->L || slot_x - (T - 1) < 0)) return MRS_ERR_ARG;
    if (bufs->A_tape && (slot_a >= cfg->L || slot_a - (T - 1) < 0)) return MRS_ERR_ARG;
    StepArgs a;
    a.actions = actions;
    a.T = T;
    a.slot_x = slot_x;
    a.slot_a = slot_a;
    a.G = 0;
    a.role = role;
    a.seq = seq;
    a.slow_slots = 0;
    a.chunk_lo = 0;
    a.nchunks = 0;
    a.X0 = a.A0 = nullptr;
    a.xstride = a.astride = 0;
    if ((unsigned long long)cfg->E * cfg->N * (cfg->N > 18 ? cfg->N : 18) >= 0xffffffffull) return MRS_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
#ifdef MRS_DEV_ONLY_MODE     // development builds: one action mode only (compile time / 8)
    if (cfg->action_type != MRS_DEV_ONLY_MODE) return MRS_ERR_UNSUPPORTED;
    return dispatch_step<MRS_DEV_ONLY_MODE>(*cfg, *bufs, a, st);
#else
    switch (cfg->action_type) {
        case MRS_SET_TARGET_VEL:   return dispatch_step<MRS_SET_TARGET_VEL>(*cfg, *bufs, a, st);
        case MRS_SET_TARGET_POS:   return dispatch_step<MRS_SET_TARGET_POS>(*cfg, *bufs, a, st);
        case MRS_SET_TARGET_ACCEL: return dispatch_step<MRS_SET_TARGET_ACCEL>(*cfg, *bufs, a, st);
        case MRS_SET_FORCE:        return dispatch_step<MRS_SET_FORCE>(*cfg, *bufs, a, st);
        case MRS_SET_TARGET_ORI:   return dispatch_step<MRS_SET_TARGET_ORI>(*cfg, *bufs, a, st);
        case MRS_SET_CONTROL:      return dispatch_step<MRS_SET_CONTROL>(*cfg, *bufs, a, st);
        case MRS_SET_SPEEDS:       return dispatch_step<MRS_SET_SPEEDS>(*cfg, *bufs, a, st);
        case MRS_NO_ACTION:        return dispatch_step<MRS_NO_ACTION>(*cfg, *bufs, a, st);
    }
    return MRS_ERR_ARG;
#endif
}

}  // namespace mrs

// ================================================================================ C ABI
using namespace mrs;

extern "C" {

int mrs_abi_version(void) { return MRS_ABI_VERSION; }

const char* mrs_strerror(int err) {
    switch (err) {
        case MRS_OK: return "ok";
        case MRS_ERR_ARG: return "invalid argument";
        case MRS_ERR_CUDA: return "CUDA error (no device, bad launch or asynchronous fault)";
        case MRS_ERR_UNSUPPORTED: return "unsupported configuration";
    }
    return "unknown error";
}

int mrs_action_dim(int action_type) {
    switch (action_type) {
        case MRS_SET_TARGET_VEL: case MRS_SET_TARGET_POS: case MRS_SET_TARGET_ACCEL: case MRS_SET_FORCE:
        case MRS_SET_TARGET_ORI: return 3;
        case MRS_SET_CONTROL: case MRS_SET_SPEEDS: return 4;
    }
    return 0;
}

int mrs_state_dim(int state_layout) { return state_dim(state_layout); }

int mrs_scratch_planes(int E, int N) {
    if (N <= 32 || E <= 0) return 0;
    if (N <= 128) return MRS_SCRATCH_PLANES;
    int jw = 0, nsplit = 0;
    pair_split(E, N, &jw, &nsplit);
    return MRS_SCRATCH_PLANES + 2 * nsplit;
}

size_t mrs_sizeof_config(void) { return sizeof(MrsConfig); }
size_t mrs_sizeof_buffers(void) { return sizeof(MrsBuffers); }

int mrs_default_config(MrsConfig* cfg) {
    if (!cfg) return MRS_ERR_ARG;
    memset(cfg, 0, sizeof(*cfg));
    cfg->E = 1; cfg->N = 1; cfg->K = 0; cfg->L = 1;
    cfg->action_type = MRS_SET_TARGET_VEL;
    cfg->state_layout = MRS_X_POS_VEL;
    cfg->dt = 0.01f;
    cfg->gravity = 9.81f;
    cfg->comm_range = INFINITY;
    MrsQuadParams& q = cfg->quad;
    // cf2x.urdf:5,11-12 and prop link CoM offsets :42,54,66,78
    q.mass = 0.027f; q.ixx = 1.4e-5f; q.iyy = 1.4e-5f; q.izz = 2.17e-5f;
    q.kf = 3.16e-10f; q.km = 7.94e-12f; q.arm = 0.0397f;
    q.gnd_eff_coeff = 11.36859f; q.prop_radius = 2.31348e-2f;
    q.drag_xy = 9.1785e-7f; q.drag_z = 10.311e-7f;
    q.dw1 = 2267.18f; q.dw2 = 0.16f; q.dw3 = -0.11f;
    const float px[4] = {0.028f, -0.028f, -0.028f, 0.028f}, py[4] = {0.028f, 0.028f, -0.028f, -0.028f};
    for (int i = 0; i < 4; ++i) { q.prop_x[i] = px[i]; q.prop_y[i] = py[i]; }
    // Quadcopter.calculate_parameters (Quadcopter.py:153-168), in double then rounded
    {
        const double g = 9.81 * 0.027, kf = 3.16e-10, t2w = 2.25, coeff = 11.36859, pr = 2.31348e-2;
        const double max_rpm = sqrt(t2w * g / (4 * kf));
        const double max_thrust = 4.0 * kf * max_rpm * max_rpm;
        q.gnd_hclip = (float)(0.25 * pr * sqrt((15.0 * max_rpm * max_rpm * kf * coeff) / max_thrust));
    }
    // QuadControl gains (QuadControl.py:14-32)
    q.pos_p = 1.5f; q.pos_i = 0.001f; q.pos_d = 1.0f;
    q.vel_p = 3.0f; q.vel_i = 0.1f; q.vel_d = 1.0f;
    const float op[3] = {70000.f, 70000.f, 60000.f}, oi[3] = {0.f, 0.f, 500.f}, od[3] = {20000.f, 20000.f, 12000.f};
    for (int i = 0; i < 3; ++i) { q.ori_p[i] = op[i]; q.ori_i[i] = oi[i]; q.ori_d[i] = od[i]; }
    q.min_pwm = 20000.f; q.max_pwm = 65535.f; q.pwm2rpm_a = 0.2685f; q.pwm2rpm_b = 4070.3f;
    q.ctrl_dt = 0.01f; q.ctrl_gravity = 9.81f;
    // 'x' mixer (Quadcopter.py:164) and its inverse; orthogonal rows => Ainv = A^T D^-1
    const double r2 = 1.0 / sqrt(2.0);
    const double A[4][4] = {{1, 1, 1, 1}, {r2, r2, -r2, -r2}, {-r2, r2, r2, -r2}, {-1, 1, -1, 1}};
    const double rown[4] = {4.0, 2.0, 2.0, 4.0};
    for (int r = 0; r < 4; ++r)
        for (int cidx = 0; cidx < 4; ++cidx) {
            q.mix_a[r * 4 + cidx] = (float)A[r][cidx];
            q.mix_ainv[cidx * 4 + r] = (float)(A[r][cidx] / rown[r]);
        }
    // least-squares solve matrices of the 16 active sets: P_S = (A_S^T A_S)^-1 A_S^T (4x4, zero rows off S)
    for (int m = 0; m < 16; ++m) {
        int cols[4], nc = 0;
        for (int cidx = 0; cidx < 4; ++cidx) if ((m >> cidx) & 1) cols[nc++] = cidx;
        double Gm[4][8];
        for (int i = 0; i < nc; ++i) {
            for (int j = 0; j < nc; ++j) {
                double acc = 0;
                for (int r = 0; r < 4; ++r) acc += A[r][cols[i]] * A[r][cols[j]];
                Gm[i][j] = acc;
            }
            for (int j = 0; j < nc; ++j) Gm[i][nc + j] = (i == j) ? 1.0 : 0.0;
        }
        for (int p = 0; p < nc; ++p) {   // Gauss-Jordan, SPD Gram matrix
            int best = p;
            for (int r = p + 1; r < nc; ++r) if (fabs(Gm[r][p]) > fabs(Gm[best][p])) best = r;
            if (best != p) for (int j = 0; j < 2 * nc; ++j) { double tmp = Gm[p][j]; Gm[p][j] = Gm[best][j]; Gm[best][j] = tmp; }
            const double piv = Gm[p][p];
            for (int j = 0; j < 2 * nc; ++j) Gm[p][j] /= piv;
            for (int r = 0; r < nc; ++r) if (r != p) {
                const double f = Gm[r][p];
                for (int j = 0; j < 2 * nc; ++j) Gm[r][j] -= f * Gm[p][j];
            }
        }
        for (int i = 0; i < nc; ++i)
            for (int r = 0; r < 4; ++r) {
                double acc = 0;
                for (int j = 0; j < nc; ++j) acc += Gm[i][nc + j] * A[r][cols[j]];
                q.nnls_tab[m * 16 + cols[i] * 4 + r] = (float)acc;
            }
    }
    MrsPhysicsParams& p = cfg->phys;   // oracle/bullet_model.py PhysicsParams
    p.mass = 0.027f;
    {
        const double hx = 0.06 + 3 * 0.001, hz = 0.0125 + 3 * 0.001, lx = 2 * hx, lz = 2 * hz, m = 0.027;
        p.inertia[0] = p.inertia[1] = (float)(m / 12.0 * (lx * lx + lz * lz));
        p.inertia[2] = (float)(m / 12.0 * (lx * lx + lx * lx));
    }
    p.lin_damping = 0.04f; p.ang_damping = 0.04f; p.max_coord_vel = 100.f; p.gyro = 1;
    p.ang_motion_threshold = 0.78539816339744830962f;
    p.erp2 = 0.08f; p.slop = 1e-5f; p.contact_margin = 0.02f;
    p.mu_ground = 0.75f; p.ground_z = 0.5f;
    p.col_radius = 0.06f; p.col_halfheight = 0.0125f; p.col_margin = 0.001f;
    p.ground_contact = 1; p.agent_contact = 1;
    p.agent_radius = 0.3f; p.contact_radius = 0.3f;
    p.mu_agent = 0.25f; p.solver_iters = 50; p.solver_tol = 1e-6f;
    return MRS_OK;
}

int mrs_config_is_baked(const MrsConfig* cfg) {
    if (check_cfg(cfg)) return 0;
    return config_is_baked(*cfg, make_derived(*cfg)) ? 1 : 0;
}

int mrs_debug_derived(const MrsConfig* cfg, void* out, size_t out_bytes) {
    if (!cfg || !out || out_bytes != sizeof(Derived)) return MRS_ERR_ARG;
    const Derived d = make_derived(*cfg);
    memcpy(out, &d, sizeof(Derived));
    return MRS_OK;
}

int mrs_step(const MrsConfig* cfg, const MrsBuffers* bufs, const float* actions, int slot_x, int slot_a, void* stream) {
    return step_impl(cfg, bufs, actions, 1, slot_x, slot_a, stream);
}

int mrs_step_many(const MrsConfig* cfg, const MrsBuffers* bufs, const float* actions, int T, int slot_x_first,
                  int slot_a_first, void* stream) {
    return step_impl(cfg, bufs, actions, T, slot_x_first, slot_a_first, stream);
}

int mrs_rollout(const MrsConfig* cfg, const MrsBuffers* bufs, const float* actions, int T, int slot_x_first,
                int slot_a_first, void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (T <= 0) return MRS_ERR_ARG;
    if (cfg->N > 32) return step_impl(cfg, bufs, actions, T, slot_x_first, slot_a_first, stream);   // per-step kernels anyway
    const size_t per_step = (size_t)cfg->E * cfg->N * (size_t)mrs_action_dim(cfg->action_type);
    constexpr int kMaxChain = 32768;         // the position travels in 16 bits of a queue entry
    for (int t = 0; t < T; ++t) {
        const int pos = t % kMaxChain;
        rc = step_impl(cfg, bufs, actions ? actions + (size_t)t * per_step : nullptr, 1, slot_x_first - t, slot_a_first - t,
                       stream, (bufs && bufs->sync) ? (pos == 0 ? 1 : 2) : 0, pos);
        if (rc) return rc;
    }
    return MRS_OK;
}

int mrs_observe(const MrsConfig* cfg, const MrsBuffers* bufs, int slot, int write_X, int write_A, void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!bufs || !bufs->state) return MRS_ERR_ARG;
    if (slot < 0 || slot >= cfg->L) return MRS_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t S = (size_t)cfg->E * cfg->N;
    if (write_X && cfg->state_layout != MRS_X_NONE) {
        if (!bufs->X_tape) return MRS_ERR_ARG;
        observe_x_kernel<<<(unsigned)((S + 255) / 256), 256, 0, st>>>(*bufs, S, cfg->state_layout, slot);
        if ((rc = last_error())) return rc;
    }
    if (write_A) {
        if (!bufs->A_tape) return MRS_ERR_ARG;
        const int comm_inf = isinf(cfg->comm_range) && cfg->comm_range > 0.f;
        rc = launch_adjacency(bufs->state, S, 1, bufs->A_tape + (size_t)slot * S * cfg->N, cfg->E, cfg->N,
                              adjacency_threshold(cfg->comm_range), comm_inf, st);
    }
    return rc;
}

int mrs_adjacency(const MrsConfig* cfg, const float* pos, float* A, void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!pos || !A) return MRS_ERR_ARG;
    const int comm_inf = isinf(cfg->comm_range) && cfg->comm_range > 0.f;
    return launch_adjacency(pos, 1, 3, A, cfg->E, cfg->N, adjacency_threshold(cfg->comm_range), comm_inf,
                            (cudaStream_t)stream);
}

int mrs_set_state(const MrsConfig* cfg, const MrsBuffers* bufs, const float* pos, const float* ori_euler,
                  const float* vel, const float* angvel, const unsigned char* env_mask, void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!bufs || !bufs->state) return MRS_ERR_ARG;
    const size_t S = (size_t)cfg->E * cfg->N;
    set_state_kernel<<<(unsigned)((S + 255) / 256), 256, 0, (cudaStream_t)stream>>>(bufs->state, S, cfg->N, pos,
                                                                                   ori_euler, vel, angvel, env_mask);
    return last_error();
}

int mrs_tape_fill(const MrsConfig* cfg, const MrsBuffers* bufs, int which, int src, int dst_first, int count,
                  void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!bufs || (which != 1 && which != 2)) return MRS_ERR_ARG;
    if (count <= 0) return count == 0 ? MRS_OK : MRS_ERR_ARG;
    if (dst_first < 0 || dst_first + count > cfg->L || src >= cfg->L) return MRS_ERR_ARG;
    if (src >= 0 && src >= dst_first && src < dst_first + count) return MRS_ERR_ARG;
    const size_t S = (size_t)cfg->E * cfg->N;
    float* tape = (which == 1) ? bufs->X_tape : bufs->A_tape;
    if (!tape) return MRS_ERR_ARG;
    const size_t slot_elems = (which == 1) ? S * (size_t)state_dim(cfg->state_layout) : S * (size_t)cfg->N;
    if (slot_elems == 0) return MRS_ERR_ARG;
    const size_t work = (slot_elems * count + 3) / 4;
    size_t blocks = (work + 255) / 256;
    const size_t cap = (size_t)(sm_count() > 0 ? sm_count() : 148) * 16;
    if (blocks > cap) blocks = cap;
    tape_fill_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        tape + (size_t)dst_first * slot_elems, src >= 0 ? tape + (size_t)src * slot_elems : nullptr, slot_elems, count);
    return last_error();
}

int mrs_pack_adjacency(const MrsConfig* cfg, const float* A, unsigned int* bits, void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!A || !bits) return MRS_ERR_ARG;
    return launch_pack_adjacency(A, bits, cfg->E, cfg->N, (cudaStream_t)stream);
}

int mrs_step_host(const MrsConfig* cfg, const MrsBuffers* bufs, const float* actions_host, float* dev_actions,
                  float* X_host, float* A_host, unsigned int* Abits_host, unsigned int* dev_Abits, int slot_x, int slot_a,
                  void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!bufs) return MRS_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t S = (size_t)cfg->E * cfg->N;
    const int adim = mrs_action_dim(cfg->action_type);
    if (adim > 0) {
        if (!actions_host || !dev_actions) return MRS_ERR_ARG;
        if (cudaMemcpyAsync(dev_actions, actions_host, S * adim * sizeof(float), cudaMemcpyHostToDevice, st) != cudaSuccess)
            return MRS_ERR_CUDA;
    }
    rc = step_impl(cfg, bufs, dev_actions, 1, slot_x, slot_a, stream);
    if (rc) return rc;
    const int D = state_dim(cfg->state_layout);
    if (X_host && bufs->X_tape && D > 0) {
        if (cudaMemcpyAsync(X_host, bufs->X_tape + (size_t)slot_x * S * D, S * D * sizeof(float), cudaMemcpyDeviceToHost,
                            st) != cudaSuccess)
            return MRS_ERR_CUDA;
    }
    if (A_host && bufs->A_tape) {
        if (cudaMemcpyAsync(A_host, bufs->A_tape + (size_t)slot_a * S * cfg->N, S * cfg->N * sizeof(float),
                            cudaMemcpyDeviceToHost, st) != cudaSuccess)
            return MRS_ERR_CUDA;
    }
    if (Abits_host && bufs->A_tape) {
        if (!dev_Abits) return MRS_ERR_ARG;
        rc = launch_pack_adjacency(bufs->A_tape + (size_t)slot_a * S * cfg->N, dev_Abits, cfg->E, cfg->N, st);
        if (rc) return rc;
        if (cudaMemcpyAsync(Abits_host, dev_Abits, S * ((cfg->N + 31) / 32) * sizeof(unsigned), cudaMemcpyDeviceToHost, st) !=
            cudaSuccess)
            return MRS_ERR_CUDA;
    }
    return cudaStreamSynchronize(st) == cudaSuccess ? MRS_OK : MRS_ERR_CUDA;
}


// Pipelined host rollout: three streams so that the H2D of step t+1's actions and the D2H of step
// t-1's X / A slices overlap the kernel of step t (PCIe is full duplex).  The compute stream is the
// caller's; the two copy streams and four events are created once per device and reused.
namespace {
struct CopyLanes {
    cudaStream_t h2d = nullptr, d2h = nullptr;
    cudaEvent_t up[2] = {nullptr, nullptr}, done[2] = {nullptr, nullptr}, packed[2] = {nullptr, nullptr}, tail = nullptr;
    bool ok = false;
};
CopyLanes g_lanes[64];
CopyLanes* copy_lanes() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lock(g_lane_mutex);
    CopyLanes& L = g_lanes[dev];
    if (!L.ok) {
        CopyLanes fresh;
        bool good = cudaStreamCreateWithFlags(&fresh.h2d, cudaStreamNonBlocking) == cudaSuccess &&
                    cudaStreamCreateWithFlags(&fresh.d2h, cudaStreamNonBlocking) == cudaSuccess;
        for (int i = 0; i < 2 && good; ++i)
            good = cudaEventCreateWithFlags(&fresh.up[i], cudaEventDisableTiming) == cudaSuccess &&
                   cudaEventCreateWithFlags(&fresh.done[i], cudaEventDisableTiming) == cudaSuccess &&
                   cudaEventCreateWithFlags(&fresh.packed[i], cudaEventDisableTiming) == cudaSuccess;
        good = good && cudaEventCreateWithFlags(&fresh.tail, cudaEventDisableTiming) == cudaSuccess;
        if (!good) {                      // release whatever was created: the next call starts from scratch
            if (fresh.h2d) cudaStreamDestroy(fresh.h2d);
            if (fresh.d2h) cudaStreamDestroy(fresh.d2h);
            for (int i = 0; i < 2; ++i) {
                if (fresh.up[i]) cudaEventDestroy(fresh.up[i]);
                if (fresh.done[i]) cudaEventDestroy(fresh.done[i]);
                if (fresh.packed[i]) cudaEventDestroy(fresh.packed[i]);
            }
            if (fresh.tail) cudaEventDestroy(fresh.tail);
            (void)cudaGetLastError();
            return nullptr;
        }
        fresh.ok = true;
        L = fresh;
    }
    return &L;
}
}  // namespace

int mrs_rollout_host(const MrsConfig* cfg, const MrsBuffers* bufs, const float* actions_host, float* dev_actions,
                     float* X_host, float* A_host, unsigned int* Abits_host, unsigned int* dev_Abits, int T,
                     int slot_x_first, int slot_a_first, void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!bufs || T <= 0) return MRS_ERR_ARG;
    const int adim = mrs_action_dim(cfg->action_type);
    if (adim <= 0 || !actions_host || !dev_actions) return MRS_ERR_ARG;
    CopyLanes* L = copy_lanes();
    if (!L) return MRS_ERR_CUDA;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t S = (size_t)cfg->E * cfg->N;
    const size_t abytes = S * adim * sizeof(float);
    const int D = mrs_state_dim(cfg->state_layout);
    const size_t xelems = S * (size_t)D, aelems = S * (size_t)cfg->N, belems = S * (size_t)((cfg->N + 31) / 32);
    if (Abits_host && !dev_Abits) return MRS_ERR_ARG;
    // the copy lanes start after whatever the caller already queued on the compute stream
    if (cudaEventRecord(L->tail, st) != cudaSuccess) return MRS_ERR_CUDA;
    if (cudaStreamWaitEvent(L->h2d, L->tail, 0) != cudaSuccess) return MRS_ERR_CUDA;
    if (cudaStreamWaitEvent(L->d2h, L->tail, 0) != cudaSuccess) return MRS_ERR_CUDA;
    for (int t = 0; t < T; ++t) {
        const int bsel = t & 1;
        float* da = dev_actions + (size_t)bsel * S * adim;
        if (t >= 2 && cudaStreamWaitEvent(L->h2d, L->done[bsel], 0) != cudaSuccess) return MRS_ERR_CUDA;
        if (cudaMemcpyAsync(da, actions_host + (size_t)t * S * adim, abytes, cudaMemcpyHostToDevice, L->h2d) != cudaSuccess)
            return MRS_ERR_CUDA;
        if (cudaEventRecord(L->up[bsel], L->h2d) != cudaSuccess) return MRS_ERR_CUDA;
        if (cudaStreamWaitEvent(st, L->up[bsel], 0) != cudaSuccess) return MRS_ERR_CUDA;
        rc = step_impl(cfg, bufs, da, 1, slot_x_first - t, slot_a_first - t, stream);
        if (rc) return rc;
        if (cudaEventRecord(L->done[bsel], st) != cudaSuccess) return MRS_ERR_CUDA;
        if (Abits_host && bufs->A_tape) {
            // pack the newest A slice on the compute stream into staging half `bsel`, once the D2H copy of step
            // t - 2 out of that half is through (packed[bsel]); done[bsel] is recorded again behind the pack kernel
            if (t >= 2 && cudaStreamWaitEvent(st, L->packed[bsel], 0) != cudaSuccess) return MRS_ERR_CUDA;
            rc = launch_pack_adjacency(bufs->A_tape + (size_t)(slot_a_first - t) * aelems, dev_Abits + (size_t)bsel * belems, cfg->E,
                                       cfg->N, st);
            if (rc) return rc;
            if (cudaEventRecord(L->done[bsel], st) != cudaSuccess) return MRS_ERR_CUDA;
        }
        if ((X_host && bufs->X_tape && D > 0) || (A_host && bufs->A_tape) || (Abits_host && bufs->A_tape)) {
            if (cudaStreamWaitEvent(L->d2h, L->done[bsel], 0) != cudaSuccess) return MRS_ERR_CUDA;
            if (X_host && bufs->X_tape && D > 0 &&
                cudaMemcpyAsync(X_host + (size_t)t * xelems, bufs->X_tape + (size_t)(slot_x_first - t) * xelems,
                                xelems * sizeof(float), cudaMemcpyDeviceToHost, L->d2h) != cudaSuccess)
                return MRS_ERR_CUDA;
            if (A_host && bufs->A_tape &&
                cudaMemcpyAsync(A_host + (size_t)t * aelems, bufs->A_tape + (size_t)(slot_a_first - t) * aelems,
                                aelems * sizeof(float), cudaMemcpyDeviceToHost, L->d2h) != cudaSuccess)
                return MRS_ERR_CUDA;
            if (Abits_host && bufs->A_tape) {
                if (cudaMemcpyAsync(Abits_host + (size_t)t * belems, dev_Abits + (size_t)bsel * belems, belems * sizeof(unsigned),
                                    cudaMemcpyDeviceToHost, L->d2h) != cudaSuccess)
                    return MRS_ERR_CUDA;
                if (cudaEventRecord(L->packed[bsel], L->d2h) != cudaSuccess) return MRS_ERR_CUDA;
            }
        }
    }
    // join: the caller's stream continues only after the last copies
    if (cudaEventRecord(L->tail, L->d2h) != cudaSuccess) return MRS_ERR_CUDA;
    if (cudaStreamWaitEvent(st, L->tail, 0) != cudaSuccess) return MRS_ERR_CUDA;
    return cudaStreamSynchronize(st) == cudaSuccess ? MRS_OK : MRS_ERR_CUDA;
}


int mrs_spawn(const MrsConfig* cfg, const MrsBuffers* bufs, const unsigned char* env_mask, unsigned long long seed,
              unsigned long long env_offset, float z_lo, float z_hi, float xy_radius, float xy_sigma, float yaw_lo, float yaw_hi, int max_rounds,
              unsigned int* failed_envs, void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!bufs || !bufs->state) return MRS_ERR_ARG;
    if (!(z_hi >= z_lo) || !(xy_radius > 0.f) || !(xy_sigma > 0.f) || max_rounds <= 0) return MRS_ERR_ARG;
    if ((size_t)cfg->E * (size_t)cfg->N > 0xffffffffull) return MRS_ERR_UNSUPPORTED;     // u32 slot indices
    SpawnArgs sp;
    sp.seed = seed; sp.env_offset = env_offset; sp.z_lo = z_lo; sp.z_hi = z_hi; sp.xy_radius = xy_radius; sp.xy_sigma = xy_sigma;
    sp.yaw_lo = yaw_lo; sp.yaw_hi = yaw_hi; sp.max_rounds = max_rounds;
    // a warp per env packs 4 envs into a CTA; past 32 agents an env takes a CTA of its own
    if (cfg->N > 32) return launch_spawn_wide(*cfg, *bufs, sp, env_mask, failed_envs, (cudaStream_t)stream);
    spawn_kernel<<<(unsigned)((cfg->E + 3) / 4), 128, 0, (cudaStream_t)stream>>>(*cfg, *bufs, sp, env_mask, failed_envs);
    return last_error();
}


int mrs_autoreset(const MrsConfig* cfg, const MrsBuffers* bufs, const MrsAutoResetArgs* args, const unsigned char* done_in,
                  int* env_steps, unsigned* episode, unsigned char* done_out, int slot_x, int slot_a, unsigned* failed_envs,
                  void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!bufs || !bufs->state || !args || !env_steps || !episode || !done_out) return MRS_ERR_ARG;
    if (!(args->z_hi >= args->z_lo) || !(args->xy_radius > 0.f) || !(args->xy_sigma > 0.f) || args->max_rounds <= 0)
        return MRS_ERR_ARG;
    if (bufs->X_tape && (cfg->state_layout == MRS_X_NONE || slot_x < 0 || slot_x >= cfg->L)) return MRS_ERR_ARG;
    if (bufs->A_tape && (slot_a < 0 || slot_a >= cfg->L)) return MRS_ERR_ARG;
    if ((size_t)cfg->E * (size_t)cfg->N > 0xffffffffull) return MRS_ERR_UNSUPPORTED;     // u32 slot indices
    AutoResetArgs a;
    a.sp.seed = args->seed; a.sp.env_offset = args->env_offset; a.sp.z_lo = args->z_lo; a.sp.z_hi = args->z_hi;
    a.sp.xy_radius = args->xy_radius; a.sp.xy_sigma = args->xy_sigma; a.sp.yaw_lo = args->yaw_lo; a.sp.yaw_hi = args->yaw_hi;
    a.sp.max_rounds = args->max_rounds;
    a.episode_length = args->episode_length; a.max_timesteps = args->max_timesteps;
    a.slot_x = slot_x; a.slot_a = slot_a;
    const Derived d = make_derived(*cfg);         // s_max / comm_inf exactly as the step kernels derive them
    a.s_max = d.s_max; a.comm_inf = d.comm_inf;
    cudaStream_t st = (cudaStream_t)stream;
    if (cfg->N > 32) {
        int threads = (cfg->N + 31) / 32 * 32;
        if (threads > 1024) threads = 1024;
        const size_t smem = 2 * (size_t)((cfg->N + 31) / 32) * sizeof(unsigned);
        static size_t configured[64] = {};
        if ((rc = ensure_dynamic_smem(autoreset_wide_kernel, smem, configured))) return rc;
        autoreset_wide_kernel<<<(unsigned)cfg->E, (unsigned)threads, smem, st>>>(*cfg, *bufs, a, done_in, env_steps, episode,
                                                                                 done_out, failed_envs);
    } else {
        autoreset_kernel<<<(unsigned)((cfg->E + 3) / 4), 128, 0, st>>>(*cfg, *bufs, a, done_in, env_steps, episode, done_out,
                                                                      failed_envs);
    }
    return last_error();
}


int mrs_proximity(const MrsConfig* cfg, const MrsBuffers* bufs, float threshold, float* gap_agent, int* nearest,
                  float* gap_ground, unsigned char* collision, void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!bufs || !bufs->state) return MRS_ERR_ARG;
    const size_t S = (size_t)cfg->E * cfg->N;
    proximity_kernel<<<(unsigned)((S + 127) / 128), 128, 0, (cudaStream_t)stream>>>(*cfg, *bufs, threshold, gap_agent,
                                                                                   nearest, gap_ground, collision);
    return last_error();
}

int mrs_raycast(const MrsConfig* cfg, const MrsBuffers* bufs, const float* directions, int n_rays, const float* offset3,
                int body_frame, float range, float* hit_dist, int* hit_id, void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!bufs || !bufs->state || !directions || n_rays <= 0 || !hit_dist || !hit_id || !(range > 0.f)) return MRS_ERR_ARG;
    const size_t total = (size_t)cfg->E * cfg->N * n_rays;
    if (total >= 0xffffffffull) return MRS_ERR_UNSUPPORTED;
    const float ox = offset3 ? offset3[0] : 0.f, oy = offset3 ? offset3[1] : 0.f, oz = offset3 ? offset3[2] : 0.f;
    raycast_kernel<<<(unsigned)((total + 127) / 128), 128, 0, (cudaStream_t)stream>>>(*cfg, *bufs, directions, n_rays, ox, oy,
                                                                                     oz, body_frame, range, hit_dist, hit_id);
    return last_error();
}

}  // extern "C"
