// mrs_contact_env.cuh -- joint contact solve of one env by one CTA (N > 32 paths): shared by contact_env_kernel
// (mrs_kernels.cu) and the fused one-CTA-per-env step kernel (mrs_step.cuh).
#pragma once
#include "mrs_common.cuh"

namespace mrs {

// Joint contact solve of ONE env of the wide path (N > 32; bullet_model.solve_contacts), one CTA per env, one thread
// per FLAGGED agent (agents within contact range of another agent: scratch plane 6, written by the pre pass).  An
// env without flagged agents costs one coalesced read of its flags.  The flagged agents' velocities live in shared
// memory; the pairs in range are listed once (they are pairs of flagged agents) with their tournament round.
// A sweep runs the ground rows of the flagged agents, then the pair rows in ascending round order (the oracle's
// order).  Two pairs that share no agent commute exactly, so the order only matters along the chains of pairs that
// share an agent: every pair gets a LEVEL = 1 + the highest level among the pairs of an earlier round that touch one
// of its two agents, and a sweep walks the levels (CTA barrier in between; the pairs of a level touch disjoint
// agents and run in parallel).  The result is bit-identical to the round-by-round walk, but a sweep costs as many
// barriers as the longest chain (a handful in a heap) instead of one per occupied round (up to N - 1).
// The levels come from a relaxation over per-agent pair lists sorted by round (kIncident entries per agent; an
// agent with more pairs in range falls back to the round-by-round walk).
// Agents that touch only the ground are solved on their own in step_post_kernel.
// Limits: blockDim flagged agents and 4 * blockDim pairs per env (blockDim = N rounded up to a warp, <= 1024);
// beyond that the surplus is left unsolved and MRS_STATUS_CONTACT_OVERFLOW is raised.
constexpr int kIncident = 16;
// words of the bit mask of occupied tournament rounds: rounds 0 .. N + (N & 1) - 2
__host__ __device__ inline int contact_env_round_words(int N) { return (N + (N & 1) - 1 + 31) / 32; }
__host__ __device__ inline size_t contact_env_smem(int threads, int N) {
    return (size_t)threads * (4 + 12 + 12 + 4 + 2 * kIncident) + (size_t)(4 * threads) * (4 + 4 + 12) +
           (size_t)contact_env_round_words(N) * 4;
}

// The CTA-wide body: every thread of the CTA calls it (CTA barriers inside) with the env's index; `smem_raw` is
// contact_env_smem(blockDim.x, c.N) bytes of shared memory.  Reads v*, the pre-step positions and the flags from the
// scratch planes 0-6 and w* from the state planes 10-12, writes the solved v and w back there.
static __device__ __noinline__ void contact_env_body(const MrsConfig& c, const Derived& d, const MrsBuffers& b, unsigned env,
                                              unsigned char* smem_raw) {
    __shared__ int n_flag, n_pair, deg_over, changed, max_level;
    __shared__ unsigned worst_bits;
    const int cap = blockDim.x, pcap = 4 * blockDim.x;
    int* fl_idx = reinterpret_cast<int*>(smem_raw);
    float* sp = reinterpret_cast<float*>(fl_idx + cap);            // [cap][3] pre-step positions
    float* sv = sp + 3 * cap;                                       // [cap][3] velocities
    unsigned* pr_ij = reinterpret_cast<unsigned*>(sv + 3 * cap);    // [pcap] lo | hi << 16 (local indices)
    int* pr_round = reinterpret_cast<int*>(pr_ij + pcap);           // [pcap] tournament round, later the level
    float* pr_lam = reinterpret_cast<float*>(pr_round + pcap);      // [pcap][3]
    const int N = c.N, tid = threadIdx.x, words = contact_env_round_words(N);
    unsigned* rmask = reinterpret_cast<unsigned*>(pr_lam + 3 * pcap);   // [words] rounds that hold a pair
    int* deg = reinterpret_cast<int*>(rmask + words);               // [cap] pairs of a flagged agent
    unsigned short* inc = reinterpret_cast<unsigned short*>(deg + cap);     // [cap][kIncident] their indices
    const size_t S = (size_t)c.E * N, env0 = (size_t)env * N;
    const MrsPhysicsParams& ph = c.phys;
    const ContactParams cp = make_contact_params(ph, d);
    const float* __restrict__ sc = b.scratch;
    if (tid == 0) { n_flag = 0; n_pair = 0; deg_over = 0; max_level = 0; }
    for (int w = tid; w < words; w += blockDim.x) rmask[w] = 0u;
    deg[tid] = 0;
    __syncthreads();
    for (int i = tid; i < N; i += blockDim.x)
        if (sc[6 * S + env0 + i] != 0.f) {
            const int f = atomicAdd(&n_flag, 1);
            if (f < cap) fl_idx[f] = i;
        }
    __syncthreads();
    if (n_flag == 0) return;
    const int F = min(n_flag, cap);
    // my agent (thread f < F)
    const bool mine = tid < F;
    const int ai = mine ? fl_idx[tid] : 0;
    const size_t s = env0 + ai;
    float R[9], wb[3] = {0.f, 0.f, 0.f};
    GroundRows g;
    g.act = 0u;
    float lam_g[4] = {0.f, 0.f, 0.f, 0.f}, fl[2] = {0.f, 0.f};
    if (mine) {
        Agent st;
        st.qx = b.state[3 * S + s]; st.qy = b.state[4 * S + s]; st.qz = b.state[5 * S + s]; st.qw = b.state[6 * S + s];
        quat_to_mat(st, R);
        const float wx = b.state[10 * S + s], wy = b.state[11 * S + s], wz = b.state[12 * S + s];
        wb[0] = R[0] * wx + R[3] * wy + R[6] * wz; wb[1] = R[1] * wx + R[4] * wy + R[7] * wz;
        wb[2] = R[2] * wx + R[5] * wy + R[8] * wz;
#pragma unroll
        for (int k = 0; k < 3; ++k) { sp[3 * tid + k] = sc[(3 + k) * S + s]; sv[3 * tid + k] = sc[k * S + s]; }
        if (ph.ground_contact && sp[3 * tid + 2] < d.gnd_skip_z) ground_setup(cp, sp[3 * tid + 2], R, g);
    }
    __syncthreads();
    if (mine) {
        for (int q = 0; q < F; ++q) {
            const int aj = fl_idx[q];
            if (aj <= ai) continue;
            const float dx = sp[3 * tid] - sp[3 * q], dy = sp[3 * tid + 1] - sp[3 * q + 1], dz = sp[3 * tid + 2] - sp[3 * q + 2];
            const float d2 = dx * dx + dy * dy + dz * dz;
            if (d2 < d.lim2 && d2 > 0.f) {
                const int k = atomicAdd(&n_pair, 1);
                if (k < pcap) {
                    const int r = tour_round(ai, aj, N);
                    pr_ij[k] = (unsigned)tid | ((unsigned)q << 16);
                    pr_round[k] = r;
                    pr_lam[3 * k] = pr_lam[3 * k + 1] = pr_lam[3 * k + 2] = 0.f;
                    atomicOr(&rmask[r >> 5], 1u << (r & 31));
                    const int u = atomicAdd(&deg[tid], 1), w = atomicAdd(&deg[q], 1);
                    if (u < kIncident) inc[tid * kIncident + u] = (unsigned short)k;
                    if (w < kIncident) inc[q * kIncident + w] = (unsigned short)k;
                    if (u >= kIncident || w >= kIncident) deg_over = 1;
                }
            }
        }
    }
    __syncthreads();
    const int P = min(n_pair, pcap);
    if ((n_flag > cap || n_pair > pcap) && tid == 0 && b.status) atomicOr(b.status, MRS_STATUS_CONTACT_OVERFLOW);
    const bool by_level = deg_over == 0;
    if (by_level) {
        // my agent's pairs in ascending round order (insertion sort of <= kIncident entries) ...
        unsigned short* my = inc + tid * kIncident;
        const int dg = mine ? deg[tid] : 0;
        for (int i = 1; i < dg; ++i) {
            const unsigned short k = my[i];
            const int r = pr_round[k];
            int j = i - 1;
            while (j >= 0 && pr_round[my[j]] > r) { my[j + 1] = my[j]; --j; }
            my[j + 1] = k;
        }
        __syncthreads();
        // ... then the levels (they replace the rounds): relax level[k] >= 1 + level[previous pair of either agent]
        for (int k = tid; k < P; k += blockDim.x) pr_round[k] = 1;
        for (;;) {
            __syncthreads();
            if (tid == 0) changed = 0;
            __syncthreads();
            int run = 0;
            bool any = false;
            for (int i = 0; i < dg; ++i) {
                const int k = my[i];
                const int lv = max(pr_round[k], run + 1);
                if (lv > pr_round[k]) { atomicMax(&pr_round[k], lv); any = true; }
                run = lv;
            }
            if (any) changed = 1;
            __syncthreads();
            if (!changed) break;
        }
        int top = 0;
        for (int k = tid; k < P; k += blockDim.x) top = max(top, pr_round[k]);
        if (top) atomicMax(&max_level, top);
        __syncthreads();
    }
    const int levels = max_level;
    auto solve_pair = [&](int k) -> float {
        const int lo = pr_ij[k] & 0xffffu, hi = pr_ij[k] >> 16;
        float dv[3];
        bool act;
        const float wr = pair_rows(cp, sp[3 * lo] - sp[3 * hi], sp[3 * lo + 1] - sp[3 * hi + 1],
                                   sp[3 * lo + 2] - sp[3 * hi + 2], sv + 3 * lo, sv + 3 * hi, pr_lam + 3 * k, dv, act);
#pragma unroll
        for (int q = 0; q < 3; ++q) { sv[3 * lo + q] += dv[q]; sv[3 * hi + q] -= dv[q]; }
        return wr;
    };
    for (int it = 0; it < ph.solver_iters; ++it) {
        if (tid == 0) worst_bits = 0u;
        float worst = 0.f;
        if (mine && g.act) {
            float v[3] = {sv[3 * tid], sv[3 * tid + 1], sv[3 * tid + 2]};
            worst = ground_sweep(cp, g, lam_g, fl, v, wb);
            sv[3 * tid] = v[0]; sv[3 * tid + 1] = v[1]; sv[3 * tid + 2] = v[2];
        }
        __syncthreads();
        if (by_level) {
            for (int lv = 1; lv <= levels; ++lv) {
                for (int k = tid; k < P; k += blockDim.x)
                    if (pr_round[k] == lv) worst = fmaxf(worst, solve_pair(k));
                __syncthreads();
            }
        } else {
            for (int w = 0; w < words; ++w) {
                for (unsigned m = rmask[w]; m; m &= m - 1u) {
                    const int r = 32 * w + __ffs(m) - 1;
                    for (int k = tid; k < P; k += blockDim.x)
                        if (pr_round[k] == r) worst = fmaxf(worst, solve_pair(k));
                    __syncthreads();
                }
            }
        }
        atomicMax(&worst_bits, __float_as_uint(worst));
        __syncthreads();
        const bool done = __uint_as_float(worst_bits) < ph.solver_tol;
        __syncthreads();
        if (done) break;
    }
    unsigned rows = 0;
    for (int k = tid; k < P; k += blockDim.x)
        if (pr_lam[3 * k] > 0.f) rows += 2;           // counted per agent, like the N <= 32 path
    if (mine) {
        float* scw = b.scratch;
#pragma unroll
        for (int k = 0; k < 3; ++k) scw[k * S + s] = sv[3 * tid + k];
        b.state[10 * S + s] = R[0] * wb[0] + R[1] * wb[1] + R[2] * wb[2];
        b.state[11 * S + s] = R[3] * wb[0] + R[4] * wb[1] + R[5] * wb[2];
        b.state[12 * S + s] = R[6] * wb[0] + R[7] * wb[1] + R[8] * wb[2];
    }
    const unsigned gnd = (mine && (lam_g[0] + lam_g[1]) + (lam_g[2] + lam_g[3]) > 0.f) ? 1u : 0u;
    const unsigned w_rows = __reduce_add_sync(kFull32, rows), w_gnd = __reduce_add_sync(kFull32, gnd);
    if ((tid & 31) == 0 && b.stats) {
        if (w_rows) atomicAdd(b.stats + MRS_STAT_AGENT_CONTACTS, (unsigned long long)w_rows);
        if (w_gnd) atomicAdd(b.stats + MRS_STAT_GROUND_CONTACTS, (unsigned long long)w_gnd);
    }
}


}  // namespace mrs
