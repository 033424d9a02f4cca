// mrs_step_pre_body.cuh -- the body of step_pre_kernel (N > 32, lanes per agent).
// Compiled into the kernel without the external wrench (EXT = false) and into its overload with it (EXT = true):
// the same text, so the kernel without is what it was before the wrench existed (the body as a shared
// __forceinline__ function lost the __launch_bounds__ range facts ptxas schedules by, and changed its SASS).
// Included only inside those kernel definitions in mrs_step.cuh; no include guard.
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
    agent_pre<MODE, EXT>(c, d, b, actions, S, s, dw, near && pair_contact);
