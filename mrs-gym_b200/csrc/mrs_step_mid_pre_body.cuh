// mrs_step_mid_pre_body.cuh -- the body of step_mid_pre_kernel (32 < N <= 128, thread per agent).
// Compiled into the kernel without the external wrench (EXT = false) and into its overload with it (EXT = true):
// the same text, so the kernel without is what it was before the wrench existed (the body as a shared
// __forceinline__ function lost the __launch_bounds__ range facts ptxas schedules by, and changed its SASS).
// Included only inside those kernel definitions in mrs_step.cuh; no include guard.
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
    if (valid) agent_pre<MODE, EXT>(c, d, b, actions, S, s, dw, near && pair_contact);
