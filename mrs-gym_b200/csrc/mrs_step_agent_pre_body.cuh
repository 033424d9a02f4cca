// mrs_step_agent_pre_body.cuh -- the body of agent_pre_kernel (N > 128).
// Compiled into the kernel without the external wrench (EXT = false) and into its overload with it (EXT = true):
// the same text, so the kernel without is what it was before the wrench existed (the body as a shared
// __forceinline__ function lost the __launch_bounds__ range facts ptxas schedules by, and changed its SASS).
// Included only inside those kernel definitions in mrs_step.cuh; no include guard.
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
    agent_pre<MODE, EXT>(c, d, b, actions, S, s, dw, fl != 0.f);
