// mrs_step_env_body.cuh -- the body of step_env_kernel (32 < N <= 128, one CTA per env).
// Compiled into the kernel without the external wrench (EXT = false) and into its overload with it (EXT = true):
// the same text, so the kernel without is what it was before the wrench existed (the body as a shared
// __forceinline__ function lost the __launch_bounds__ range facts ptxas schedules by, and changed its SASS).
// Included only inside those kernel definitions in mrs_step.cuh; no include guard.
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
    ExtWrench xw{};
    if constexpr (EXT) xw = load_wrench(b.wrench, S, s);      // (idle threads read the env's last agent)
    apply_wrench<MODE != MRS_NO_ACTION, EXT>(c, d, st, R, rpm, dw, xw);
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
