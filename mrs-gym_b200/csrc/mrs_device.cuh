// Per-agent device math of the mrs-gym step path (sm_100a).  fp32 throughout, no fast-math:
// the adjacency must be bit-exact and the dynamics must hold 1e-4 relative on one-step deltas.
//
// Reference being reproduced (files under /root/reference/mrsgym):
//   QuadControl.py:35-127   cascaded PID (pos -> vel -> accel -> attitude -> pwm -> rpm)
//   Quadcopter.py:26-65     action modes, Quadcopter.py:172-208 nnlsRPM mixer
//   Quadcopter.py:38-45     rotor thrust / yaw torque, Quadcopter.py:69-115 aero "dynamics"
//   BulletSim.py:46-47      p.stepSimulation (Bullet3 semantics: oracle/bullet_model.py)
// The controller works on rotation matrices straight from the quaternion (the reference's
// matrix->euler->matrix round trips are identity maps on SO(3)).
#pragma once
#include <cuda_runtime.h>
#include <math.h>

#include "mrs_b200.h"

namespace mrs {

struct Agent {
    float px, py, pz;
    float qx, qy, qz, qw;
    float vx, vy, vz;
    float wx, wy, wz;
};

// minb: resident CTAs per SM the group kernel is compiled for (register budget per mode)
// PID planes touched per mode (the rest of the 18 ctrl planes stay untouched in HBM)
struct Ctrl {
    float io[3];   // integral_ori_e
    float ip[3];   // integral_pos_e
    float iv[3];   // integral_vel_e
    float lve[3];  // last_vel_e (x = NaN: never called)
    float dve[3];  // d_vel_e
    float ltv[3];  // last_target_vel
};

#ifndef MRS_MINB_VEL
#define MRS_MINB_VEL 5
#endif
#ifndef MRS_MINB_POS
#define MRS_MINB_POS 6
#endif
#ifndef MRS_MINB_ACC
#define MRS_MINB_ACC 6
#endif
template <int MODE> struct ModeTraits;
template <> struct ModeTraits<MRS_SET_TARGET_VEL>   { static constexpr int A = 3; static constexpr bool io = true,  ip = false, vel = true;  static constexpr int minb = MRS_MINB_VEL; };
template <> struct ModeTraits<MRS_SET_TARGET_POS>   { static constexpr int A = 3; static constexpr bool io = true,  ip = true,  vel = false;  static constexpr int minb = MRS_MINB_POS; };
template <> struct ModeTraits<MRS_SET_TARGET_ACCEL> { static constexpr int A = 3; static constexpr bool io = true,  ip = false, vel = false;  static constexpr int minb = MRS_MINB_ACC; };
template <> struct ModeTraits<MRS_SET_FORCE>        { static constexpr int A = 3; static constexpr bool io = true,  ip = false, vel = false;  static constexpr int minb = MRS_MINB_ACC; };
template <> struct ModeTraits<MRS_SET_TARGET_ORI>   { static constexpr int A = 3; static constexpr bool io = true,  ip = false, vel = false;  static constexpr int minb = MRS_MINB_ACC; };
template <> struct ModeTraits<MRS_SET_CONTROL>      { static constexpr int A = 4; static constexpr bool io = false, ip = false, vel = false;  static constexpr int minb = 7; };
#ifndef MRS_MINB_SPEEDS
#define MRS_MINB_SPEEDS 7
#endif
template <> struct ModeTraits<MRS_SET_SPEEDS>       { static constexpr int A = 4; static constexpr bool io = false, ip = false, vel = false;  static constexpr int minb = MRS_MINB_SPEEDS; };
template <> struct ModeTraits<MRS_NO_ACTION>        { static constexpr int A = 0; static constexpr bool io = false, ip = false, vel = false;  static constexpr int minb = 7; };

// PID planes a mode carries through the prefetch stage, in stage order: io (planes 0-2), then ip
// (3-5) or the 12 velocity-controller planes (6-17)
template <int MODE> __host__ __device__ constexpr int mode_nctrl() {
    return (ModeTraits<MODE>::io ? 3 : 0) + (ModeTraits<MODE>::ip ? 3 : 0) + (ModeTraits<MODE>::vel ? 12 : 0);
}
template <int MODE> __host__ __device__ constexpr int mode_ctrl_plane(int ordinal) {
    return (ModeTraits<MODE>::vel && ordinal >= 3) ? ordinal + 3 : ordinal;
}
template <int MODE> __host__ __device__ constexpr int mode_stage_floats() {
    return (13 + mode_nctrl<MODE>()) * 32 + ModeTraits<MODE>::A * 32;
}

__host__ __device__ __forceinline__ int state_dim(int layout) {
    return layout == MRS_X_POS_VEL ? 6 : (layout == MRS_X_FULL ? 13 : 0);
}

__device__ __forceinline__ float clampf(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }

// body->world rotation, row-major R[3*i+j], from an xyzw unit quaternion
__device__ __forceinline__ void quat_to_mat(const Agent& s, float* R) {
    const float x = s.qx, y = s.qy, z = s.qz, w = s.qw;
    R[0] = 1.f - 2.f * (y * y + z * z); R[1] = 2.f * (x * y - z * w);       R[2] = 2.f * (x * z + y * w);
    R[3] = 2.f * (x * y + z * w);       R[4] = 1.f - 2.f * (x * x + z * z); R[5] = 2.f * (y * z - x * w);
    R[6] = 2.f * (x * z - y * w);       R[7] = 2.f * (y * z + x * w);       R[8] = 1.f - 2.f * (x * x + y * y);
}

// ------------------------------------------------------------------------------------------
// Host-derived constants (reciprocals, products) so that the per-agent code carries no uniform
// divisions.  Not part of the C ABI: step_impl() fills it from MrsConfig for every call.
struct Derived {
    float inv_mass, inv_I[3];
    float gnd_c;         // kf * gnd_eff_coeff * (prop_radius/4)^2      (ground effect numerator)
    float dw_c;          // dw1 * (prop_radius/4)^2                      (downwash alpha numerator)
    float rpm2rad;       // 2*pi/60
    float q_x2;          // 0.25*dt^2: squared half rotation angle per unit |w|^2
    float cap_w2;        // (ang_motion_threshold/dt)^2
    float cap_k, cap_c;  // sin(pi/8) / ((pi/4)/dt), cos(pi/8): Bullet's capped angular step
    float lim2;          // (2*contact_radius + contact_margin)^2
    float gnd_skip_z;    // above this height the ground contact row cannot be active
    float inv_dt, erp_dt;
    float s_max;         // adjacency threshold on the squared distance
    int comm_inf;
    float inv_ctrl_dt;   // 1 / QuadControl DT
    float inv_4kf;       // 1 / (4 kf)
    float inv_pwm_a;     // 1 / pwm2rpm_a
    float inv_qmass;     // 1 / quad mass (set_force := set_target_accel(F / Mass))
};

__device__ __forceinline__ float fast_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_rsqrt(float x) { float y; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_sqrt(float x) { float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// 1/sqrt(x) to full float32 accuracy: SFU seed + one Newton step (x > 0)
__device__ __forceinline__ float rsqrt_nr(float x) {
    const float y = fast_rsqrt(x);
    return y * (1.5f - 0.5f * x * y * y);
}

// ------------------------------------------------------------------------------------------
// QuadControl.attitude_control (QuadControl.py:93-127) on matrices.  Rt = target rotation
// (columns t0 t1 t2, row-major like R), ta = target acceleration incl. gravity.
__device__ __forceinline__ void attitude_control(const MrsQuadParams& q, const Derived& d, const float* R, const float* Rt,
                                                 const float* ta, float nrm, float inv_nrm, const Agent& s, float* io,
                                                 float* rpm) {
    // rot_matrix_e = Rt^T R - R^T Rt ; rot_e = [e21, e02, e10]
    float re[3];
    re[0] = (Rt[2] * R[1] + Rt[5] * R[4] + Rt[8] * R[7]) - (R[2] * Rt[1] + R[5] * Rt[4] + R[8] * Rt[7]);
    re[1] = (Rt[0] * R[2] + Rt[3] * R[5] + Rt[6] * R[8]) - (R[0] * Rt[2] + R[3] * Rt[5] + R[6] * Rt[8]);
    re[2] = (Rt[1] * R[0] + Rt[4] * R[3] + Rt[7] * R[6]) - (R[1] * Rt[0] + R[4] * Rt[3] + R[7] * Rt[6]);
    const float we[3] = {-s.wx, -s.wy, -s.wz};   // target_angvel(0) - world angvel
    float tt[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float v = clampf(io[k] - re[k] * q.ctrl_dt, -1500.f, 1500.f);
        if (k < 2) v = clampf(v, -1.f, 1.f);
        io[k] = v;
        tt[k] = clampf(-q.ori_p[k] * re[k] + q.ori_i[k] * v + q.ori_d[k] * we[k], -3200.f, 3200.f);
    }
    // thrust: |a| m / max(cos(angle(a, body z)), 0.2); nrm = |a|, inv_nrm = 1/|a| (0 if |a| = 0)
    const float cosang = (ta[0] * R[2] + ta[1] * R[5] + ta[2] * R[8]) * inv_nrm;
    const float scalar_thrust = (nrm != 0.f) ? nrm * q.mass * fast_rcp(fmaxf(cosang, 0.2f)) : 0.f;
    const float thrust = (fast_sqrt(scalar_thrust * d.inv_4kf) - q.pwm2rpm_b) * d.inv_pwm_a;
    // MixerMatrix rows (QuadControl.py:26): [.5,-.5,-1] [.5,.5,1] [-.5,.5,-1] [-.5,-.5,1]
    const float m0 = 0.5f * tt[0], m1 = 0.5f * tt[1], m2 = tt[2];
    float pwm[4] = {thrust + m0 - m1 - m2, thrust + m0 + m1 + m2, thrust - m0 + m1 - m2, thrust - m0 - m1 + m2};
#pragma unroll
    for (int i = 0; i < 4; ++i) rpm[i] = q.pwm2rpm_a * clampf(pwm[i], q.min_pwm, q.max_pwm) + q.pwm2rpm_b;
}

// QuadControl.accel_control (QuadControl.py:73-90): target frame z = a/|a|,
// x = R[:,1] x z, y = z x x, columns normalised (= scipy from_matrix on orthogonal columns).
__device__ __forceinline__ void accel_control(const MrsQuadParams& q, const Derived& d, const float* R, const float* a_in,
                                              const Agent& s, float* io, float* rpm) {
    const float ta[3] = {a_in[0], a_in[1], a_in[2] + q.ctrl_gravity};
    const float n2 = ta[0] * ta[0] + ta[1] * ta[1] + ta[2] * ta[2];
    float z[3] = {0.f, 0.f, 1.f};
    float inv = 0.f;
    if (n2 > 0.f) {   // |a| == 0 -> NaN -> [0,0,1] in the reference
        inv = rsqrt_nr(n2);
        z[0] = ta[0] * inv; z[1] = ta[1] * inv; z[2] = ta[2] * inv;
    }
    // x = R[:,1] x z
    float x[3] = {R[4] * z[2] - R[7] * z[1], R[7] * z[0] - R[1] * z[2], R[1] * z[1] - R[4] * z[0]};
    const float xi = rsqrt_nr(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
    x[0] *= xi; x[1] *= xi; x[2] *= xi;
    const float y[3] = {z[1] * x[2] - z[2] * x[1], z[2] * x[0] - z[0] * x[2], z[0] * x[1] - z[1] * x[0]};
    const float Rt[9] = {x[0], y[0], z[0], x[1], y[1], z[1], x[2], y[2], z[2]};
    attitude_control(q, d, R, Rt, ta, n2 * inv, inv, s, io, rpm);
}

// rotation matrix of scipy euler 'xyz' (extrinsic) = Rz(yaw) Ry(pitch) Rx(roll)
__device__ __forceinline__ void euler_to_mat(float roll, float pitch, float yaw, float* M) {
    float sr, cr, sp, cp, sy, cy;
    sincosf(roll, &sr, &cr); sincosf(pitch, &sp, &cp); sincosf(yaw, &sy, &cy);
    M[0] = cy * cp; M[1] = cy * sp * sr - sy * cr; M[2] = cy * sp * cr + sy * sr;
    M[3] = sy * cp; M[4] = sy * sp * sr + cy * cr; M[5] = sy * sp * cr - cy * sr;
    M[6] = -sp;     M[7] = cp * sr;                M[8] = cp * cr;
}

// nnlsRPM (Quadcopter.py:172-208).  The 4x4 NNLS is solved by enumerating the 16 active
// sets: the optimum is the primal-feasible subset solution of least residual.
static __device__ __noinline__ void nnls_enumerate(const MrsQuadParams& q, const float* B, float* sq) {
    float best = INFINITY;
    for (int m = 0; m < 16; ++m) {
        float x[4];
        bool ok = true;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float* t = q.nnls_tab + m * 16 + i * 4;
            x[i] = t[0] * B[0] + t[1] * B[1] + t[2] * B[2] + t[3] * B[3];
            ok = ok && (x[i] >= 0.f);
        }
        if (!ok) continue;
        float res = 0.f;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const float* a = q.mix_a + r * 4;
            const float d = a[0] * x[0] + a[1] * x[1] + a[2] * x[2] + a[3] * x[3] - B[r];
            res += d * d;
        }
        if (res < best) {
            best = res;
            sq[0] = x[0]; sq[1] = x[1]; sq[2] = x[2]; sq[3] = x[3];
        }
    }
}

// q: scalar model constants (compile-time values in the baked kernels), qt: the mixer tables, always
// read from the kernel parameter (they are indexed at run time)
__device__ __forceinline__ void set_control(const MrsQuadParams& q, const MrsQuadParams& qt, const float* act, float* rpm) {
    const float inv_kfl = 1.f / (q.kf * q.arm);
    const float B[4] = {act[0] * q.mass / q.kf, act[1] * q.ixx * inv_kfl, act[2] * q.iyy * inv_kfl,
                        act[3] * q.izz / q.km};
    float sq[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float* a = qt.mix_ainv + i * 4;
        sq[i] = a[0] * B[0] + a[1] * B[1] + a[2] * B[2] + a[3] * B[3];
    }
    if (fminf(fminf(sq[0], sq[1]), fminf(sq[2], sq[3])) < 0.f) nnls_enumerate(qt, B, sq);
#pragma unroll
    for (int i = 0; i < 4; ++i) rpm[i] = sqrtf(sq[i]);
}

// ------------------------------------------------------------------------------------------
// action -> rpm for one agent (Quadcopter.set_* -> QuadControl.*).
template <int MODE>
__device__ __forceinline__ void action_to_rpm(const MrsConfig& c, const MrsQuadParams& qt, const Derived& d, const Agent& s,
                                              const float* R, const float* act, Ctrl& k, float* rpm) {
    const MrsQuadParams& q = c.quad;
    if constexpr (MODE == MRS_SET_SPEEDS) {
#pragma unroll
        for (int i = 0; i < 4; ++i) rpm[i] = act[i];
    } else if constexpr (MODE == MRS_SET_CONTROL) {
        set_control(q, qt, act, rpm);
    } else if constexpr (MODE == MRS_SET_TARGET_ORI) {
        float Rt[9];
        euler_to_mat(act[0], act[1], act[2], Rt);
        const float ta[3] = {0.f, 0.f, 9.81f};   // literal in Quadcopter.py:64
        attitude_control(q, d, R, Rt, ta, 9.81f, 1.f / 9.81f, s, k.io, rpm);
    } else if constexpr (MODE == MRS_SET_TARGET_ACCEL) {
        accel_control(q, d, R, act, s, k.io, rpm);
    } else if constexpr (MODE == MRS_SET_FORCE) {
        const float a[3] = {act[0] * d.inv_qmass, act[1] * d.inv_qmass, act[2] * d.inv_qmass};
        accel_control(q, d, R, a, s, k.io, rpm);
    } else if constexpr (MODE == MRS_SET_TARGET_POS) {
        // QuadControl.pos_control (QuadControl.py:35-48)
        const float p[3] = {s.px, s.py, s.pz}, v[3] = {s.vx, s.vy, s.vz};
        float a[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float e = act[i] - p[i];
            k.ip[i] = k.ip[i] + e * q.ctrl_dt;
            a[i] = q.pos_p * e + q.pos_i * k.ip[i] + q.pos_d * (0.f - v[i]);
        }
        accel_control(q, d, R, a, s, k.io, rpm);
    } else if constexpr (MODE == MRS_SET_TARGET_VEL) {
        // QuadControl.vel_control (QuadControl.py:51-70)
        const float v[3] = {s.vx, s.vy, s.vz};
        const bool first = isnan(k.lve[0]);
        float a[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float e = act[i] - v[i];
            const float le = first ? e : k.lve[i];
            const float lt = first ? act[i] : k.ltv[i];
            const float d0 = first ? 0.f : k.dve[i];
            const float dv = (((e - le) - (act[i] - lt)) * d.inv_ctrl_dt) * 0.5f + d0 * 0.5f;
            k.dve[i] = dv;
            k.lve[i] = e;
            k.ltv[i] = act[i];
            k.iv[i] = k.iv[i] + e * q.ctrl_dt;
            a[i] = q.vel_p * e + q.vel_i * k.iv[i] + q.vel_d * dv;
        }
        accel_control(q, d, R, a, s, k.io, rpm);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) rpm[i] = 0.f;
    }
}

// One pair of the downwash loop (Quadcopter.py:99-115): body-z force on agent i caused by agent
// j (rel = p_j - p_i):  -alpha * exp(-0.5 (dxy/beta)^2), alpha = dw1 (prop_radius/(4 dz))^2,
// beta = dw2 dz + dw3, applied iff dz > 0 and dxy < 10.  Branch-free: only squares of dxy and
// beta appear, so no sqrt; reciprocals and the exponential go to the SFU (rel. error <= 2e-6 of
// a term that is itself <= ~0.3 of the weight; the parity floor is 5e-7 m/s per step).
__device__ __forceinline__ float downwash_pair(const MrsQuadParams& q, const Derived& d, float dxy2, float rz) {
    const float beta = q.dw2 * rz + q.dw3;
    // beta^2 is floored at 1e-30: at beta == 0 the reference gets exp(-inf) = 0 (or NaN for dxy == 0, a
    // bug of its own); the floor keeps both factors finite and yields the same 0
    const float bb = fmaxf(beta * beta, 1e-30f), zz = rz * rz;
    // two SFU reciprocals: one rcp(bb * zz) shared by both factors costs three more FMULs per pair than it
    // saves in SFU work, and the kernel is issue-bound, not SFU-bound (XU pipe ~20 % busy): 17.3 -> 17.05 us at C5
    const float ibb = fast_rcp(bb), izz = fast_rcp(zz);
    const float e = -0.72134752044448170368f * dxy2 * ibb;         // -0.5*log2(e)*(dxy/beta)^2
    const float f = -d.dw_c * izz * fast_ex2(e);
    return (rz > 0.f && dxy2 < 100.f) ? f : 0.f;
}

// The caller's external wrench of one agent (MrsBuffers.wrench): force at the CoM and torque, both world frame.
struct ExtWrench {
    float f[3], t[3];
};

// rotor thrust + yaw torque (Quadcopter.py:38-45), ground effect / drag (Quadcopter.py:69-98),
// downwash sum `dw` -> Bullet unconstrained velocity update (bullet_model.unconstrained_velocities).
// EXT: the external wrench xw joins the applied wrench (force after the rotation of the body-frame sum, torque
// rotated into the body frame before I^-1), so the contact solve sees it like any other applied force.  Without
// EXT the code is the one of the kernels that never read a wrench (x + 0 does not fold under IEEE rules).
// Overwrites s.v / s.w with the unconstrained velocities v*, w*.
template <bool FORCES, bool EXT = false>
__device__ __forceinline__ void apply_wrench(const MrsConfig& c, const Derived& d, Agent& s, const float* R,
                                             const float* rpm, float dw, const ExtWrench& xw = ExtWrench{}) {
    const MrsQuadParams& q = c.quad;
    const MrsPhysicsParams& ph = c.phys;
    float Fb[3] = {0.f, 0.f, 0.f}, Tb[3] = {0.f, 0.f, 0.f};
    if constexpr (FORCES) {
        float w2[4], fz = 0.f;
        const bool gnd_ok = (R[8] > 0.f) || (R[7] < 0.f);   // roll < pi/2 (pitch < pi/2 always)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            w2[i] = rpm[i] * rpm[i];
            float f = w2[i] * q.kf;
            if (gnd_ok) {
                const float h = fmaxf(s.pz + R[6] * q.prop_x[i] + R[7] * q.prop_y[i], q.gnd_hclip);
                f += w2[i] * d.gnd_c * fast_rcp(h * h);
            }
            fz += f;
            Tb[0] += q.prop_y[i] * f;
            Tb[1] -= q.prop_x[i] * f;
        }
        Tb[2] = q.km * (-w2[0] + w2[1] - w2[2] + w2[3]);
        // drag = R (c * v) applied again in the link frame
        const float ssum = d.rpm2rad * (rpm[0] + rpm[1] + rpm[2] + rpm[3]);
        const float cx = -q.drag_xy * ssum * s.vx, cy = -q.drag_xy * ssum * s.vy, cz = -q.drag_z * ssum * s.vz;
        Fb[0] = R[0] * cx + R[1] * cy + R[2] * cz;
        Fb[1] = R[3] * cx + R[4] * cy + R[5] * cz;
        Fb[2] = R[6] * cx + R[7] * cy + R[8] * cz + fz + dw;
    }
    if constexpr (EXT) {    // external torque, world -> body: R^T tau
        Tb[0] += R[0] * xw.t[0] + R[3] * xw.t[1] + R[6] * xw.t[2];
        Tb[1] += R[1] * xw.t[0] + R[4] * xw.t[1] + R[7] * xw.t[2];
        Tb[2] += R[2] * xw.t[0] + R[5] * xw.t[1] + R[8] * xw.t[2];
    }
    // linear: a = (R Fb + F_ext) / m - g z - v (k + k|v|)
    const float im = d.inv_mass;
    const float vn = fast_sqrt(s.vx * s.vx + s.vy * s.vy + s.vz * s.vz);
    const float kl = ph.lin_damping + ph.lin_damping * vn;
    float ax, ay, az;
    if constexpr (EXT) {
        ax = ((R[0] * Fb[0] + R[1] * Fb[1] + R[2] * Fb[2]) + xw.f[0]) * im - s.vx * kl;
        ay = ((R[3] * Fb[0] + R[4] * Fb[1] + R[5] * Fb[2]) + xw.f[1]) * im - s.vy * kl;
        az = ((R[6] * Fb[0] + R[7] * Fb[1] + R[8] * Fb[2]) + xw.f[2]) * im - c.gravity - s.vz * kl;
    } else {
        ax = (R[0] * Fb[0] + R[1] * Fb[1] + R[2] * Fb[2]) * im - s.vx * kl;
        ay = (R[3] * Fb[0] + R[4] * Fb[1] + R[5] * Fb[2]) * im - s.vy * kl;
        az = (R[6] * Fb[0] + R[7] * Fb[1] + R[8] * Fb[2]) * im - c.gravity - s.vz * kl;
    }
    // angular in the body frame: I wdot = tau - w x Iw - Iw (k + k|w|)
    const float wb[3] = {R[0] * s.wx + R[3] * s.wy + R[6] * s.wz, R[1] * s.wx + R[4] * s.wy + R[7] * s.wz,
                         R[2] * s.wx + R[5] * s.wy + R[8] * s.wz};
    const float Iw[3] = {ph.inertia[0] * wb[0], ph.inertia[1] * wb[1], ph.inertia[2] * wb[2]};
    const float wn = fast_sqrt(wb[0] * wb[0] + wb[1] * wb[1] + wb[2] * wb[2]);
    const float ka = ph.ang_damping + ph.ang_damping * wn;
    float rhs[3] = {Tb[0] - Iw[0] * ka, Tb[1] - Iw[1] * ka, Tb[2] - Iw[2] * ka};
    if (ph.gyro) {
        rhs[0] -= wb[1] * Iw[2] - wb[2] * Iw[1];
        rhs[1] -= wb[2] * Iw[0] - wb[0] * Iw[2];
        rhs[2] -= wb[0] * Iw[1] - wb[1] * Iw[0];
    }
    const float wd[3] = {rhs[0] * d.inv_I[0], rhs[1] * d.inv_I[1], rhs[2] * d.inv_I[2]};
    const float mv = ph.max_coord_vel;
    s.vx = clampf(s.vx + c.dt * ax, -mv, mv);
    s.vy = clampf(s.vy + c.dt * ay, -mv, mv);
    s.vz = clampf(s.vz + c.dt * az, -mv, mv);
    s.wx = clampf(s.wx + c.dt * (R[0] * wd[0] + R[1] * wd[1] + R[2] * wd[2]), -mv, mv);
    s.wy = clampf(s.wy + c.dt * (R[3] * wd[0] + R[4] * wd[1] + R[5] * wd[2]), -mv, mv);
    s.wz = clampf(s.wz + c.dt * (R[6] * wd[0] + R[7] * wd[1] + R[8] * wd[2]), -mv, mv);
}

// ------------------------------------------------------------------------------------------
// Contact solver (bullet_model.solve_contacts): velocity-level sequential impulses, restitution 0, Baumgarte
// push-out, `solver_iters` Gauss-Seidel sweeps with early exit below `solver_tol`.  Sweep order: the ground rows
// of every agent (four lower-rim points of the collision cylinder, normal rows applied AT the points -> righting
// torque; two friction rows at the CoM), then the agent-agent rows (CONTACT_RADIUS spheres: central normal row +
// two friction rows on the CoM velocities) in round-robin-tournament order -- the rows of one round touch disjoint
// agents, so a warp (N <= 32) or a CTA (N > 32) processes a round in parallel without changing the result.

// the constants the contact rows use, gathered from MrsPhysicsParams / Derived at the call site: a plain value
// (the out-of-line warp solver takes it by value, so the hot kernels never have to keep their configuration in memory)
struct ContactParams {
    float mass, inv_mass, inv_I[3];
    float col_radius, col_halfheight, col_margin, ground_z, contact_margin, slop, inv_dt, erp_dt;
    float mu_ground, mu_agent, contact_radius, lim2, gnd_skip_z, solver_tol;
    int solver_iters, ground_contact, agent_contact;
};
__device__ __forceinline__ ContactParams make_contact_params(const MrsPhysicsParams& ph, const Derived& d) {
    ContactParams cp;
    cp.mass = ph.mass; cp.inv_mass = d.inv_mass;
    cp.inv_I[0] = d.inv_I[0]; cp.inv_I[1] = d.inv_I[1]; cp.inv_I[2] = d.inv_I[2];
    cp.col_radius = ph.col_radius; cp.col_halfheight = ph.col_halfheight; cp.col_margin = ph.col_margin;
    cp.ground_z = ph.ground_z; cp.contact_margin = ph.contact_margin; cp.slop = ph.slop;
    cp.inv_dt = d.inv_dt; cp.erp_dt = d.erp_dt;
    cp.mu_ground = ph.mu_ground; cp.mu_agent = ph.mu_agent; cp.contact_radius = ph.contact_radius;
    cp.lim2 = d.lim2; cp.gnd_skip_z = d.gnd_skip_z; cp.solver_tol = ph.solver_tol;
    cp.solver_iters = ph.solver_iters; cp.ground_contact = ph.ground_contact; cp.agent_contact = ph.agent_contact;
    return cp;
}

// velocity bound of a normal row: vn >= bias after the solve (bullet_model._contact_bias)
__device__ __forceinline__ float contact_bias(const ContactParams& cp, float dist) {
    const float pen = dist + cp.slop;
    return (pen > 0.f) ? -pen * cp.inv_dt : -pen * cp.erp_dt;
}

// ground rows of one agent.  nb = world z in the body frame (row 2 of R); the contact points are
// c_p = (+-r, 0, cz), (0, +-r, cz) on the rim of the face that looks down (cz = -h sign(R22));
// a_p = c_p x nb is the angular Jacobian of point p's normal row in the body frame.
struct GroundRows {
    float A, B, rnx, rny, rnz;      // a_0 = (A, B - rnz, rny), a_1 = (A + rnz, B, -rnx), a_2 = (A, B + rnz, -rny), a_3 = (A - rnz, B, rnx)
    float K[4], invK[4], bias[4];
    unsigned act;                   // bit p: point p is within the contact margin
};

__device__ __forceinline__ void ground_point_jacobian(const GroundRows& g, int p, float* a) {
    a[0] = g.A + ((p == 1) ? g.rnz : (p == 3) ? -g.rnz : 0.f);
    a[1] = g.B + ((p == 0) ? -g.rnz : (p == 2) ? g.rnz : 0.f);
    a[2] = (p == 0) ? g.rny : (p == 1) ? -g.rnx : (p == 2) ? -g.rny : g.rnx;
}

__device__ __forceinline__ void ground_setup(const ContactParams& cp, float pz, const float* R,
                                             GroundRows& g) {
    const float nx = R[6], ny = R[7], nz = R[8];
    const float cz = (nz >= 0.f) ? -cp.col_halfheight : cp.col_halfheight;
    g.A = -cz * ny; g.B = cz * nx;
    g.rnx = cp.col_radius * nx; g.rny = cp.col_radius * ny; g.rnz = cp.col_radius * nz;
    const float zc = pz + cz * nz - cp.col_margin - cp.ground_z;
    const float dist[4] = {zc + g.rnx, zc + g.rny, zc - g.rnx, zc - g.rny};
    g.act = 0u;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        float a[3];
        ground_point_jacobian(g, p, a);
        g.K[p] = cp.inv_mass + a[0] * a[0] * cp.inv_I[0] + a[1] * a[1] * cp.inv_I[1] + a[2] * a[2] * cp.inv_I[2];
        g.invK[p] = 1.f / g.K[p];
        g.bias[p] = contact_bias(cp, dist[p]);
        if (dist[p] < cp.contact_margin) g.act |= 1u << p;
    }
}

// one sweep over the ground rows of one agent; v world, wb body-frame angular velocity; returns the largest
// change of a row's contact-point velocity in the sweep
__device__ __forceinline__ float ground_sweep(const ContactParams& cp, const GroundRows& g, float* lam,
                                              float* fl, float* v, float* wb) {
    float worst = 0.f;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        float a[3];
        ground_point_jacobian(g, p, a);
        const float vn = v[2] + a[0] * wb[0] + a[1] * wb[1] + a[2] * wb[2];
        const float ln = fmaxf(lam[p] + (g.bias[p] - vn) * g.invK[p], 0.f);
        const float dl = ((g.act >> p) & 1u) ? ln - lam[p] : 0.f;
        lam[p] += dl;
        v[2] += dl * cp.inv_mass;
        wb[0] += a[0] * cp.inv_I[0] * dl; wb[1] += a[1] * cp.inv_I[1] * dl; wb[2] += a[2] * cp.inv_I[2] * dl;
        worst = fmaxf(worst, fabsf(dl) * g.K[p]);
    }
    const float lim = cp.mu_ground * ((lam[0] + lam[1]) + (lam[2] + lam[3]));
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const float ln = clampf(fl[k] - v[k] * cp.mass, -lim, lim);
        const float dl = ln - fl[k];
        fl[k] = ln;
        v[k] += dl * cp.inv_mass;
        worst = fmaxf(worst, fabsf(dl) * cp.inv_mass);
    }
    return worst;
}

// ground rows only (an agent that touches nothing but the ground): all sweeps at once.  Returns true when a
// normal impulse acted.
__device__ __forceinline__ bool ground_solve(const ContactParams& cp, Agent& s, const float* R, unsigned* sweeps = nullptr) {
    GroundRows g;
    ground_setup(cp, s.pz, R, g);
    if (g.act == 0u) return false;
    float lam[4] = {0.f, 0.f, 0.f, 0.f}, fl[2] = {0.f, 0.f};
    float v[3] = {s.vx, s.vy, s.vz};
    float wb[3] = {R[0] * s.wx + R[3] * s.wy + R[6] * s.wz, R[1] * s.wx + R[4] * s.wy + R[7] * s.wz,
                   R[2] * s.wx + R[5] * s.wy + R[8] * s.wz};
    unsigned n = 0;
    for (int it = 0; it < cp.solver_iters; ++it) {
        ++n;
        if (ground_sweep(cp, g, lam, fl, v, wb) < cp.solver_tol) break;
    }
    if (sweeps) *sweeps = n;
    s.vx = v[0]; s.vy = v[1]; s.vz = v[2];
    s.wx = R[0] * wb[0] + R[1] * wb[1] + R[2] * wb[2];
    s.wy = R[3] * wb[0] + R[4] * wb[1] + R[5] * wb[2];
    s.wz = R[6] * wb[0] + R[7] * wb[1] + R[8] * wb[2];
    return (lam[0] + lam[1]) + (lam[2] + lam[3]) > 0.f;
}

// btPlaneSpace1: two unit tangents of the unit normal n (p is odd in n, q even: the two agents of a pair derive
// the same rows from n and -n)
__device__ __forceinline__ void plane_space(const float* n, float* p, float* q) {
    if (fabsf(n[2]) > 0.7071067811865475f) {
        const float a = n[1] * n[1] + n[2] * n[2];
        const float k = rsqrt_nr(a);
        p[0] = 0.f; p[1] = -n[2] * k; p[2] = n[1] * k;
        q[0] = a * k; q[1] = -n[0] * p[2]; q[2] = n[0] * p[1];
    } else {
        const float a = n[0] * n[0] + n[1] * n[1];
        const float k = rsqrt_nr(a);
        p[0] = -n[1] * k; p[1] = n[0] * k; p[2] = 0.f;
        q[0] = -n[2] * p[1]; q[1] = n[2] * p[0]; q[2] = a * k;
    }
}

// agent-agent rows of one pair as seen from agent `me` (d = p_me - p_partner, dv = v_me - v_partner): updates the
// three accumulated impulses and returns the velocity change of `me` (the partner, evaluating the same rows from
// its side with -d and -dv, gets the exact opposite).  mass-normalised: both agents weigh the same, K = 2 / m.
__device__ __forceinline__ float pair_rows(const ContactParams& cp, float dx, float dy, float dz,
                                           const float* vme, const float* vpt, float* lam3, float* dv_me, bool& active) {
    const float d2 = dx * dx + dy * dy + dz * dz;
    const float inv = rsqrt_nr(fmaxf(d2, 1e-30f));
    const float dist = d2 * inv - 2.f * cp.contact_radius;
    active = (dist < cp.contact_margin) && (d2 > 0.f);
    dv_me[0] = dv_me[1] = dv_me[2] = 0.f;
    if (!active) return 0.f;
    const float n[3] = {dx * inv, dy * inv, dz * inv};
    float t1[3], t2[3];
    plane_space(n, t1, t2);
    const float half_m = 0.5f * cp.mass;
    float rel[3] = {vme[0] - vpt[0], vme[1] - vpt[1], vme[2] - vpt[2]};
    float worst = 0.f;
    // normal row
    {
        const float vr = n[0] * rel[0] + n[1] * rel[1] + n[2] * rel[2];
        const float ln = fmaxf(lam3[0] + (contact_bias(cp, dist) - vr) * half_m, 0.f);
        const float dl = (ln - lam3[0]) * cp.inv_mass;
        lam3[0] = ln;
#pragma unroll
        for (int k = 0; k < 3; ++k) { dv_me[k] += n[k] * dl; rel[k] += 2.f * n[k] * dl; }
        worst = 2.f * fabsf(dl);
    }
    const float lim = cp.mu_agent * lam3[0];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const float* u = r ? t2 : t1;
        const float vr = u[0] * rel[0] + u[1] * rel[1] + u[2] * rel[2];
        const float ln = clampf(lam3[1 + r] - vr * half_m, -lim, lim);
        const float dl = (ln - lam3[1 + r]) * cp.inv_mass;
        lam3[1 + r] = ln;
#pragma unroll
        for (int k = 0; k < 3; ++k) { dv_me[k] += u[k] * dl; rel[k] += 2.f * u[k] * dl; }
        worst = fmaxf(worst, 2.f * fabsf(dl));
    }
    return worst;
}

// round-robin tournament over M = N rounded up to even (bullet_model.tournament_partner): partner of agent i in
// round r (i itself = sits out), and the round in which i < j meet
__device__ __forceinline__ int tour_partner(int r, int i, int N) {
    const int M = N + (N & 1), m1 = M - 1;
    int j;
    if (i == m1) j = r;
    else {
        j = 2 * r - i;
        if (j < 0) j += m1;
        if (j >= m1) j -= m1;
        if (j == i) j = m1;
    }
    return (j >= N) ? i : j;
}
__device__ __forceinline__ int tour_round_small(int i, int j, int N) {    // i < j < N <= 32: 32-bit arithmetic
    const int M = N + (N & 1), m1 = M - 1;
    if (j == m1) return i;
    return ((i + j) * (M / 2)) % m1;
}
__device__ __forceinline__ int tour_round(int i, int j, int N) {          // i < j < N
    const int M = N + (N & 1), m1 = M - 1;
    if (j == m1) return i;
    return (int)(((long long)(i + j) * (M / 2)) % m1);
}

// btMultiBody::stepPositionsMultiDof (bullet_model.integrate_positions): p += dt v; q <- dq (x) q
// with dq = [w sin(x)/|w|, cos(x)], x = |w| dt / 2 <= pi/8.  sin(x)/x and cos(x) are evaluated as
// Taylor polynomials in x^2 = dt^2 |w|^2 / 4 (truncation < 2e-9 relative at the cap), so the
// step needs no sqrt, sincos or division; Bullet's own small-angle Taylor branch is the same
// series.  |w| dt > pi/4 takes Bullet's capped step (constants in Derived).
__device__ __forceinline__ void integrate(const MrsConfig& c, const Derived& d, Agent& s) {
    const float dt = c.dt;
    s.px += dt * s.vx; s.py += dt * s.vy; s.pz += dt * s.vz;
    const float w2 = s.wx * s.wx + s.wy * s.wy + s.wz * s.wz;
    float k, cw;
    if (w2 > d.cap_w2) {
        k = d.cap_k; cw = d.cap_c;
    } else {
        const float x2 = d.q_x2 * w2;
        const float sinc = 1.f + x2 * (-1.f / 6.f + x2 * (1.f / 120.f + x2 * (-1.f / 5040.f + x2 * (1.f / 362880.f))));
        cw = 1.f + x2 * (-0.5f + x2 * (1.f / 24.f + x2 * (-1.f / 720.f + x2 * (1.f / 40320.f + x2 * (-1.f / 3628800.f)))));
        k = 0.5f * dt * sinc;
    }
    const float ax = s.wx * k, ay = s.wy * k, az = s.wz * k;
    // q <- dq (x) q, xyzw
    const float nx = cw * s.qx + ax * s.qw + ay * s.qz - az * s.qy;
    const float ny = cw * s.qy - ax * s.qz + ay * s.qw + az * s.qx;
    const float nz = cw * s.qz + ax * s.qy - ay * s.qx + az * s.qw;
    const float nw = cw * s.qw - ax * s.qx - ay * s.qy - az * s.qz;
    const float n2 = nx * nx + ny * ny + nz * nz + nw * nw;
    float inv = fast_rsqrt(n2);
    inv = inv * (1.5f - 0.5f * n2 * inv * inv);      // one Newton step: full float32 accuracy
    s.qx = nx * inv; s.qy = ny * inv; s.qz = nz * inv; s.qw = nw * inv;
}

// MRS.calc_A pair (MRS.py:117-124), bit-exact with torch CPU float32 norm:
// d = sqrt_rn(fma(dz,dz,fma(dy,dy,dx*dx))), A = d <= COMM_RANGE (NaN -> 0).
// sqrt_rn is monotone, so d <= range  <=>  s <= s_max with s_max the largest float whose
// correctly rounded root is <= range (computed on the host, adjacency_threshold()): the
// comparison is done on the squared distance, bit-identical and without the sqrt.
__device__ __forceinline__ float adjacency_pair(float xi, float yi, float zi, float xj, float yj, float zj, float s_max) {
    const float dx = __fsub_rn(xi, xj), dy = __fsub_rn(yi, yj), dz = __fsub_rn(zi, zj);
    const float s = __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
    return (s <= s_max) ? 1.f : 0.f;
}

// Non-finite state detector.  Position and attitude are where every other component ends up within one step:
// p <- p + dt v (a NaN / inf velocity reaches p at once), q <- normalise(dq(w) (x) q) (a NaN / inf angular velocity
// or one NaN quaternion component makes all four NaN), and the +-100 coordinate clamp keeps finite velocities from
// overflowing p.  So three adds on (p, qw) flag the same trajectories as the 12-add sum over all components, at the
// latest one step later (the status bit is sticky).
__device__ __forceinline__ bool agent_finite(const Agent& s) {
    return isfinite((s.px + s.py) + (s.pz + s.qw));
}

}  // namespace mrs
