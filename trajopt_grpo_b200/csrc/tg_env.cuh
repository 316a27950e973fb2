// Environment dynamics, rewards and termination for one environment held in
// registers.  R = float (throughput mode) or double (parity mode, the
// reference's numpy float64 state).  In both modes the wrapped action and the
// rotor sums are float32, exactly as the reference's numpy promotion rules
// make them (SURVEY.md s8c "precision facts").
//
// Each Env<KIND> provides
//   S, A                     state/obs and action dims
//   step<R, WRAPPED>(s, a, p, steps_done, bal, reward) -> done
// where `s` is advanced in place, `bal` is the Pendulum balanced-step counter; WRAPPED = the action is
// already the wrapped control (Env._dynamics' argument) instead of the raw policy sample.
#pragma once
#include <type_traits>

#include "tg_common.cuh"

struct EnvParams {
    double dt;
    int max_steps;
    int time_limit_step;
    int balanced_limit;
    // derived from the physical constructor arguments on the host, in Python-float (double) arithmetic and the
    // reference's operation order:
    //   CartPole: k[0] = masscart + masspole, k[1] = masspole * length, k[2] = length, k[3] = gravity, k[4] = masspole
    //   Pendulum: k[0] = 1 / (mass * length**2), k[1] = mass * gravity * length
    double k[5];
};
// validates `env` and derives its EnvParams (tg_rollout.cu)
int tg_fill_env_params(const tg_env_cfg *env, EnvParams *p);

// Calls f(std::integral_constant<int, KIND>()) for the env kind of a validated tg_env_cfg.
template <typename F> auto tg_with_env_kind(int kind, F &&f) {
    switch (kind) {
        case TG_ENV_CARTPOLE: return f(std::integral_constant<int, TG_ENV_CARTPOLE>());
        case TG_ENV_PENDULUM: return f(std::integral_constant<int, TG_ENV_PENDULUM>());
        case TG_ENV_QUADPOLE2D: return f(std::integral_constant<int, TG_ENV_QUADPOLE2D>());
        default: return f(std::integral_constant<int, TG_ENV_QUADPOLE>());
    }
}

template <typename R> struct Mth;
template <> struct Mth<float> {
    static TG_D float atan2(float y, float x) { return atan2f(y, x); }
    static TG_D void sincos(float a, float *s, float *c) { sincosf(a, s, c); }
    static TG_D float sqrt(float a) { return sqrtf(a); }
    static TG_D float abs(float a) { return fabsf(a); }
};
template <> struct Mth<double> {
    static TG_D double atan2(double y, double x) { return ::atan2(y, x); }
    static TG_D void sincos(double a, double *s, double *c) { ::sincos(a, s, c); }
    static TG_D double sqrt(double a) { return ::sqrt(a); }
    static TG_D double abs(double a) { return fabs(a); }
};

TG_D float clip1(float a) { return fminf(fmaxf(a, -1.0f), 1.0f); }
template <typename R> TG_D R clipr(R a, R lo, R hi) { return a < lo ? lo : (a > hi ? hi : a); }
// hover + hover*clip(a) as numpy evaluates it in float32: a rounded product, then a
// rounded sum (no FMA contraction) -- quadrotor_env.py:409-413, 928
TG_D float wrap_hover(float hov, float a) { return __fadd_rn(hov, __fmul_rn(hov, clip1(a))); }

#define TG_G 9.80665

template <int KIND> struct Env;

// ---------------------------------------------------------------------------
// CartPole -- environments/cartpole_env.py:48-49 (_wrap_action), 51-92
// (_dynamics), 138-182 (step)
// ---------------------------------------------------------------------------
template <> struct Env<TG_ENV_CARTPOLE> {
    static constexpr int S = 5, A = 1;
    template <typename R, bool WRAPPED = false>
    static TG_D bool step(R *s, const float *a, const EnvParams &p, int steps_done, int &bal, R &reward) {
        const float u32 = WRAPPED ? a[0] : 5.0f * clip1(a[0]);   // :48-49, float32
        R x = s[0], xd = s[1], sn = s[2], cs = s[3], thd = s[4];
        thd = clipr<R>(thd, (R)-10, (R)10);                      // :58
        const R u = (R)u32;
        const R M = (R)p.k[0], mpl = (R)p.k[1], l = (R)p.k[2], g = (R)p.k[3], mp = (R)p.k[4], dt = (R)p.dt;
        R theta = Mth<R>::atan2(sn, cs);                         // :68
        const R thd2 = thd * thd;
        const R alpha = (g * sn + cs * ((-u - mpl * thd2 * sn) / M)) /
                        (l * ((R)(4.0 / 3.0) - (mp * (cs * cs)) / M));   // :71-73
        const R acc = (u + mpl * (thd2 * sn - alpha * cs)) / M;  // :76
        xd = xd + acc * dt;                                      // :79
        x = x + xd * dt;                                         // :80
        thd = thd + alpha * dt;                                  // :82
        theta = theta + thd * dt;                                // :83
        Mth<R>::sincos(theta, &sn, &cs);
        s[0] = x; s[1] = xd; s[2] = sn; s[3] = cs; s[4] = thd;
        // reward (:158-167): the list's last two items are one expression (missing comma)
        const R theta_cost = -(cs * cs * cs);
        const R thd_cost = thd * thd;
        const float e_act = 0.001f * (u32 * u32);                // float32 (:165)
        const R term3 = -((R)20 * theta_cost - (R)20) * ((R)1 / ((R)1 + (R)2 * thd_cost)) - (R)e_act;
        R r = dt * ((((R)-5 * (x * x)) + ((R)-0.5 * (xd * xd))) + term3);
        const bool oob = Mth<R>::abs(x) > (R)1;                  // :168
        if (Mth<R>::abs(x) < (R)0.1 && cs > (R)0.95 && Mth<R>::abs(thd) < (R)0.1)   // :173
            r = r + (R)(100.0 * p.dt);
        if (oob) r = r - (R)50;                                  // :179-180
        reward = r;
        return oob || (steps_done + 1 >= p.time_limit_step);     // :168 (_time > max_time)
    }
};

// ---------------------------------------------------------------------------
// Pendulum -- environments/pendulum_env.py:45-46, 48-75, 125-162
// ---------------------------------------------------------------------------
template <> struct Env<TG_ENV_PENDULUM> {
    static constexpr int S = 3, A = 1;
    template <typename R, bool WRAPPED = false>
    static TG_D bool step(R *s, const float *a, const EnvParams &p, int steps_done, int &bal, R &reward) {
        const float u32 = WRAPPED ? a[0] : clip1(a[0]);          // :45-46
        R sn = s[0], cs = s[1], thd = s[2];
        const R dt = (R)p.dt;
        thd = clipr<R>(thd, (R)-10, (R)10);                      // :57
        R theta = Mth<R>::atan2(sn, cs);                         // :59
        R s0, c0;
        Mth<R>::sincos(theta, &s0, &c0);                         // np.sin(theta) (:61)
        const R alpha = (R)p.k[0] * ((R)u32 - (R)p.k[1] * s0);   // :61
        thd = thd + alpha * dt;                                  // :63
        theta = theta + thd * dt;                                // :64
        Mth<R>::sincos(theta, &sn, &cs);
        s[0] = sn; s[1] = cs; s[2] = thd;
        bal = (cs <= (R)-0.99) ? bal + 1 : 0;                    // :138
        const float e_act = -(0.001f * (u32 * u32));             // float32 (:147)
        R r = dt * ((((R)-10 * Mth<R>::sqrt(Mth<R>::abs((R)-1 - cs))) + ((R)-0.1 * (thd * thd))) + (R)e_act);
        if (bal > 0) r = r + (R)1;                               // :150-151
        reward = r;
        return (steps_done + 1 >= p.time_limit_step) || (bal >= p.balanced_limit);  // :154-155
    }
};

// ---------------------------------------------------------------------------
// QuadPole2D -- environments/quadrotor_env.py:912-928, 1044-1130, 1132-1223
// ---------------------------------------------------------------------------
template <> struct Env<TG_ENV_QUADPOLE2D> {
    static constexpr int S = 10, A = 2;
    template <typename R, bool WRAPPED = false>
    static TG_D bool step(R *s, const float *a, const EnvParams &p, int steps_done, int &bal, R &reward) {
        const float hov = (float)((1.5 + 0.5) * TG_G / 2);       // :895
        const float u1 = WRAPPED ? a[0] : wrap_hover(hov, a[0]);   // :928 (float32 mul then add, unfused)
        const float u2 = WRAPPED ? a[1] : wrap_hover(hov, a[1]);
        R x = s[0], z = s[1], vx = s[2], vz = s[3], sth = s[4], cth = s[5], thd = s[6];
        R sph = s[7], cph = s[8], phd = s[9];
        const R mq = (R)1.5, mp = (R)0.5, Lp = (R)0.75, g = (R)TG_G, dt = (R)p.dt;
        const R F = (R)(u2 + u1);                                // :1088 float32 add
        const R M = mq + mp;
        const float ddth32 = (float)(0.5 / 0.4) * (u2 - u1);     // :1093 stays float32 (NEP 50)
        const R ddph = -F * (sph * cth - sth * cph) / (mq * Lp); // :1097
        const R ddx = (-sth * F - (mp * Lp) * cph * ddph + (mp * Lp) * sph * (phd * phd)) / M;          // :1101
        const R ddz = (cth * F - M * g - (mp * Lp) * sph * ddph - (mp * Lp) * cph * (phd * phd)) / M;   // :1104
        const R vxn = vx + ddx * dt, vzn = vz + ddz * dt;        // :1108-1109
        const R thdn = thd + (R)(ddth32 * (float)p.dt);          // :1110 (float32 product)
        const R phdn = phd + ddph * dt;
        const R xn = x + vxn * dt, zn = z + vzn * dt;            // :1114-1115
        const R th = Mth<R>::atan2(sth, cth);                    // :1119 -- advances with the OLD rate
        const R ph = Mth<R>::atan2(sph, cph);
        Mth<R>::sincos(th + thd * dt, &sth, &cth);
        Mth<R>::sincos(ph + phd * dt, &sph, &cph);
        s[0] = xn; s[1] = zn; s[2] = vxn; s[3] = vzn; s[4] = sth; s[5] = cth; s[6] = thdn;
        s[7] = sph; s[8] = cph; s[9] = phdn;
        const R pos_cost = (Mth<R>::abs(xn) + Mth<R>::abs(zn)) + (xn * xn + zn * zn);   // :1186
        const R vel_cost = vxn * vxn + vzn * vzn;
        const R theta_cost = (R)1 - Mth<R>::abs(cth);
        const R omega_cost = thdn * thdn;
        const R phi_cost = cph * cph * cph;
        const R phd_cost = phdn * phdn;
        R r = dt * ((((((R)-15 * pos_cost) + ((R)-0.5 * vel_cost)) + ((R)-5 * theta_cost)) + ((R)-5 * omega_cost)) +
                    (-((R)25 * phi_cost - (R)25) * ((R)1 / ((R)1 + (R)5 * phd_cost))));  // :1194-1201
        if (Mth<R>::sqrt(xn * xn + zn * zn) < (R)0.25 && cph < (R)-0.95 && Mth<R>::abs(phdn) < (R)0.1)
            r = r + (R)(100.0 * p.dt);                           // :1204-1206
        const bool oob = xn < (R)-2 || xn > (R)2 || zn < (R)-2 || zn > (R)2;   // :1020-1022
        if (oob) r = r - (R)(1000.0 * p.dt);                     // :1215-1217
        reward = r;
        return oob || (steps_done + 1 >= p.max_steps);           // :1220
    }
};

// ---------------------------------------------------------------------------
// QuadPole (3-D quadrotor + slung payload, quaternions) --
// environments/quadrotor_env.py:190-228 (quaternion helpers), 409-413, 417-528, 625-713
// ---------------------------------------------------------------------------
template <typename R> struct Q4 { R w, x, y, z; };
template <typename R> TG_D Q4<R> qmul(const Q4<R> &q, const Q4<R> &r) {   // :190-202
    Q4<R> o;
    o.w = q.w * r.w - q.x * r.x - q.y * r.y - q.z * r.z;
    o.x = q.w * r.x + q.x * r.w + q.y * r.z - q.z * r.y;
    o.y = q.w * r.y - q.x * r.z + q.y * r.w + q.z * r.x;
    o.z = q.w * r.z + q.x * r.y - q.y * r.x + q.z * r.w;
    return o;
}

template <> struct Env<TG_ENV_QUADPOLE> {
    static constexpr int S = 20, A = 4;
    template <typename R, bool WRAPPED = false>
    static TG_D bool step(R *s, const float *a, const EnvParams &p, int steps_done, int &bal, R &reward) {
        const float hov = (float)((1.5 + 0.5) * TG_G / 4);       // :376
        const float u1 = WRAPPED ? a[0] : wrap_hover(hov, a[0]), u2 = WRAPPED ? a[1] : wrap_hover(hov, a[1]);   // :409-413
        const float u3 = WRAPPED ? a[2] : wrap_hover(hov, a[2]), u4 = WRAPPED ? a[3] : wrap_hover(hov, a[3]);
        const R ut = (R)(((u1 + u2) + u3) + u4);                 // :442 float32 adds
        const R m0 = (R)1.5, mp = (R)0.5, L = (R)0.5, arm = (R)0.5;
        const R Ixx = (R)0.4, Iyy = (R)0.4, Izz = (R)0.25, g = (R)TG_G, dt = (R)p.dt;
        const R q0 = s[6], q1 = s[7], q2 = s[8], q3 = s[9];
        const R om0 = s[10], om1 = s[11], om2 = s[12];
        const Q4<R> qp = {s[13], s[14], s[15], s[16]};
        const R op0 = s[17], op1 = s[18], op2 = s[19];
        // thrust in the inertial frame = third column of R(q) times u_total (:208-215, :461-464)
        const R F0 = (R)2 * (q1 * q3 + q0 * q2) * ut;
        const R F1 = (R)2 * (q2 * q3 - q0 * q1) * ut;
        const R F2 = ((R)1 - (R)2 * (q1 * q1 + q2 * q2)) * ut;
        // tether direction = rotate_vector(q_p, [0,0,-1]) (:217-224, :468)
        const Q4<R> v = {(R)0, (R)0, (R)0, (R)-1};
        const Q4<R> t = qmul(qp, v);
        const Q4<R> qc = {qp.w, -qp.x, -qp.y, -qp.z};
        const Q4<R> rot = qmul(t, qc);
        const R t0 = rot.x, t1 = rot.y, t2 = rot.z;
        const R ud0 = op1 * t2 - op2 * t1, ud1 = op2 * t0 - op0 * t2, ud2 = op0 * t1 - op1 * t0;   // :471
        const R nrm = Mth<R>::sqrt(ud0 * ud0 + ud1 * ud1 + ud2 * ud2);
        const R Fdot = F0 * t0 + F1 * t1 + F2 * t2;
        const R Tn = mp / (m0 + mp) * (Fdot - m0 * L * (nrm * nrm));   // :474
        const R gz = -g;
        const R inv_m0 = (R)1 / m0;
        const R a0 = inv_m0 * (m0 * (R)0 + F0 - Tn * t0);        // :478
        const R a1 = inv_m0 * (m0 * (R)0 + F1 - Tn * t1);
        const R a2 = inv_m0 * (m0 * gz + F2 - Tn * t2);
        const R v0 = s[3] + a0 * dt, v1 = s[4] + a1 * dt, v2 = s[5] + a2 * dt;   // :481
        const R p0 = s[0] + v0 * dt, p1 = s[1] + v1 * dt, p2 = s[2] + v2 * dt;   // :482
        const R r2h = (R)0.70710678118654757;                    // np.sqrt(2)/2
        const R tau_x = r2h * (R)(((u1 + u3) - u2) - u4) * arm - (Izz - Iyy) * om1 * om2;   // :485
        const R tau_y = r2h * (R)(((u3 + u4) - u1) - u2) * arm - (Izz - Ixx) * om0 * om2;   // :486
        const R tau_z = (R)(0.1f * (((u1 + u4) - u2) - u3));     // :487 float32 product (NEP 50)
        const R J0 = Ixx * om0, J1 = Iyy * om1, J2 = Izz * om2;
        const R c0 = om1 * J2 - om2 * J1, c1 = om2 * J0 - om0 * J2, c2 = om0 * J1 - om1 * J0;   // :492
        const R on0 = om0 + ((tau_x - c0) / Ixx) * dt;           // :493-498
        const R on1 = om1 + ((tau_y - c1) / Iyy) * dt;
        const R on2 = om2 + ((tau_z - c2) / Izz) * dt;
        const Q4<R> q = {q0, q1, q2, q3};
        const Q4<R> w = {(R)0, on0, on1, on2};
        const Q4<R> qd = qmul(q, w);                             // :502
        R n0 = q0 + (R)0.5 * qd.w * dt, n1 = q1 + (R)0.5 * qd.x * dt;
        R n2 = q2 + (R)0.5 * qd.y * dt, n3 = q3 + (R)0.5 * qd.z * dt;
        R nn = Mth<R>::sqrt(n0 * n0 + n1 * n1 + n2 * n2 + n3 * n3);   // :504
        n0 = n0 / nn; n1 = n1 / nn; n2 = n2 / nn; n3 = n3 / nn;
        // payload: cross(L*u, T*u + g*m_p) / (m_p L^2) (:509)
        const R A0 = L * t0, A1 = L * t1, A2 = L * t2;
        const R B0 = Tn * t0 + (R)0 * mp, B1 = Tn * t1 + (R)0 * mp, B2 = Tn * t2 + gz * mp;
        const R den = mp * (L * L);
        const R pn0 = op0 + ((A1 * B2 - A2 * B1) / den) * dt;
        const R pn1 = op1 + ((A2 * B0 - A0 * B2) / den) * dt;
        const R pn2 = op2 + ((A0 * B1 - A1 * B0) / den) * dt;
        const Q4<R> wp = {(R)0, pn0, pn1, pn2};
        const Q4<R> qpd = qmul(wp, qp);                          // :513 (left multiplication)
        R m0_ = qp.w + (R)0.5 * qpd.w * dt, m1_ = qp.x + (R)0.5 * qpd.x * dt;
        R m2_ = qp.y + (R)0.5 * qpd.y * dt, m3_ = qp.z + (R)0.5 * qpd.z * dt;
        nn = Mth<R>::sqrt(m0_ * m0_ + m1_ * m1_ + m2_ * m2_ + m3_ * m3_);
        m0_ = m0_ / nn; m1_ = m1_ / nn; m2_ = m2_ / nn; m3_ = m3_ / nn;
        s[0] = p0; s[1] = p1; s[2] = p2; s[3] = v0; s[4] = v1; s[5] = v2;
        s[6] = n0; s[7] = n1; s[8] = n2; s[9] = n3; s[10] = on0; s[11] = on1; s[12] = on2;
        s[13] = m0_; s[14] = m1_; s[15] = m2_; s[16] = m3_; s[17] = pn0; s[18] = pn1; s[19] = pn2;
        // reward (:668-697): strict left-to-right sum of 7 terms
        const R thq = (R)1 - Mth<R>::abs(n0), thp = (R)1 - Mth<R>::abs(m0_);
        const R cpos = p0 * p0 + p1 * p1 + p2 * p2;
        const R cvel = (v0 * v0 + v1 * v1) + v2 * v2;
        const R cqr = (on0 * on0 + on1 * on1) + on2 * on2;
        const R cpr = (pn0 * pn0 + pn1 * pn1) + pn2 * pn2;
        R tot = (R)1 + (R)5 / ((R)1 + (R)10 * cpos);
        tot = tot + (R)10 / ((R)1 + (R)10 * cvel);
        tot = tot + (R)0.1 / ((R)1 + thq * thq);
        tot = tot + (R)5 / ((R)1 + cqr);
        tot = tot + (R)10 / ((R)1 + (R)10 * (thp * thp));
        tot = tot + (R)1 / ((R)1 + (R)10 * cpr);
        R r = dt * tot;
        const bool oob = p0 < (R)-1.5 || p0 > (R)1.5 || p1 < (R)-1.5 || p1 > (R)1.5 || p2 < (R)-1.5 || p2 > (R)1.5;
        if (oob) r = r - (R)(10000.0 * p.dt);                    // :703-704
        reward = r;
        return oob || (steps_done + 1 >= p.max_steps);           // :708
    }
};

// Quadrotor._dynamics -- quadrotor_env.py:113-169 (12-state, explicit Euler;
// R[2][1] reproduced as written).  Controls are taken as given (no wrapping).
template <typename R> TG_D void quadrotor12_step(R *s, const R *u, R dt) {
    const R mass = 1, arm = (R)0.2, Ixx = (R)0.005, Iyy = (R)0.005, Izz = (R)0.006, kt = (R)0.017, g = (R)TG_G;
    const R ut = ((u[0] + u[1]) + u[2]) + u[3];
    R sphi, cphi, sth, cth;
    Mth<R>::sincos(s[6], &sphi, &cphi);
    Mth<R>::sincos(s[7], &sth, &cth);
    const R ax = (R)1 / mass * ((-sth) * ut + (R)0);
    const R ay = (R)1 / mass * ((sphi * cth) * ut + (R)0);
    const R az = (R)1 / mass * ((cphi * cth) * ut + (-mass * g));
    const R tth = sth / cth;
    const R pp = s[9], qq = s[10], rr = s[11];
    const R e0 = (pp + sphi * tth * qq) + cphi * tth * rr;
    const R e1 = ((R)0 * pp + cphi * qq) + (-sphi) * rr;
    const R e2 = ((R)0 * pp + sphi / cth * qq) + cphi / cth * rr;
    const R r2h = (R)0.70710678118654757;
    const R al0 = (r2h * (((u[0] + u[2]) - u[1]) - u[3]) * arm - (Izz - Iyy) * qq * rr) / Ixx;
    const R al1 = (r2h * (((u[2] + u[3]) - u[0]) - u[1]) * arm - (Izz - Ixx) * pp * rr) / Iyy;
    const R al2 = (kt * (((u[0] + u[3]) - u[1]) - u[2])) / Izz;
    const R rates[12] = {s[3], s[4], s[5], ax, ay, az, e0, e1, e2, al0, al1, al2};
#pragma unroll
    for (int i = 0; i < 12; ++i) s[i] = s[i] + rates[i] * dt;
}
