// socp_b200/csrc/models.cuh -- device code of the five SOCP models (sm_100a, fp64).
//
// Each model is a struct with
//     DIM, N = 2*DIM, NP (parameter block length), NCTRL
//     struct Ctx     per-trajectory constants held in registers (parameters, switching times,
//                    and -- interceptor -- the chart / stage the reference keeps as hidden
//                    mutable model state, interceptor.cpp:27-29)
//     load(ctx, mparams, sw)            fill Ctx from the parameter block
//     rhs(ctx, t, X, dX)                odeTools::Model  = (dH/dp, -dH/dx) with the PMP control
//     control(ctx, t, X, u)             model::Control
//     hamiltonian(ctx, t, X)            model::Hamiltonian (isJac == 0)
// The formulas restate /root/reference/src/models/*/*.cpp (file:line at each function); common
// subexpressions (1/r, 1/m, exp(-kr(r-1)), sin/cos of the angles) are evaluated once, which
// changes rounding by a few ulp only -- parity is checked to <= 1e-12 against the oracle.
#pragma once
#include <math.h>

namespace socp {

enum { GODDARD = 0, DOUBLE_INTEGRATOR = 1, COVID19 = 2, VTOL_UAV = 3, INTERCEPTOR = 4 };

#define SOCP_MAX_OBS 32
// obstacle table of the vtolUAV penalty map: per obstacle {type, pos[3], rad[3]} (obstacle.cpp:24-36)
__constant__ double c_obstacles[SOCP_MAX_OBS * 7];
__constant__ int c_num_obstacles;

#define SOCP_DEV __device__ __forceinline__

template <int MODEL> struct Model;

// =============================== goddard ======================================================
template <> struct Model<GODDARD> {
    static constexpr int DIM = 7, N = 14, NP = 8, NCTRL = 3, DEFAULT_STEPS = 10;
    static constexpr int MINB = 1;      // CTAs/SM asked of the trajectory kernels: 240 registers, no spills (a cap of 168 costs 30%)
    struct Ctx { double C, b, KD, kr, umax, mu1, mu2, sing, sw0, sw1, half_inv_mu2; };
    // the switching times before the first SwitchingTimesUpdate (goddard.cpp:27-29)
    static constexpr double SW0_GUESS = 0.0227, SW1_GUESS = 0.08;
    SOCP_DEV static void load(Ctx &c, const double *m, const double *sw) {
        c.C = m[0]; c.b = m[1]; c.KD = m[2]; c.kr = m[3]; c.umax = m[4]; c.mu1 = m[5]; c.mu2 = m[6];
        c.sing = m[7];
        c.half_inv_mu2 = 0.5 / c.mu2;     // hoisted out of the RHS: alpha_u = -Switch / 2 / mu2
        c.sw0 = sw ? sw[0] : SW0_GUESS;
        c.sw1 = sw ? sw[1] : SW1_GUESS;
    }

    // goddard.cpp:188-253 (true singular control), expression order of the reference.  Out of line:
    // it is only reached with mu2 == 0 inside the switching window, and inlining its ~600 instructions
    // into every RHS copy of the RK4 loop overflows the instruction cache.  Every operand travels BY VALUE:
    // with pointer arguments (the state array, the context) the caller had to keep both in addressable local
    // memory, and the compiler stored the whole state to the stack in every RHS evaluation for a call that
    // the benchmark workload never makes (mu2 > 0): 60 STL sites, 19.5 % of the LSU bandwidth of the RK4 kernel.
    __device__ __noinline__ static double singular(double b, double C, double KD, double kr,
                                                   double x, double y, double z, double vx, double vy, double vz, double mass,
                                                   double p_x, double p_y, double p_z, double p_vx, double p_vy, double p_vz) {
        double r = sqrt(x * x + y * y + z * z);
        double v = sqrt(vx * vx + vy * vy + vz * vz);
        double rdotv = x * vx + y * vy + z * vz;
        double pvdotv = p_vx * vx + p_vy * vy + p_vz * vz;
        double g = 1 / r / r;
        double norm_pv = sqrt(p_vx * p_vx + p_vy * p_vy + p_vz * p_vz);
        double ex = exp(-kr * (r - 1));
        double D = KD * ex;
        double p_xdot = -kr * KD / mass * v * ex * x / r * pvdotv + g * (p_vx * (1 - 3 * x * x / r / r) / r - p_vy * 3 * x * y / r / r / r - p_vz * 3 * x * z / r / r / r);
        double p_ydot = -kr * KD / mass * v * ex * y / r * pvdotv + g * (-p_vx * 3 * y * x / r / r / r + p_vy * (1 - 3 * y * y / r / r) / r - p_vz * 3 * y * z / r / r / r);
        double p_zdot = -kr * KD / mass * v * ex * z / r * pvdotv + g * (-p_vx * 3 * z * x / r / r / r - p_vy * 3 * z * y / r / r / r + p_vz * (1 - 3 * z * z / r / r) / r);
        double p_vxdot = -p_x + KD / mass * ex * (pvdotv * vx / v + p_vx * v);
        double p_vydot = -p_y + KD / mass * ex * (pvdotv * vy / v + p_vy * v);
        double p_vzdot = -p_z + KD / mass * ex * (pvdotv * vz / v + p_vz * v);
        double prdotdotpv = p_xdot * p_vx + p_ydot * p_vy + p_zdot * p_vz;
        double prdotpvdot = p_x * p_vxdot + p_y * p_vydot + p_z * p_vzdot;
        double prdotpv = p_x * p_vx + p_y * p_vy + p_z * p_vz;
        double pvdotdotv = p_vxdot * vx + p_vydot * vy + p_vzdot * vz;
        double pvdotdotpv = p_vxdot * p_vx + p_vydot * p_vy + p_vzdot * p_vz;
        double vdotg = vx * g * x / r + vy * g * y / r + vz * g * z / r;
        double pvdotg = p_vx * g * x / r + p_vy * g * y / r + p_vz * g * z / r;
        double au = 2 * norm_pv * C / mass * pvdotv + 2 * pvdotv * C / mass * norm_pv
                  - b / mass * (2 * pvdotv * pvdotv + norm_pv * norm_pv * v * v)
                  - b / D * v * prdotpv - C / D * prdotpv / v * pvdotv / norm_pv;
        double bu = -2 * norm_pv * norm_pv * (vdotg + D / mass * v * v * v) + 2 * v * v * pvdotdotpv
                  - 2 * pvdotv * (pvdotg + D / mass * v * pvdotv - pvdotdotv)
                  + b / C * (2 * norm_pv * pvdotv * (vdotg + D / mass * v * v * v) + norm_pv * v * v * (pvdotg + D / mass * v * pvdotv - pvdotdotv) - v * v * pvdotv / norm_pv * pvdotdotpv)
                  - mass / D * kr * rdotv / r * v * prdotpv + mass / D * prdotpv / v * (vdotg + D / mass * v * v * v) - mass / D * v * (prdotdotpv + prdotpvdot);
        return bu / au;
    }

    // goddard.cpp:104-185.  Returns the control and |u| (= min(|alpha_u|, u_max)).
    // |p_v| and 1/|p_v| come from one rsqrt (a sqrt plus a divide otherwise).
    SOCP_DEV static void control_norm(const Ctx &c, double t, const double *X, double minv,
                                      double *u, double &norm_u) {
        double p_vx = X[10], p_vy = X[11], p_vz = X[12], p_mass = X[13];
        double pv2 = p_vx * p_vx + p_vy * p_vy + p_vz * p_vz;
        double pvinv = rsqrt(pv2);
        double norm_pv = pv2 * pvinv;
        double Switch = c.mu1 - c.b * p_mass - c.C * minv * norm_pv;
        double alpha_u = 0.0;
        if (c.mu2 > 0) {
            if (Switch < 0) alpha_u = -Switch * c.half_inv_mu2;
        } else {
            if (t <= c.sw0) alpha_u = 1.0;
            else if (t <= c.sw1)
                alpha_u = (c.sing < 0) ? singular(c.b, c.C, c.KD, c.kr, X[0], X[1], X[2], X[3], X[4], X[5], X[6], X[7], X[8], X[9],
                                                  p_vx, p_vy, p_vz)
                                       : c.sing;
        }
        double a = fabs(alpha_u);
        double scale = -alpha_u * pvinv;            // u = -p_v * alpha_u / |p_v|
        norm_u = a;
        if (a > c.umax) { scale = scale / a * c.umax; norm_u = c.umax; }
        u[0] = p_vx * scale; u[1] = p_vy * scale; u[2] = p_vz * scale;
    }
    SOCP_DEV static void control(const Ctx &c, double t, const double *X, double *u) {
        double nu;
        control_norm(c, t, X, 1.0 / X[6], u, nu);
    }

    // goddard.cpp:48-101
    SOCP_DEV static void rhs(const Ctx &c, double t, const double *X, double *dX) {
        double x = X[0], y = X[1], z = X[2], vx = X[3], vy = X[4], vz = X[5], mass = X[6];
        double p_x = X[7], p_y = X[8], p_z = X[9], p_vx = X[10], p_vy = X[11], p_vz = X[12];
        // r, 1/r and v, 1/v from one rsqrt each (instead of a sqrt and a divide)
        double r2 = x * x + y * y + z * z;
        double rinv = rsqrt(r2);
        double r = r2 * rinv;
        double v2 = vx * vx + vy * vy + vz * vz;
        double vinv = rsqrt(v2);
        double v = v2 * vinv;
        double minv = 1.0 / mass;
        double pvdotv = p_vx * vx + p_vy * vy + p_vz * vz;
        double ex = exp(-c.kr * (r - 1));
        double g = rinv * rinv;                      // normalised gravity 1/r^2
        double u[3], norm_u;
        control_norm(c, t, X, minv, u, norm_u);
        double pvdotu = p_vx * u[0] + p_vy * u[1] + p_vz * u[2];
        double Dm = c.KD * ex * minv;                // KD exp(-kr(r-1)) / m
        double drag = Dm * v;
        double gr = g * rinv;                        // 1/r^3
        double Cm = c.C * minv;
        dX[0] = vx; dX[1] = vy; dX[2] = vz;
        dX[3] = -drag * vx - gr * x + Cm * u[0];
        dX[4] = -drag * vy - gr * y + Cm * u[1];
        dX[5] = -drag * vz - gr * z + Cm * u[2];
        dX[6] = -c.b * norm_u;
        double kd = c.kr * drag * rinv * pvdotv;     // kr KD/m v e^.. pv.v / r
        double xdotpv = x * p_vx + y * p_vy + z * p_vz;
        double w = 3.0 * xdotpv * g;                 // 3 (x.p_v) / r^2
        dX[7] = -kd * x + gr * (p_vx - w * x);
        dX[8] = -kd * y + gr * (p_vy - w * y);
        dX[9] = -kd * z + gr * (p_vz - w * z);
        double pv_v = pvdotv * vinv;
        dX[10] = -p_x + Dm * (pv_v * vx + p_vx * v);
        dX[11] = -p_y + Dm * (pv_v * vy + p_vy * v);
        dX[12] = -p_z + Dm * (pv_v * vz + p_vz * v);
        dX[13] = -Dm * minv * v * pvdotv + Cm * minv * pvdotu;
    }

    // goddard.cpp:256-295
    SOCP_DEV static double hamiltonian(const Ctx &c, double t, const double *X) {
        double x = X[0], y = X[1], z = X[2], vx = X[3], vy = X[4], vz = X[5], mass = X[6];
        double p_x = X[7], p_y = X[8], p_z = X[9], p_vx = X[10], p_vy = X[11], p_vz = X[12], p_mass = X[13];
        double r = sqrt(x * x + y * y + z * z);
        double v = sqrt(vx * vx + vy * vy + vz * vz);
        double ex = exp(-c.kr * (r - 1));
        double g = 1 / r / r;
        double u[3], nu;
        control_norm(c, t, X, 1.0 / mass, u, nu);
        double norm_u = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
        return c.mu1 * norm_u + c.mu2 * norm_u * norm_u + p_x * vx + p_y * vy + p_z * vz
             + p_vx * (-c.KD * v * vx * ex / mass - g * x / r + c.C * u[0] / mass)
             + p_vy * (-c.KD * v * vy * ex / mass - g * y / r + c.C * u[1] / mass)
             + p_vz * (-c.KD * v * vz * ex / mass - g * z / r + c.C * u[2] / mass)
             - p_mass * c.b * norm_u;
    }
};

// =============================== doubleIntegrator =============================================
template <> struct Model<DOUBLE_INTEGRATOR> {
    static constexpr int DIM = 6, N = 12, NP = 3, NCTRL = 3, DEFAULT_STEPS = 30;
    static constexpr int MINB = 1;
    struct Ctx { double umax, amax, muT, iamax; };
    SOCP_DEV static void load(Ctx &c, const double *m, const double *) { c.umax = m[0]; c.amax = m[1]; c.muT = m[2]; c.iamax = 1.0 / c.amax; }
    // doubleIntegrator.cpp:218-259 (u = -p_v / a_max through the hoisted reciprocal; one rsqrt when saturated)
    SOCP_DEV static void control(const Ctx &c, double, const double *X, double *u) {
        u[0] = -X[9] * c.iamax; u[1] = -X[10] * c.iamax; u[2] = -X[11] * c.iamax;
        double nu2 = u[0] * u[0] + u[1] * u[1] + u[2] * u[2];
        if (nu2 > c.umax * c.umax) {
            double k = c.umax * rsqrt(nu2);
            u[0] = u[0] * k; u[1] = u[1] * k; u[2] = u[2] * k;
        }
    }
    // doubleIntegrator.cpp:67-108
    SOCP_DEV static void rhs(const Ctx &c, double t, const double *X, double *dX) {
        double u[3];
        control(c, t, X, u);
        dX[0] = X[3]; dX[1] = X[4]; dX[2] = X[5];
        dX[3] = c.amax * u[0]; dX[4] = c.amax * u[1]; dX[5] = c.amax * u[2];
        dX[6] = 0; dX[7] = 0; dX[8] = 0;
        dX[9] = -X[6]; dX[10] = -X[7]; dX[11] = -X[8];
    }
    // doubleIntegrator.cpp:264-300 (isJac == 0)
    SOCP_DEV static double hamiltonian(const Ctx &c, double t, const double *X) {
        double u[3];
        control(c, t, X, u);
        double nu = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
        return c.muT + c.amax * c.amax * nu * nu / 2 + X[6] * X[3] + X[7] * X[4] + X[8] * X[5]
             + c.amax * (X[9] * u[0] + X[10] * u[1] + X[11] * u[2]);
    }
};

// =============================== covid19 ======================================================
template <> struct Model<COVID19> {
    static constexpr int DIM = 4, N = 8, NP = 8, NCTRL = 1, DEFAULT_STEPS = 1000;
    static constexpr int MINB = 1;
    // The reference divides by Tinf, Tinc and N thirteen times per RHS; an fp64 divide is ~20 pipe
    // instructions (123 cycles of latency), so the three reciprocals are formed once per trajectory and the
    // RHS multiplies (<= 1 ulp per operation, far inside the 1e-12 trajectory tolerance).
    struct Ctx { double R0, Tinf, Tinc, Npop, Imax, muI, umin, umax, iTinf, iTinc, iN; };
    SOCP_DEV static void load(Ctx &c, const double *m, const double *) {
        c.R0 = m[0]; c.Tinf = m[1]; c.Tinc = m[2]; c.Npop = m[3]; c.Imax = m[4]; c.muI = m[5];
        c.umin = m[6]; c.umax = m[7];
        c.iTinf = 1.0 / c.Tinf; c.iTinc = 1.0 / c.Tinc; c.iN = 1.0 / c.Npop;
    }
    // covid19.cpp:98-129
    SOCP_DEV static void control(const Ctx &c, double, const double *X, double *u) {
        double v = (X[5] - X[4]) * X[0] * X[2] * c.iTinf * c.iN * c.R0;
        if (v <= c.umin) v = c.umin;
        if (v >= c.umax) v = c.umax;
        u[0] = v;
    }
    // covid19.cpp:53-95 -- the costate rows use R = X[3] where Rt was presumably meant; kept
    SOCP_DEV static void rhs(const Ctx &c, double t, const double *X, double *dX) {
        double S = X[0], E = X[1], I = X[2], R = X[3], pS = X[4], pE = X[5], pI = X[6], pR = X[7];
        double u;
        control(c, t, X, &u);
        double Rt = c.R0 * (1 - u);
        double Ipen = 0;
        if (I >= c.Imax) Ipen = -c.muI * (I - c.Imax);
        double inf = Rt * c.iTinf * c.iN * S * I;
        double EoT = E * c.iTinc, IoT = I * c.iTinf;
        dX[0] = -inf;
        dX[1] = inf - EoT;
        dX[2] = EoT - IoT;
        dX[3] = IoT;
        dX[4] = (pS - pE) * R * I * c.iTinf * c.iN;
        dX[5] = (pE - pI) * c.iTinc;
        dX[6] = (pS - pE) * R * S * c.iTinf * c.iN + (pI - pR) * c.iTinf + Ipen;
        dX[7] = 0;
    }
    // covid19.cpp:132-168
    SOCP_DEV static double hamiltonian(const Ctx &c, double t, const double *X) {
        double S = X[0], E = X[1], I = X[2], pS = X[4], pE = X[5], pI = X[6], pR = X[7];
        double u;
        control(c, t, X, &u);
        double Rt = c.R0 * (1 - u);
        double Ipen = 0;
        if (I >= c.Imax) Ipen = c.muI * (I - c.Imax) * (I - c.Imax) / 2;
        return u * u / 2 + Ipen + pS * (-Rt / c.Tinf / c.Npop * S * I)
             + pE * (Rt / c.Tinf / c.Npop * S * I - E / c.Tinc) + pI * (E / c.Tinc - I / c.Tinf)
             + pR * (I / c.Tinf);
    }
};

// =============================== vtolUAV + obstacle map =======================================
// obstacle.cpp:155-178 (Function / Gradient; the waypoint terms are commented out there),
// :183-231 (penalty) and :236-316 (gradient; the ellipsoid gradient ignores z, :260-265).
// The sum over the obstacles has ONE canonical order whatever the thread mapping: four partial sums over the
// obstacles i = q (mod 4), combined as (s0 + s2) + (s1 + s3).  One thread per trajectory keeps the four partial
// sums itself; a cooperative group of four lanes per trajectory (coop_lanes == 4: lane q owns the obstacles
// i = q (mod 4), two xor-shuffles combine) produces the same bits, so a trajectory does not depend on which of the
// two kernels integrated it.
struct ObsAcc { double f, g0, g1, g2; };
SOCP_DEV void obstacle_one(int i, double muObs, double imu, const double *pos, bool want_f, bool want_g, ObsAcc &a) {
    const double *o = &c_obstacles[i * 7];
    double type = o[0], x = o[1], y = o[2], z = o[3], radx = o[4], rady = o[5], radz = o[6];
    if (type == 0) {
        double hx = pos[0] - x, hy = pos[1] - y, hz = pos[2] - z;
        double d = sqrt(hx * hx + hy * hy + hz * hz);
        if (want_f) {
            double rad = d / sqrt(hx * hx / radx / radx + hy * hy / rady / rady + hz * hz / radz / radz);
            a.f = a.f + (1 - tanh((d - rad) / muObs)) / 2;
        }
        if (want_g) {
            double sq = sqrt(hx * hx / radx / radx + hy * hy / rady / rady);
            double rad = d / sq;
            double th = tanh((d - rad) / muObs);
            double rho2 = (radx * radx - rady * rady) / (radx * radx * rady * rady) / sq / sq / sq;
            a.g0 = a.g0 - hx / d * (1 - hy * hy * rho2) / muObs * (1 - th * th) / 2;
            a.g1 = a.g1 - hy / d * (1 + hx * hx * rho2) / muObs * (1 - th * th) / 2;
        }
    } else if (type == 1) {
        // box: the nine divides per obstacle of the reference (three "/ muObs" in the tanh arguments and
        // "d / |d| / muObs" in each gradient component) become multiplications by 1/muObs and a sign;
        // d == 0 keeps the reference's 0/0 = NaN (which zeroes the whole component below)
        double dx = pos[0] - x, dy = pos[1] - y, dz = pos[2] - z;
        // 1 - tanh(a) = 2 r and 1 - tanh(a)^2 = 4 r (1 - r) with r = 1 / (1 + exp(2a)): one exp and one
        // reciprocal per axis instead of a library tanh (exp + divide + range logic, ~2x the instructions)
        // and no cancellation in 1 - tanh far inside an obstacle's shadow; exp overflow gives r = 0, the limit
        double rx = 1.0 / (1.0 + exp(2.0 * ((fabs(dx) - radx) * imu)));
        double ry = 1.0 / (1.0 + exp(2.0 * ((fabs(dy) - rady) * imu)));
        double rz = 1.0 / (1.0 + exp(2.0 * ((fabs(dz) - radz) * imu)));
        double ax = 2.0 * rx, ay = 2.0 * ry, az = 2.0 * rz;
        a.f = a.f + ax * ay * az / 8;
        if (want_g) {
            const double nan_ = __longlong_as_double(0x7ff8000000000000LL);
            double sx = (dx == 0.) ? nan_ : copysign(imu, dx), sy = (dy == 0.) ? nan_ : copysign(imu, dy),
                   sz = (dz == 0.) ? nan_ : copysign(imu, dz);
            a.g0 = a.g0 - sx * (4.0 * rx * (1.0 - rx)) * ay * az / 8;
            a.g1 = a.g1 - sy * (4.0 * ry * (1.0 - ry)) * ax * az / 8;
            a.g2 = a.g2 - sz * (4.0 * rz * (1.0 - rz)) * ax * ay / 8;
        }
    }
}

// coop_lanes == 1: this thread evaluates every obstacle; == 4: it is lane `cq` of a group of four (shuffle mask `cmask`)
SOCP_DEV void obstacle_eval(double muObs, double phiObs, const double *pos, double *func, double *grad,
                            int coop_lanes = 1, int cq = 0, unsigned cmask = 0) {
    const double imu = 1.0 / muObs;
    const int n = c_num_obstacles;
    double f, g0, g1, g2;
    if (coop_lanes == 4) {
        ObsAcc a = {0., 0., 0., 0.};
        for (int i = cq; i < n; i += 4) obstacle_one(i, muObs, imu, pos, func != nullptr, grad != nullptr, a);
        f = a.f + __shfl_xor_sync(cmask, a.f, 2); f = f + __shfl_xor_sync(cmask, f, 1);
        g0 = a.g0 + __shfl_xor_sync(cmask, a.g0, 2); g0 = g0 + __shfl_xor_sync(cmask, g0, 1);
        g1 = a.g1 + __shfl_xor_sync(cmask, a.g1, 2); g1 = g1 + __shfl_xor_sync(cmask, g1, 1);
        g2 = a.g2 + __shfl_xor_sync(cmask, a.g2, 2); g2 = g2 + __shfl_xor_sync(cmask, g2, 1);
    } else {
        // the same four partial sums one after the other, in the order 0, 2, 1, 3 (one inlined copy of the
        // obstacle code, twelve live doubles): (s0 + s2) + (s1 + s3)
        ObsAcc acc = {0., 0., 0., 0.}, t02 = acc;
#pragma unroll 1
        for (int k = 0; k < 4; ++k) {
            const int q = ((k & 1) << 1) | (k >> 1);
            ObsAcc a = {0., 0., 0., 0.};
#pragma unroll 1
            for (int i = q; i < n; i += 4) obstacle_one(i, muObs, imu, pos, func != nullptr, grad != nullptr, a);
            if (k == 2) { t02 = acc; acc = a; }
            else if (k == 0) acc = a;
            else { acc.f = acc.f + a.f; acc.g0 = acc.g0 + a.g0; acc.g1 = acc.g1 + a.g1; acc.g2 = acc.g2 + a.g2; }
        }
        f = t02.f + acc.f; g0 = t02.g0 + acc.g0; g1 = t02.g1 + acc.g1; g2 = t02.g2 + acc.g2;
    }
    if (func) *func = phiObs * (isnan(f) ? 0.0 : f);
    if (grad) {
        grad[0] = phiObs * (isnan(g0) ? 0.0 : g0);
        grad[1] = phiObs * (isnan(g1) ? 0.0 : g1);
        grad[2] = phiObs * (isnan(g2) ? 0.0 : g2);
    }
}

template <> struct Model<VTOL_UAV> {
    static constexpr int DIM = 6, N = 12, NP = 13, NCTRL = 3, DEFAULT_STEPS = 100;
    static constexpr int MINB = 4;      // 128 registers, +45% throughput over 1 (occupancy hides the exp chains)
    // coop_lanes / cq / cmask: the thread mapping of the obstacle sum (see obstacle_eval), set by the cooperative kernels
    struct Ctx { double umax, amax, alphaT, alphaV, invSigma, Vd, ca, phiObs, muObs; int coop_lanes, cq; unsigned cmask; };
    SOCP_DEV static void load(Ctx &c, const double *m, const double *) {
        c.umax = m[0]; c.amax = m[1]; c.alphaT = m[2]; c.alphaV = m[3]; c.invSigma = m[4];
        c.Vd = m[5]; c.ca = m[6]; c.phiObs = m[9]; c.muObs = m[11];
        c.coop_lanes = 1; c.cq = 0; c.cmask = 0;
    }
    // vtolUAV.cpp:110-148
    SOCP_DEV static void control(const Ctx &c, double, const double *X, double *u) {
        u[0] = -X[9] / c.amax; u[1] = -X[10] / c.amax; u[2] = -X[11] / c.amax;
        double nu = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
        if (nu > c.umax) {
            u[0] = u[0] / nu * c.umax; u[1] = u[1] / nu * c.umax; u[2] = u[2] / nu * c.umax;
        }
    }
    // vtolUAV.cpp:58-107
    SOCP_DEV static void rhs(const Ctx &c, double t, const double *X, double *dX) {
        double vx = X[3], vy = X[4], vz = X[5];
        double p_x = X[6], p_y = X[7], p_z = X[8], p_vx = X[9], p_vy = X[10], p_vz = X[11];
        double normV = sqrt(vx * vx + vy * vy + vz * vz);
        double u[3], grad[3];
        control(c, t, X, u);
        obstacle_eval(c.muObs, c.phiObs, X, nullptr, grad, c.coop_lanes, c.cq, c.cmask);
        dX[0] = vx; dX[1] = vy; dX[2] = vz;
        dX[3] = c.amax * u[0] - c.ca * vx * normV;
        dX[4] = c.amax * u[1] - c.ca * vy * normV;
        dX[5] = c.amax * u[2] - c.ca * vz * normV;
        dX[6] = 0 - grad[0]; dX[7] = 0 - grad[1]; dX[8] = 0 - grad[2];
        const double iv = 1.0 / normV;                 // one divide instead of twelve
        dX[9] = -p_x + c.ca * (p_vx * (normV + vx * vx * iv) + p_vy * (vy * vx * iv) + p_vz * (vz * vx * iv)) - c.alphaV * vx * iv * (normV - c.Vd);
        dX[10] = -p_y + c.ca * (p_vy * (normV + vy * vy * iv) + p_vx * (vx * vy * iv) + p_vz * (vz * vy * iv)) - c.alphaV * vy * iv * (normV - c.Vd);
        dX[11] = -p_z + c.ca * (p_vz * (normV + vz * vz * iv) + p_vx * (vx * vz * iv) + p_vy * (vy * vz * iv)) - c.alphaV * vz * iv * (normV - c.Vd);
    }
    // vtolUAV.cpp:151-192
    SOCP_DEV static double hamiltonian(const Ctx &c, double t, const double *X) {
        double vx = X[3], vy = X[4], vz = X[5];
        double p_x = X[6], p_y = X[7], p_z = X[8], p_vx = X[9], p_vy = X[10], p_vz = X[11];
        double normV = sqrt(vx * vx + vy * vy + vz * vz);
        double u[3], obs = 0;
        control(c, t, X, u);
        double nu = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
        obstacle_eval(c.muObs, c.phiObs, X, &obs, nullptr, c.coop_lanes, c.cq, c.cmask);
        return c.alphaT * 1 + c.alphaV / 2 * (normV - c.Vd) * (normV - c.Vd) + obs + c.amax * c.amax * nu * nu / 2
             + p_x * vx + p_y * vy + p_z * vz
             + (p_vx * (c.amax * u[0] - c.ca * vx * normV) + p_vy * (c.amax * u[1] - c.ca * vy * normV) + p_vz * (c.amax * u[2] - c.ca * vz * normV));
    }
};

// =============================== interceptor ==================================================
#define SOCP_R_EARTH 6378145.0      // interceptor.cpp:51
#define SOCP_MU0 3.986e14           // interceptor.cpp:52
#define SOCP_CHART_LIMIT 0.1        // interceptor.cpp:57
#define SOCP_PI 3.14159265358979323846

template <> struct Model<INTERCEPTOR> {
    static constexpr int DIM = 6, N = 12, NP = 17, NCTRL = 2, DEFAULT_STEPS = 50;
    static constexpr int MINB = 4;      // 128 registers, +65% throughput over 1 (occupancy hides the sin/cos chains)
    struct Ctx {
        double c0, hr, d0, eta, mprop, mempty, q, ve, alphamax, umax, mugft, muT, muV, muC;
        int chart, stage;
    };
    SOCP_DEV static void load(Ctx &c, const double *m, const double *) {
        c.c0 = m[0]; c.hr = m[1]; c.d0 = m[2]; c.eta = m[3]; c.mprop = m[4]; c.mempty = m[5];
        c.q = m[6]; c.ve = m[7]; c.alphamax = m[8]; c.umax = m[9]; c.mugft = m[13]; c.muT = m[14];
        c.muV = m[15]; c.muC = m[16];
        c.chart = 1; c.stage = 0;
    }
    struct Tmp { double mass, c_max, d, r, g, ft; };
    // the "temporary variables" block (interceptor.cpp:293-306) and ComputeMass (:984-999)
    SOCP_DEV static void common(const Ctx &c, double t, double h, Tmp &k) {
        double qm = c.stage * c.q * c.mugft;
        double qm_mass = c.q * c.mugft;
        double t1 = c.mprop / c.q;
        k.mass = (c.stage == 1) ? c.mempty + c.mprop - qm_mass * t : c.mempty + c.mprop - qm_mass * t1;
        double e = exp(-h / c.hr) * (c.mprop + c.mempty) / k.mass;
        k.c_max = c.c0 * e;
        k.d = c.d0 * e;
        k.r = h + SOCP_R_EARTH;
        k.g = SOCP_MU0 / k.r / k.r * c.mugft;
        k.ft = c.ve * qm;
    }
    // interceptor.cpp:342-389 (chart 1) and :519-566 (chart 2): u and beta, with cos/sin(beta)
    SOCP_DEV static void control_full(const Ctx &c, const Tmp &k, const double *X, double cang,
                                      double &u, double &beta, double &sb, double &cb) {
        double v = X[1], p_v = X[7], p_a = X[8], p_b = X[9];
        double s = (c.chart == 1) ? 1.0 : -1.0;   // chart 2 flips the sign of the p_phi terms
        beta = atan2(s * p_b, p_a * cang);
        sincos(beta, &sb, &cb);
        double am = c.alphamax / k.mass / v;
        u = (p_a * (v * k.c_max * cb + k.ft * cb * am)
             + s * p_b * (v * k.c_max * sb / cang + k.ft * sb / cang * am))
            / (p_v * (2 * c.eta * k.c_max * v * v + k.ft * c.alphamax * c.alphamax / k.mass) - c.muC);
        if (fabs(u) > c.umax) u = c.umax * u / fabs(u);
    }
    SOCP_DEV static void control(const Ctx &c, double t, const double *X, double *ctl) {
        Tmp k;
        common(c, t, X[0], k);
        double u, beta, sb, cb;
        control_full(c, k, X, cos(X[2]), u, beta, sb, cb);
        ctl[0] = u; ctl[1] = beta;
    }

    // interceptor.cpp:275-339 (Model_1) and :445-516 (Model_2)
    SOCP_DEV static void rhs(const Ctx &c, double t, const double *X, double *dX) {
        double h = X[0], v = X[1], p_h = X[6], p_v = X[7], p_L = X[10], p_l = X[11];
        Tmp k;
        common(c, t, h, k);
        double mass = k.mass, c_max = k.c_max, d = k.d, r = k.r, g = k.g, ft = k.ft, eta = c.eta, hr = c.hr;
        double sL, cL;
        sincos(X[4], &sL, &cL);
        // one reciprocal per denominator (r, v, mass, cos(L), hr, cos(gamma) / cos(theta)) instead of the ~45
        // divides per RHS of the formulas as written
        const double ir = 1.0 / r, iv = 1.0 / v, im = 1.0 / mass, icL = 1.0 / cL, ihr = 1.0 / hr;
        double tL = sL * icL;
        double u, beta, sb, cb;
        if (c.chart == 1) {
            double p_gamma = X[8], p_chi = X[9];
            double sg, cg, sc, cc;
            sincos(X[2], &sg, &cg);
            sincos(X[3], &sc, &cc);
            const double icg = 1.0 / cg;
            control_full(c, k, X, cg, u, beta, sb, cb);
            double sa, ca;
            sincos(c.alphamax * u, &sa, &ca);
            double dd = d + eta * c_max * u * u;
            dX[0] = v * sg;
            dX[1] = -dd * v * v - g * sg + ft * ca * im;
            dX[2] = v * c_max * u * cb - g * iv * cg + ft * sa * cb * im * iv + v * cg * ir;
            dX[3] = v * c_max * u * sb * icg + ft * sa * sb * icg * im * iv + v * cg * tL * sc * ir;
            dX[4] = v * cg * cc * ir;
            dX[5] = v * cg * sc * icL * ir;
            dX[6] = -p_v * ihr * dd * v * v - 2 * g * ir * (p_gamma * iv * cg + p_v * sg)
                  + p_L * v * cg * cc * ir * ir + p_gamma * v * cg * ir * ir + p_gamma * v * c_max * u * cb * ihr
                  + p_l * v * cg * sc * icL * ir * ir + p_chi * v * cg * tL * sc * ir * ir + p_chi * v * c_max * u * sb * icg * ihr;
            dX[7] = -(p_L * cg * cc * ir + p_l * cg * sc * icL * ir + p_h * sg
                      + p_gamma * (c_max * u * cb + g * iv * iv * cg - ft * sa * cb * im * iv * iv + cg * ir)
                      + p_chi * (c_max * u * sb * icg - ft * sa * sb * icg * im * iv * iv + cg * tL * sc * ir)
                      - p_v * 2 * dd * v);
            dX[8] = v * (p_L * sg * cc * ir + p_l * sg * sc * icL * ir - p_h * cg)
                  - g * (p_gamma * iv * sg - p_v * cg)
                  + p_gamma * v * sg * ir + p_chi * v * sg * tL * sc * ir
                  - p_chi * (v * c_max * u * sb + ft * sa * sb * im * iv) * sg * icg * icg;
            dX[9] = v * (p_L * cg * sc * ir - p_l * cg * cc * icL * ir - p_chi * cg * tL * cc * ir);
            dX[10] = -p_l * v * cg * sc * sL * icL * icL * ir - p_chi * v * cg * (1 + tL * tL) * sc * ir;
            dX[11] = 0.0;
        } else {
            double p_theta = X[8], p_phi = X[9];
            double st, ct, sp, cp;
            sincos(X[2], &st, &ct);
            sincos(X[3], &sp, &cp);
            const double ict = 1.0 / ct;
            double tt = st * ict;
            control_full(c, k, X, ct, u, beta, sb, cb);
            double sa, ca;
            sincos(c.alphamax * u, &sa, &ca);
            double dd = d + eta * c_max * u * u;
            double w1 = cp + sp * tL;                       // cos(phi) + sin(phi) tan(L)
            double w2 = sp + tt * tt * (sp - tL * cp);      // sin(phi) + tan^2(theta)(sin(phi) - tan(L) cos(phi))
            dX[0] = -v * ct * cp;
            dX[1] = -dd * v * v + g * ct * cp + ft * ca * im;
            dX[2] = v * c_max * u * cb + v * st * w1 * ir + (ft * sa * cb * (im * iv) - g * st * cp * iv);
            dX[3] = -v * c_max * u * sb * ict + v * ct * w2 * ir - (ft * sa * sb * (im * iv * ict) + g * sp * (iv * ict));
            dX[4] = v * ct * sp * ir;
            dX[5] = v * st * (ir * icL);
            dX[6] = -p_v * ihr * dd * v * v - 2 * g * ir * (p_theta * st * cp * iv + p_phi * sp * ict * iv - p_v * ct * cp)
                  + p_L * v * ct * sp * ir * ir + v * p_theta * st * w1 * ir * ir + p_theta * v * c_max * u * cb * ihr
                  + p_l * v * st * icL * ir * ir + v * p_phi * ct * w2 * ir * ir - p_phi * v * c_max * u * sb * ict * ihr;
            dX[7] = -(p_L * ct * sp * ir + p_l * st * (ir * icL) - p_h * ct * cp
                      + p_theta * (c_max * u * cb + g * iv * iv * st * cp - ft * sa * cb * im * iv * iv + st * w1 * ir)
                      + p_phi * (-c_max * u * sb * ict + g * iv * iv * sp * ict + ft * sa * sb * ict * im * iv * iv + ct * w2 * ir)
                      - p_v * 2 * dd * v);
            dX[8] = -v * (-p_L * st * sp * ir + p_l * ct * (ir * icL) + p_h * st * cp)
                  - g * (-p_theta * ct * cp * iv - p_phi * sp * tt * (iv * ict) - p_v * st * cp)
                  - p_theta * v * ct * w1 * ir + p_phi * v * st * w2 * ir
                  - p_phi * v * ct * (2 * tt * (1 + tt * tt) * (sp - tL * cp)) * ir
                  - p_phi * (-v * c_max * u * sb - ft * sa * sb * im * iv) * tt * ict;
            dX[9] = -v * (p_h * ct * sp + p_L * ct * cp * ir)
                  - g * (p_theta * st * sp * iv - p_phi * cp * (iv * ict) - p_v * ct * sp)
                  - p_theta * (v * st * (-sp + cp * tL) * ir)
                  - p_phi * v * ct * (cp + tt * tt * (cp + tL * sp)) * ir;
            dX[10] = -p_l * v * st * tL * icL * ir - v * (1 + tL * tL) * (p_theta * st * sp - p_phi * ct * cp * tt * tt) * ir;
            dX[11] = 0.0;
        }
    }

    // interceptor.cpp:392-442 (Hamiltonian_1) and :569-619 (Hamiltonian_2)
    SOCP_DEV static double hamiltonian(const Ctx &c, double t, const double *X) {
        double h = X[0], v = X[1], p_h = X[6], p_v = X[7], p_a = X[8], p_b = X[9], p_L = X[10], p_l = X[11];
        Tmp k;
        common(c, t, h, k);
        double mass = k.mass, c_max = k.c_max, d = k.d, r = k.r, g = k.g, ft = k.ft, eta = c.eta;
        double sL, cL, s2, c2, s3, c3;
        sincos(X[4], &sL, &cL);
        sincos(X[2], &s2, &c2);
        sincos(X[3], &s3, &c3);
        double tL = sL / cL;
        double u, beta, sb, cb;
        control_full(c, k, X, c2, u, beta, sb, cb);
        double sa, ca;
        sincos(c.alphamax * u, &sa, &ca);
        if (c.chart == 1) {
            return p_L * v * c2 * c3 / r + p_l * v * c2 * s3 / cL / r + p_h * v * s2
                 + p_a * (v * c_max * u * cb - g / v * c2 + ft * sa * cb / mass / v + v * c2 / r)
                 + p_b * (v * c_max * u * sb / c2 + ft * sa * sb / c2 / mass / v + v * c2 * tL * s3 / r)
                 - p_v * ((d + eta * c_max * u * u) * v * v + g * s2 - ft * ca / mass)
                 + c.muC * u * u / 2;
        }
        double tt = s2 / c2;
        return p_L * v * c2 * s3 / r + p_l * v * s2 / (r * cL) - p_h * v * c2 * c3
             + p_a * (v * c_max * u * cb + v * s2 * (c3 + s3 * tL) / r + (ft * sa * cb / (mass * v) - g * s2 * c3 / v))
             + p_b * (-v * c_max * u * sb / c2 + v * c2 * (s3 + tt * tt * (s3 - tL * c3)) / r - (ft * sa * sb / (mass * v * c2) + g * s3 / (v * c2)))
             - p_v * ((d + eta * c_max * u * u) * v * v - g * c2 * c3 - ft * ca / mass)
             + c.muC * u * u / 2;
    }

    // ---- chart handling (interceptor.cpp:622-841, 958-981) ----------------------------------
    // Jacobians of the Cartesian embedding wrt chart 1 (gamma, chi) / chart 2 (theta, phi)
    SOCP_DEV static void jac(int chart, double J[6][6], double L, double l, double r, double v, double a, double b) {
        double sL, cL, sl, cl, sa, ca, sb, cb;
        sincos(L, &sL, &cL); sincos(l, &sl, &cl); sincos(a, &sa, &ca); sincos(b, &sb, &cb);
        J[0][0] = cL * cl; J[1][0] = -r * sL * cl; J[2][0] = -r * cL * sl; J[3][0] = 0; J[4][0] = 0; J[5][0] = 0;
        J[0][1] = cL * sl; J[1][1] = -r * sL * sl; J[2][1] = r * cL * cl; J[3][1] = 0; J[4][1] = 0; J[5][1] = 0;
        J[0][2] = sL; J[1][2] = r * cL; J[2][2] = 0; J[3][2] = 0; J[4][2] = 0; J[5][2] = 0;
        J[0][3] = 0; J[0][4] = 0; J[0][5] = 0; J[2][5] = 0;
        if (chart == 1) {       // a = gamma, b = chi
            J[1][3] = (-cL * cl * ca * cb - sL * cl * sa) * v;
            J[2][3] = (sL * sl * ca * cb - cl * ca * sb - cL * sl * sa) * v;
            J[3][3] = (sL * cl * sa * cb + sl * sa * sb + cL * cl * ca) * v;
            J[4][3] = (sL * cl * ca * sb - sl * ca * cb) * v;
            J[5][3] = (-sL * cl * ca * cb - sl * ca * sb + cL * cl * sa) * v;
            J[1][4] = (-cL * sl * ca * cb - sL * sl * sa) * v;
            J[2][4] = (-sL * cl * ca * cb - sl * ca * sb + cL * cl * sa) * v;
            J[3][4] = (sL * sl * sa * cb - cl * sa * sb + cL * sl * ca) * v;
            J[4][4] = (sL * sl * ca * sb + cl * ca * cb) * v;
            J[5][4] = (-sL * sl * ca * cb + cl * ca * sb + cL * sl * sa) * v;
            J[1][5] = (-sL * ca * cb + cL * sa) * v;
            J[3][5] = (-cL * sa * cb + sL * ca) * v;
            J[4][5] = -cL * ca * sb * v;
            J[5][5] = (cL * ca * cb + sL * sa) * v;
        } else {                // a = theta, b = phi
            J[1][3] = (-cL * cl * ca * sb + sL * cl * ca * cb) * v;
            J[2][3] = (sL * sl * ca * sb - cl * sa + cL * sl * ca * cb) * v;
            J[3][3] = (sL * cl * sa * sb - sl * ca + cL * cl * sa * cb) * v;
            J[4][3] = (-sL * cl * ca * cb + cL * cl * ca * sb) * v;
            J[5][3] = (-sL * cl * ca * sb - sl * sa - cL * cl * ca * cb) * v;
            J[1][4] = (-cL * sl * ca * sb + sL * sl * ca * cb) * v;
            J[2][4] = (-sL * cl * ca * sb - sl * sa - cL * cl * ca * cb) * v;
            J[3][4] = (sL * sl * sa * sb + cl * ca + cL * sl * sa * cb) * v;
            J[4][4] = (-sL * sl * ca * cb + cL * sl * ca * sb) * v;
            J[5][4] = (-sL * sl * ca * sb + cl * sa - cL * sl * ca * cb) * v;
            J[1][5] = (-sL * ca * sb - cL * ca * cb) * v;
            J[3][5] = (-cL * sa * sb + sL * sa * cb) * v;
            J[4][5] = (cL * ca * cb + sL * ca * sb) * v;
            J[5][5] = (cL * ca * sb - sL * ca * cb) * v;
        }
    }
    // 6x6 partial-pivot LU solve (stands in for Eigen's lu().solve(), interceptor.cpp:715,829)
    __device__ static void lu6_solve(double A[6][6], const double *b, double *x) {
        int piv[6];
        for (int i = 0; i < 6; ++i) piv[i] = i;
        for (int k = 0; k < 6; ++k) {
            int pr = k;
            double best = fabs(A[k][k]);
            for (int i = k + 1; i < 6; ++i)
                if (fabs(A[i][k]) > best) { best = fabs(A[i][k]); pr = i; }
            if (pr != k) {
                for (int j = 0; j < 6; ++j) { double t = A[k][j]; A[k][j] = A[pr][j]; A[pr][j] = t; }
                int ti = piv[k]; piv[k] = piv[pr]; piv[pr] = ti;
            }
            for (int i = k + 1; i < 6; ++i) {
                A[i][k] /= A[k][k];
                for (int j = k + 1; j < 6; ++j) A[i][j] -= A[i][k] * A[k][j];
            }
        }
        double y[6];
        for (int i = 0; i < 6; ++i) y[i] = b[piv[i]];
        for (int i = 0; i < 6; ++i)
            for (int j = 0; j < i; ++j) y[i] -= A[i][j] * y[j];
        for (int i = 5; i >= 0; --i) {
            for (int j = i + 1; j < 6; ++j) y[i] -= A[i][j] * y[j];
            y[i] /= A[i][i];
        }
        for (int i = 0; i < 6; ++i) x[i] = y[i];
    }
    // ConversionState12 (from == 1) / ConversionState21 (from == 2), in place
    __device__ static void convert(int from, double *X) {
        const double eps = 1e-18;
        double v = X[1], a = X[2], b = X[3], L = X[4], l = X[5];
        double r = X[0] + SOCP_R_EARTH;
        double na, nb;
        if (from == 1) {                     // (gamma, chi) -> (theta, phi)
            double gamma = a, chi = b;
            if (gamma == SOCP_PI / 2.0) { na = 0; nb = -SOCP_PI; }
            else if (gamma == -SOCP_PI / 2.0) { na = 0; nb = 0; }
            else {
                double sg = sin(gamma), cg = cos(gamma), sc = sin(chi), cc = cos(chi);
                na = acos(sqrt(sg * sg + cg * cg * cc * cc));
                if (cg * sc < 0) na = -na;
                double ct = cos(na);
                double sinPhi = cg * cc / ct;
                if (fabs(sinPhi) < eps && sg / ct < 0) nb = 0;
                else if (fabs(sinPhi) < eps && sg / ct > 0) nb = -SOCP_PI;
                else if (sinPhi > 0) nb = acos(-sg / ct);
                else nb = -acos(-sg / ct);
            }
        } else {                             // (theta, phi) -> (gamma, chi)
            double theta = a, phi = b;
            if (theta == SOCP_PI / 2.0) { na = 0; nb = SOCP_PI / 2.0; }
            else if (theta == -SOCP_PI / 2.0) { na = 0; nb = -SOCP_PI / 2.0; }
            else {
                double st = sin(theta), ct = cos(theta), sp = sin(phi), cp = cos(phi);
                na = acos(sqrt(st * st + ct * ct * sp * sp));
                if (ct * cp > 0) na = -na;
                double cg = cos(na);
                double sinChi = st / cg;
                if (fabs(sinChi) < eps && sp * ct / cg > 0) nb = 0;
                else if (fabs(sinChi) < eps && sp * ct / cg < 0) nb = -SOCP_PI;
                else if (sinChi > 0) nb = acos(sp * ct / cg);
                else nb = -acos(sp * ct / cg);
            }
        }
        double Jf[6][6], Jt[6][6];
        jac(from, Jf, L, l, r, v, a, b);
        jac(3 - from, Jt, L, l, r, v, na, nb);
        double pf[6] = {X[6], X[10], X[11], X[8], X[9], X[7]}, tmp[6], pt[6];
        lu6_solve(Jf, pf, tmp);
        for (int i = 0; i < 6; ++i) {
            double s = 0;
            for (int j = 0; j < 6; ++j) s += Jt[i][j] * tmp[j];
            pt[i] = s;
        }
        X[2] = na; X[3] = nb;
        X[6] = pt[0]; X[7] = pt[5]; X[8] = pt[3]; X[9] = pt[4]; X[10] = pt[1]; X[11] = pt[2];
    }
    // SetChart (interceptor.cpp:958-981)
    SOCP_DEV static void set_chart(Ctx &c, double *X) {
        if (fabs(cos(X[2])) >= SOCP_CHART_LIMIT) return;
        convert(c.chart, X);
        c.chart = 3 - c.chart;
    }
};

}  // namespace socp
