// Device-side synthetic state generation (one state per thread), hand-written.
// Counter-based Philox4x32-10 keyed by the seed and indexed by the GLOBAL state index, so every
// GPU generates its own shard and the union is independent of the GPU count.
// Value ranges follow the reference's generators:
//   ClusterJoints::Base::randomJointState        src/Dynamics/ClusterJoints/ClusterJoint.cpp:74-81
//   ClusterJoints::Free::randomJointState        FreeJoint.cpp:49-60 (rpy -> quaternion,
//                                                include/grbda/Utils/OrientationTools.h:160-199,293-300)
//   ClusterJoints::Generic::randomJointState     GenericJoint.cpp:290-385 (independent coordinates
//                                                uniform, dependent ones by Newton on phi from a
//                                                guess in [-0.1, 0.1], up to 45 restarts)
// The per-cluster constraint function (phi, K_d) is generated code (struct C below).
#ifndef GRBDA_KERNELS_STATEGEN_CUH // (NVRTC sees this header under two include names: #pragma once is not enough)
#define GRBDA_KERNELS_STATEGEN_CUH
#include "batched_kernel.cuh" // integer typedefs that also work under NVRTC

namespace grbda_kernels
{
    struct Philox
    {
        uint32_t key0, key1, idx0, idx1, draw;
        uint32_t buf[4];

        __device__ Philox(uint64_t seed, uint64_t state_index)
            : key0((uint32_t)seed), key1((uint32_t)(seed >> 32)), idx0((uint32_t)state_index),
              idx1((uint32_t)(state_index >> 32)), draw(0) {}

        __device__ void block(uint32_t blk)
        {
            uint32_t c0 = idx0, c1 = idx1, c2 = blk, c3 = 0x67726264u;
            uint32_t k0 = key0, k1 = key1;
#pragma unroll
            for (int i = 0; i < 10; i++)
            {
                const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
                const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
                const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
                c0 = n0;
                c1 = lo1;
                c2 = n2;
                c3 = lo0;
                k0 += 0x9E3779B9u;
                k1 += 0xBB67AE85u;
            }
            buf[0] = c0;
            buf[1] = c1;
            buf[2] = c2;
            buf[3] = c3;
        }
        // uniform double in [-1, 1) from 53 random bits
        __device__ double uniform()
        {
            if ((draw & 1u) == 0)
                block(draw >> 1);
            const uint32_t lo = buf[2 * (draw & 1u)], hi = buf[2 * (draw & 1u) + 1];
            draw++;
            const uint64_t bits = (((uint64_t)hi << 32) | lo) >> 11;
            return (double)bits * (2.0 / 9007199254740992.0) - 1.0;
        }
    };

    // rpy -> quaternion (w, x, y, z) through the coordinate rotation matrix, exactly as
    // ori::rpyToQuat = rotationMatrixToQuaternion(rpyToRotMat(rpy)).
    __device__ inline void rpyToQuat(const double rpy[3], double q[4])
    {
        double sr, cr, sp, cp, sy, cy;
        sincos(rpy[0], &sr, &cr);
        sincos(rpy[1], &sp, &cp);
        sincos(rpy[2], &sy, &cy);
        // R = Rx(r) Ry(p) Rz(y) with coordinate rotations
        const double Rx[9] = {1, 0, 0, 0, cr, sr, 0, -sr, cr};
        const double Ry[9] = {cp, 0, -sp, 0, 1, 0, sp, 0, cp};
        const double Rz[9] = {cy, sy, 0, -sy, cy, 0, 0, 0, 1};
        double A[9], R[9];
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++)
            {
                double s = 0;
                for (int k = 0; k < 3; k++)
                    s += Rx[3 * i + k] * Ry[3 * k + j];
                A[3 * i + j] = s;
            }
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++)
            {
                double s = 0;
                for (int k = 0; k < 3; k++)
                    s += A[3 * i + k] * Rz[3 * k + j];
                R[3 * i + j] = s;
            }
        // r = R^T
        auto r = [&](int i, int j) { return R[3 * j + i]; };
        const double tr = r(0, 0) + r(1, 1) + r(2, 2);
        if (tr > 0.0)
        {
            const double S = sqrt(tr + 1.0) * 2.0;
            q[0] = 0.25 * S;
            q[1] = (r(2, 1) - r(1, 2)) / S;
            q[2] = (r(0, 2) - r(2, 0)) / S;
            q[3] = (r(1, 0) - r(0, 1)) / S;
        }
        else if ((r(0, 0) > r(1, 1)) && (r(0, 0) > r(2, 2)))
        {
            const double S = sqrt(1.0 + r(0, 0) - r(1, 1) - r(2, 2)) * 2.0;
            q[0] = (r(2, 1) - r(1, 2)) / S;
            q[1] = 0.25 * S;
            q[2] = (r(0, 1) + r(1, 0)) / S;
            q[3] = (r(0, 2) + r(2, 0)) / S;
        }
        else if (r(1, 1) > r(2, 2))
        {
            const double S = sqrt(1.0 + r(1, 1) - r(0, 0) - r(2, 2)) * 2.0;
            q[0] = (r(0, 2) - r(2, 0)) / S;
            q[1] = (r(0, 1) + r(1, 0)) / S;
            q[2] = 0.25 * S;
            q[3] = (r(1, 2) + r(2, 1)) / S;
        }
        else
        {
            const double S = sqrt(1.0 + r(2, 2) - r(0, 0) - r(1, 1)) * 2.0;
            q[0] = (r(1, 0) - r(0, 1)) / S;
            q[1] = (r(0, 2) + r(2, 0)) / S;
            q[2] = (r(1, 2) + r(2, 1)) / S;
            q[3] = 0.25 * S;
        }
    }

    // Solve the NC x NC system A x = b in place (partial pivoting); returns false when singular.
    template <int NC>
    __device__ inline bool smallSolve(double *A, double *b)
    {
        for (int k = 0; k < NC; k++)
        {
            int p = k;
            double best = fabs(A[k * NC + k]);
            for (int i = k + 1; i < NC; i++)
                if (fabs(A[i * NC + k]) > best)
                {
                    best = fabs(A[i * NC + k]);
                    p = i;
                }
            if (best == 0.0 || !(best == best))
                return false;
            if (p != k)
            {
                for (int j = 0; j < NC; j++)
                {
                    const double t = A[k * NC + j];
                    A[k * NC + j] = A[p * NC + j];
                    A[p * NC + j] = t;
                }
                const double t = b[k];
                b[k] = b[p];
                b[p] = t;
            }
            for (int i = k + 1; i < NC; i++)
            {
                const double f = A[i * NC + k] / A[k * NC + k];
                for (int j = k + 1; j < NC; j++)
                    A[i * NC + j] -= f * A[k * NC + j];
                b[i] -= f * b[k];
            }
        }
        for (int i = NC - 1; i >= 0; i--)
        {
            double s = b[i];
            for (int k = i + 1; k < NC; k++)
                s -= A[i * NC + k] * b[k];
            b[i] = s / A[i * NC + i];
        }
        return true;
    }

    // Frobenius-norm condition estimate |A| |A^-1| (same estimate as the oracle's generator).
    template <int NC>
    __device__ inline double condEstimate(const double *A)
    {
        double nA = 0, nI = 0;
        for (int i = 0; i < NC * NC; i++)
            nA += A[i] * A[i];
        for (int c = 0; c < NC; c++)
        {
            double M[NC * NC], e[NC];
            for (int i = 0; i < NC * NC; i++)
                M[i] = A[i];
            for (int i = 0; i < NC; i++)
                e[i] = i == c ? 1.0 : 0.0;
            if (!smallSolve<NC>(M, e))
                return 1e300;
            for (int i = 0; i < NC; i++)
                nI += e[i] * e[i];
        }
        return sqrt(nA) * sqrt(nI);
    }

    // Random valid spanning position of one implicit cluster. C provides
    //   N, NC, IND[], DEP[] and  static __device__ void eval(const double *q, double *phi, double *Kd)
    template <typename C>
    __device__ inline bool randomImplicitPosition(Philox &rng, double *q)
    {
        constexpr int N = C::N, NC = C::NC;
        double phi[NC], Kd[NC * NC];
        for (int attempt = 0; attempt < 45; attempt++)
        {
            for (int i = 0; i < N - NC; i++)
                q[C::ind(i)] = rng.uniform();
            for (int i = 0; i < NC; i++)
                q[C::dep(i)] = 0.1 * rng.uniform();
            bool ok = false, failed = false;
            for (int it = 0; it < 30 && !ok && !failed; it++)
            {
                C::eval(q, phi, Kd);
                double nrm = 0;
                for (int i = 0; i < NC; i++)
                    nrm = fmax(nrm, fabs(phi[i]));
                if (!(nrm == nrm))
                    failed = true;
                else if (nrm < 1e-13)
                    ok = true;
                else if (!smallSolve<NC>(Kd, phi))
                    failed = true;
                else
                    for (int i = 0; i < NC; i++)
                        q[C::dep(i)] -= phi[i];
            }
            if (!ok && !failed)
            {
                C::eval(q, phi, Kd);
                double s = 0;
                for (int i = 0; i < NC; i++)
                    s += phi[i] * phi[i];
                ok = sqrt(s) < 1e-10;
            }
            if (ok)
            {
                C::eval(q, phi, Kd);
                ok = condEstimate<NC>(Kd) < 1e6;
            }
            if (ok)
                return true;
        }
        return false;
    }

    // ---- integration step (SURVEY 8 f2) ------------------------------------------------------------------
    // quaternion (w, x, y, z) after rotating for dt with the WORLD-frame angular velocity omega:
    // ori::integrateQuat, include/grbda/Utils/OrientationTools.h:387-413 (axis-angle increment, product, renormalise)
    __device__ inline void integrateQuat(const double q[4], const double omega[3], double dt, double out[4])
    {
        double ang = sqrt(omega[0] * omega[0] + omega[1] * omega[1] + omega[2] * omega[2]);
        double axis[3] = {1.0, 0.0, 0.0};
        if (ang > 0.0)
            for (int i = 0; i < 3; i++)
                axis[i] = omega[i] / ang;
        ang *= dt;
        double s, c;
        sincos(0.5 * ang, &s, &c);
        const double d[4] = {c, s * axis[0], s * axis[1], s * axis[2]};
        // quatProduct(d, q) (OrientationTools.h:343-360)
        double r[4] = {d[0] * q[0] - d[1] * q[1] - d[2] * q[2] - d[3] * q[3],
                       d[0] * q[1] + d[1] * q[0] + d[2] * q[3] - d[3] * q[2],
                       d[0] * q[2] - d[1] * q[3] + d[2] * q[0] + d[3] * q[1],
                       d[0] * q[3] + d[1] * q[2] - d[2] * q[1] + d[3] * q[0]};
        const double n = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2] + r[3] * r[3]);
        for (int i = 0; i < 4; i++)
            out[i] = r[i] / n;
    }
    // Free joint (Joint.h:61-68, FreeJoint.cpp:29-46): q = [p world; quat], yd = [omega_body; v_body]. With
    // E = R(quat)^T (world -> body, OrientationTools.h:251-269): p' = p + dt E^T v_body, quat' =
    // integrateQuat(quat, E^T omega_body, dt).
    __device__ inline void integrateFreeQuaternion(const double *q, const double *yd, double dt, double *q_out)
    {
        const double w = q[3], x = q[4], y = q[5], z = q[6];
        // body -> world rotation R(quat)
        const double R[9] = {1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
                             2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                             2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)};
        double om[3], v[3];
        for (int i = 0; i < 3; i++)
        {
            om[i] = R[3 * i] * yd[0] + R[3 * i + 1] * yd[1] + R[3 * i + 2] * yd[2];
            v[i] = R[3 * i] * yd[3] + R[3 * i + 1] * yd[4] + R[3 * i + 2] * yd[5];
        }
        for (int i = 0; i < 3; i++)
            q_out[i] = q[i] + dt * v[i];
        integrateQuat(q + 3, om, dt, q_out + 3);
    }
    // Dependent coordinates of an implicit cluster back onto phi(q) = 0 (Newton on the dependent coordinates,
    // independent ones held; the same iteration the state generator uses). Returns false when it did not converge.
    template <typename C>
    __device__ inline bool projectImplicitPosition(double *q)
    {
        constexpr int NC = C::NC;
        double phi[NC], Kd[NC * NC];
        for (int it = 0; it < 30; it++)
        {
            C::eval(q, phi, Kd);
            double nrm = 0;
            for (int i = 0; i < NC; i++)
                nrm = fmax(nrm, fabs(phi[i]));
            if (!(nrm == nrm))
                return false;
            if (nrm < 1e-13)
                return true;
            if (!smallSolve<NC>(Kd, phi))
                return false;
            for (int i = 0; i < NC; i++)
                q[C::dep(i)] -= phi[i];
        }
        C::eval(q, phi, Kd);
        double s = 0;
        for (int i = 0; i < NC; i++)
            s += phi[i] * phi[i];
        return sqrt(s) < 1e-10;
    }

    // ---- reverse mode of the integration step -------------------------------------------------------------
    // The adjoints re-run the primal of their cluster and pull the cotangent q_out_bar of its new positions back:
    // q_bar (written) is the exact derivative of what the step computes for every stored position entry, yd_bar
    // (accumulated) is the part that reaches the new velocities through the positions.

    // Free joint (integrateFreeQuaternion): p' = p + dt R(quat) v_b, quat' = normalise(d(R(quat) w_b) (x) quat) with
    // the increment d(omega) = (cos(a t), sin(a t) / t omega), a = dt / 2, t = |omega|. R is the polynomial of the raw
    // stored entries, so a quaternion off the unit sphere gets the derivative of exactly that polynomial. Jacobian of d:
    //   d d0 / d omega = -a S omega^T,   d dvec / d omega = S I + c2 omega omega^T,
    //   S = sin(a t) / t,   c2 = (a cos(a t) - S) / t^2.
    // Below a t = 1e-2 both are Taylor series (S = a - a^3 t^2 / 6 + ..., c2 = -a^3 / 3 + a^5 t^2 / 30 - ...), so the
    // adjoint is finite and continuous at rest, where the primal takes d = (1, 0, 0, 0). At the switch the series
    // are exact to rounding; the closed form of c2 loses ~3e-12 of itself to cancellation there, but c2 enters
    // multiplied by t^2, i.e. ~3e-16 relative to S.
    __device__ inline void integrateFreeQuaternionVjp(const double *q, const double *yd, double dt, const double *q_out_bar,
                                                      double *q_bar, double *yd_bar)
    {
        const double w = q[3], x = q[4], y = q[5], z = q[6];
        const double R[9] = {1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
                             2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                             2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)};
        double om[3];
        for (int i = 0; i < 3; i++)
            om[i] = R[3 * i] * yd[0] + R[3 * i + 1] * yd[1] + R[3 * i + 2] * yd[2];
        // primal of the orientation, as integrateQuat computes it
        const double t = sqrt(om[0] * om[0] + om[1] * om[1] + om[2] * om[2]);
        double axis[3] = {1.0, 0.0, 0.0};
        if (t > 0.0)
            for (int i = 0; i < 3; i++)
                axis[i] = om[i] / t;
        double s, c;
        sincos(0.5 * (t * dt), &s, &c);
        const double d[4] = {c, s * axis[0], s * axis[1], s * axis[2]};
        const double *qq = q + 3;
        const double r[4] = {d[0] * qq[0] - d[1] * qq[1] - d[2] * qq[2] - d[3] * qq[3],
                             d[0] * qq[1] + d[1] * qq[0] + d[2] * qq[3] - d[3] * qq[2],
                             d[0] * qq[2] - d[1] * qq[3] + d[2] * qq[0] + d[3] * qq[1],
                             d[0] * qq[3] + d[1] * qq[2] - d[2] * qq[1] + d[3] * qq[0]};
        const double n = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2] + r[3] * r[3]);
        // out = r / n
        const double *ob = q_out_bar + 3;
        const double proj = (r[0] * ob[0] + r[1] * ob[1] + r[2] * ob[2] + r[3] * ob[3]) / (n * n);
        double rb[4];
        for (int i = 0; i < 4; i++)
            rb[i] = (ob[i] - r[i] * proj) / n;
        // r = d (x) quat
        const double db[4] = {rb[0] * qq[0] + rb[1] * qq[1] + rb[2] * qq[2] + rb[3] * qq[3],
                              -rb[0] * qq[1] + rb[1] * qq[0] - rb[2] * qq[3] + rb[3] * qq[2],
                              -rb[0] * qq[2] + rb[1] * qq[3] + rb[2] * qq[0] - rb[3] * qq[1],
                              -rb[0] * qq[3] - rb[1] * qq[2] + rb[2] * qq[1] + rb[3] * qq[0]};
        double qb[4] = {rb[0] * d[0] + rb[1] * d[1] + rb[2] * d[2] + rb[3] * d[3],
                        -rb[0] * d[1] + rb[1] * d[0] + rb[2] * d[3] - rb[3] * d[2],
                        -rb[0] * d[2] - rb[1] * d[3] + rb[2] * d[0] + rb[3] * d[1],
                        -rb[0] * d[3] + rb[1] * d[2] - rb[2] * d[1] + rb[3] * d[0]};
        // d(omega)
        const double a = 0.5 * dt, u = a * a * t * t;
        double S, c2;
        if (fabs(a) * t < 1e-2)
        {
            S = a * (1.0 - u / 6.0 * (1.0 - u / 20.0 * (1.0 - u / 42.0)));
            c2 = -a * a * a / 3.0 * (1.0 - u / 10.0 * (1.0 - u / 28.0 * (1.0 - u / 54.0)));
        }
        else
        {
            S = s / t;
            c2 = (a * c - S) / (t * t);
        }
        const double om_db = om[0] * db[1] + om[1] * db[2] + om[2] * db[3];
        double omb[3], vb[3];
        for (int i = 0; i < 3; i++)
        {
            omb[i] = -a * S * om[i] * db[0] + S * db[1 + i] + c2 * om[i] * om_db;
            vb[i] = dt * q_out_bar[i]; // p' = p + dt R v_b
            q_bar[i] = q_out_bar[i];
        }
        // om = R w_b, v = R v_b: R_bar = omb w_b^T + vb v_b^T, yd_bar += R^T [omb; vb]
        double Rb[9];
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++)
            {
                Rb[3 * i + j] = omb[i] * yd[j] + vb[i] * yd[3 + j];
                yd_bar[j] += R[3 * i + j] * omb[i];
                yd_bar[3 + j] += R[3 * i + j] * vb[i];
            }
        qb[0] += 2 * (-Rb[1] * z + Rb[2] * y + Rb[3] * z - Rb[5] * x - Rb[6] * y + Rb[7] * x);
        qb[1] += 2 * (Rb[1] * y + Rb[2] * z + Rb[3] * y - 2 * Rb[4] * x - Rb[5] * w + Rb[6] * z + Rb[7] * w - 2 * Rb[8] * x);
        qb[2] += 2 * (-2 * Rb[0] * y + Rb[1] * x + Rb[2] * w + Rb[3] * x + Rb[5] * z - Rb[6] * w + Rb[7] * z - 2 * Rb[8] * y);
        qb[3] += 2 * (-2 * Rb[0] * z - Rb[1] * w + Rb[2] * x + Rb[3] * w - 2 * Rb[4] * z + Rb[5] * y + Rb[6] * x + Rb[7] * y);
        for (int i = 0; i < 4; i++)
            q_bar[3 + i] = qb[i];
    }

    // Implicit cluster at its projected point q_span (projectImplicitPosition converged there), by the implicit
    // function theorem: the new dependent coordinates are g(q_ind') with d g / d q_ind' = -K_dep^-1 K_ind, so
    //   K_dep^T lambda = q_out_bar_dep,   q_ind_bar = q_out_bar_ind - K_ind^T lambda   (= G^T q_out_bar)
    // and q_ind' = q_ind + dt yd_ind adds dt q_ind_bar to the cluster's velocities. The old dependent coordinates are
    // only Newton's starting point: their q_bar is 0. C provides N, NC, ind(), dep() and
    //   static void jacobian(const double *q, double *Kd, double *Ki)   (row-major per constraint).
    template <typename C>
    __device__ inline void implicitPositionVjp(const double *q_span, double dt, const double *q_out_bar, double *q_bar,
                                               double *yd_bar)
    {
        constexpr int N = C::N, NC = C::NC, NI = N - NC;
        double Kd[NC * NC], Ki[NC * NI], A[NC * NC], lambda[NC];
        C::jacobian(q_span, Kd, Ki);
        for (int i = 0; i < NC; i++)
        {
            for (int j = 0; j < NC; j++)
                A[i * NC + j] = Kd[j * NC + i];
            lambda[i] = q_out_bar[C::dep(i)];
        }
        if (!smallSolve<NC>(A, lambda))
            for (int i = 0; i < NC; i++)
                lambda[i] = nan("");
        for (int k = 0; k < NI; k++)
        {
            double s = q_out_bar[C::ind(k)];
            for (int i = 0; i < NC; i++)
                s -= Ki[i * NI + k] * lambda[i];
            q_bar[C::ind(k)] = s;
            yd_bar[k] += dt * s;
        }
        for (int i = 0; i < NC; i++)
            q_bar[C::dep(i)] = 0.0;
    }

    // One state of the reverse integration step. StepVjp::run(q, yd_new, dt, q_out_bar, q_bar, v_bar) is generated per
    // model (compiler/compile.h emitIntegrateVjp): it re-runs the step cluster by cluster, Newton projections included,
    // writes q_bar and adds the position part to v_bar. yd' = yd + dt ydd: yd_bar = v_bar, ydd_bar = dt v_bar.
    template <typename StepVjp>
    __device__ inline bool integrateVjpState(const double *q, const double *yd, const double *ydd, double dt,
                                             const double *q_out_bar, const double *yd_out_bar, double *q_bar,
                                             double *yd_bar, double *ydd_bar)
    {
        double ydn[StepVjp::NV];
        for (int k = 0; k < StepVjp::NV; k++)
        {
            ydn[k] = yd[k] + dt * ydd[k];
            yd_bar[k] = yd_out_bar[k];
        }
        const bool ok = StepVjp::run(q, ydn, dt, q_out_bar, q_bar, yd_bar);
        for (int k = 0; k < StepVjp::NV; k++)
            ydd_bar[k] = dt * yd_bar[k];
        return ok;
    }

    template <typename StepVjp>
    __global__ void __launch_bounds__(128)
        grbda_integrate_vjp_kernel(const double *__restrict__ q, const double *__restrict__ yd,
                                   const double *__restrict__ ydd, double dt, const double *__restrict__ q_out_bar,
                                   const double *__restrict__ yd_out_bar, int64_t count, double *__restrict__ q_bar,
                                   double *__restrict__ yd_bar, double *__restrict__ ydd_bar, int32_t *__restrict__ flags)
    {
        const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= count)
            return;
        constexpr int NQ = StepVjp::NQ, NV = StepVjp::NV;
        double ql[NQ], ydl[NV], yddl[NV], qob[NQ], ydob[NV], qb[NQ], ydb[NV], yddb[NV];
        for (int k = 0; k < NQ; k++)
        {
            ql[k] = q[i * NQ + k];
            qob[k] = q_out_bar[i * NQ + k];
        }
        for (int k = 0; k < NV; k++)
        {
            ydl[k] = yd[i * NV + k];
            yddl[k] = ydd[i * NV + k];
            ydob[k] = yd_out_bar[i * NV + k];
        }
        const bool ok = integrateVjpState<StepVjp>(ql, ydl, yddl, dt, qob, ydob, qb, ydb, yddb);
        for (int k = 0; k < NQ; k++)
            q_bar[i * NQ + k] = qb[k];
        for (int k = 0; k < NV; k++)
        {
            yd_bar[i * NV + k] = ydb[k];
            ydd_bar[i * NV + k] = yddb[k];
        }
        if (flags)
            flags[i] = ok ? 0 : 1;
    }

    // Step::run advances one state (generated per model): semi-implicit Euler, yd' = yd + dt ydd, q' from yd'
    template <typename Step>
    __global__ void __launch_bounds__(128)
        grbda_integrate_kernel(const double *__restrict__ q, const double *__restrict__ yd, const double *__restrict__ ydd,
                               double dt, int64_t count, double *__restrict__ q_out, double *__restrict__ yd_out,
                               int32_t *__restrict__ flags)
    {
        const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= count)
            return;
        double ql[Step::NQ], ydl[Step::NV], qn[Step::NQ];
        for (int k = 0; k < Step::NQ; k++)
            ql[k] = q[i * Step::NQ + k];
        for (int k = 0; k < Step::NV; k++)
            ydl[k] = yd[i * Step::NV + k] + dt * ydd[i * Step::NV + k];
        const bool ok = Step::run(ql, ydl, dt, qn);
        for (int k = 0; k < Step::NQ; k++)
            q_out[i * Step::NQ + k] = qn[k];
        for (int k = 0; k < Step::NV; k++)
            yd_out[i * Step::NV + k] = ydl[k];
        if (flags)
            flags[i] = ok ? 0 : 1;
    }

    // Gen::run fills one state (generated per model, csrc/generated/<model>_gen.cu)
    template <typename Gen>
    __global__ void __launch_bounds__(128)
        grbda_generate_kernel(uint64_t seed, int64_t first_index, int64_t count, double *__restrict__ q,
                              double *__restrict__ yd, double *__restrict__ aux, int32_t *__restrict__ flags)
    {
        const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= count)
            return;
        Philox rng(seed, (uint64_t)(first_index + i));
        double ql[Gen::NQ], ydl[Gen::NV], auxl[Gen::NV];
        const bool ok = Gen::run(rng, ql, ydl, auxl);
        for (int k = 0; k < Gen::NQ; k++)
            q[i * Gen::NQ + k] = ql[k];
        for (int k = 0; k < Gen::NV; k++)
        {
            yd[i * Gen::NV + k] = ydl[k];
            aux[i * Gen::NV + k] = auxl[k];
        }
        if (flags)
            flags[i] = ok ? 0 : 1;
    }

} // namespace grbda_kernels
#endif // GRBDA_KERNELS_STATEGEN_CUH
