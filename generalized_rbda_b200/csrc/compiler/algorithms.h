// Device-side model compiler, part 1: the cluster-tree algorithms evaluated symbolically.
//
// Each routine runs ONE evaluation of the algorithm over sym::Sym scalars for a given
// ClusterTreeModel; the resulting expression DAG is the per-state program that compiler/emit.h
// turns into a straight-line sm_100a kernel body (one state per thread).
//
// What is computed (reference, all under /root/reference):
//   kinematics   TreeModel::forwardKinematics                 src/Dynamics/TreeModel.cpp:7-32
//                per-type updateKinematics                    src/Dynamics/ClusterJoints/*.cpp
//                GenericImplicit K, G, k, g                   GenericJoint.cpp:58-91
//   ID           recursiveNewtonEulerAlgorithm                TreeModel.cpp:35-57,174-212
//   FD           updateArticulatedBodies + forwardDynamics    ClusterTreeDynamics.cpp:85-191
//   H            compositeRigidBodyAlgorithm                  TreeModel.cpp:116-160
//   FK outputs   getPosition/getOrientation/get*Velocity      ClusterTreeModel.cpp:319-373
//
// How it is restructured for the GPU (not a translation):
//   * every cluster type (Revolute, RevoluteWithRotor, RevolutePair(WithRotor), Generic, ...) is the
//     same object here — revolute bodies on a spanning tree plus G (constant or from phi) — so the
//     per-type dispatch of the reference disappears at model-compile time;
//   * ID and H run on the spanning tree at body level and are projected with G (tau = G^T tau_s,
//     H = G^T H_s G), which is algebraically identical to the cluster recursion (S = X_intra S_s G)
//     but never forms the 6N x n motion subspace;
//   * FD is the cluster (constraint-embedded) ABA. X^T Ia X is evaluated as
//     sum_i X_i^T IA_ii X_i - W D^-1 W^T with W = X^T U (6 x n) instead of the reference's dense
//     6N x 6N products; rigid 10-parameter inertias are kept as long as possible;
//   * D^-1 is an unrolled LDL^T (D = S^T IA S is SPD); the reference uses ColPivHouseholderQR.
#pragma once
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <algorithm>
#include <functional>
#include <map>
#include "../host/model.h"
#include "spatial_sym.h"
#include "autodiff.h"

namespace grbda
{
    namespace compiler
    {
        // Input arrays of a generated kernel
        enum InputArray
        {
            IN_Q = 0,  // nq  positions (spanning coordinates for implicit clusters)
            IN_YD = 1, // nv  independent velocities
            IN_AUX = 2 // nv  ydd (ID) or tau (FD)
        };

        // second-order Taylor scalar over Sym for phi derivatives (K = dphi/dq, k = -qd^T H qd)
        struct Taylor2
        {
            Sym c0, c1, c2;
            Taylor2() {}
            Taylor2(double x) : c0(x), c1(0.0), c2(0.0) {}
            Taylor2(const Sym &a, const Sym &b, const Sym &c) : c0(a), c1(b), c2(c) {}
        };
        inline Taylor2 operator+(const Taylor2 &a, const Taylor2 &b) { return {a.c0 + b.c0, a.c1 + b.c1, a.c2 + b.c2}; }
        inline Taylor2 operator-(const Taylor2 &a, const Taylor2 &b) { return {a.c0 - b.c0, a.c1 - b.c1, a.c2 - b.c2}; }
        inline Taylor2 operator-(const Taylor2 &a) { return {-a.c0, -a.c1, -a.c2}; }
        inline Taylor2 operator*(const Taylor2 &a, const Taylor2 &b)
        {
            return {a.c0 * b.c0, a.c0 * b.c1 + a.c1 * b.c0, a.c0 * b.c2 + a.c1 * b.c1 + a.c2 * b.c0};
        }
        inline Taylor2 operator/(const Taylor2 &a, const Taylor2 &b)
        {
            // only division by a constant occurs in constraint functions
            if (!b.c0.isConst() || !b.c1.isZero() || !b.c2.isZero())
                throw std::runtime_error("phi: division by a non-constant is not supported");
            return {a.c0 / b.c0, a.c1 / b.c0, a.c2 / b.c0};
        }
        inline Taylor2 sin(const Taylor2 &a)
        {
            const Sym s = sym::sin(a.c0), c = sym::cos(a.c0);
            return {s, c * a.c1, c * a.c2 - Sym(0.5) * s * a.c1 * a.c1};
        }
        inline Taylor2 cos(const Taylor2 &a)
        {
            const Sym s = sym::sin(a.c0), c = sym::cos(a.c0);
            return {c, -(s * a.c1), -(s * a.c2) - Sym(0.5) * c * a.c1 * a.c1};
        }

        // Unrolled LDL^T of a small SPD matrix
        struct LDLT
        {
            int n = 0;
            std::vector<Sym> L;    // n x n, unit lower (only i > j used)
            std::vector<Sym> dinv; // 1 / d_j

            void factor(const std::vector<Sym> &D, int n_)
            {
                n = n_;
                L.assign(n * n, Sym(0.0));
                dinv.assign(n, Sym(0.0));
                std::vector<Sym> d(n);
                for (int j = 0; j < n; j++)
                {
                    Sym dj = D[j * n + j];
                    for (int k = 0; k < j; k++)
                        dj = dj - L[j * n + k] * L[j * n + k] * d[k];
                    d[j] = dj;
                    dinv[j] = Sym(1.0) / dj;
                    for (int i = j + 1; i < n; i++)
                    {
                        Sym lij = D[i * n + j];
                        for (int k = 0; k < j; k++)
                            lij = lij - L[i * n + k] * L[j * n + k] * d[k];
                        L[i * n + j] = lij * dinv[j];
                    }
                }
            }
            std::vector<Sym> solve(std::vector<Sym> b) const
            {
                for (int i = 0; i < n; i++)
                    for (int k = 0; k < i; k++)
                        b[i] = b[i] - L[i * n + k] * b[k];
                for (int i = 0; i < n; i++)
                    b[i] = b[i] * dinv[i];
                for (int i = n - 1; i >= 0; i--)
                    for (int k = i + 1; k < n; k++)
                        b[i] = b[i] - L[k * n + i] * b[k];
                return b;
            }
        };

        // Inverse of a small regular (non symmetric) matrix, static pivot order.
        inline std::vector<Sym> smallInverse(const std::vector<Sym> &A, int n)
        {
            std::vector<Sym> inv(n * n);
            if (n == 1)
                inv[0] = Sym(1.0) / A[0];
            else if (n == 2)
            {
                const Sym idet = Sym(1.0) / (A[0] * A[3] - A[1] * A[2]);
                inv = {A[3] * idet, -(A[1] * idet), -(A[2] * idet), A[0] * idet};
            }
            else if (n == 3)
            {
                auto a = [&](int i, int j) { return A[3 * i + j]; };
                std::vector<Sym> cof(9);
                for (int i = 0; i < 3; i++)
                    for (int j = 0; j < 3; j++)
                    {
                        const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
                        cof[3 * i + j] = a(i1, j1) * a(i2, j2) - a(i1, j2) * a(i2, j1);
                    }
                const Sym idet = Sym(1.0) / (a(0, 0) * cof[0] + a(0, 1) * cof[1] + a(0, 2) * cof[2]);
                for (int i = 0; i < 3; i++)
                    for (int j = 0; j < 3; j++)
                        inv[3 * i + j] = cof[3 * j + i] * idet;
            }
            else
            {
                // Gauss-Jordan without pivoting (structure known only symbolically)
                std::vector<Sym> M = A;
                for (int i = 0; i < n; i++)
                    for (int j = 0; j < n; j++)
                        inv[i * n + j] = Sym(i == j ? 1.0 : 0.0);
                for (int k = 0; k < n; k++)
                {
                    if (M[k * n + k].isZero())
                        throw std::runtime_error("constraint Jacobian K_d has a structurally zero pivot");
                    const Sym ip = Sym(1.0) / M[k * n + k];
                    for (int j = 0; j < n; j++)
                    {
                        M[k * n + j] = M[k * n + j] * ip;
                        inv[k * n + j] = inv[k * n + j] * ip;
                    }
                    for (int i = 0; i < n; i++)
                        if (i != k)
                        {
                            const Sym f = M[i * n + k];
                            for (int j = 0; j < n; j++)
                            {
                                M[i * n + j] = M[i * n + j] - f * M[k * n + j];
                                inv[i * n + j] = inv[i * n + j] - f * inv[k * n + j];
                            }
                        }
                }
            }
            return inv;
        }

        class ModelCompiler
        {
        public:
            explicit ModelCompiler(const ClusterTreeModel &model) : m_(model) { findAxisymmetricLeaves(); }

            // Inputs of the programs. The operational-space programs (contact Jacobians aside) reuse the dynamics
            // below with substituted inputs: velocities and gravity set to zero, generalized forces given as
            // expressions (solveMassMatrix); structural zeros then fold everything velocity-dependent away.
            Sym inYd(int i) const { return yd_override_ ? (*yd_override_)[i] : Sym::input(IN_YD, i); }
            Sym inAux(int i) const { return aux_override_ ? (*aux_override_)[i] : Sym::input(IN_AUX, i); }

            // A leaf body whose inertia is symmetric about its own joint axis (a motor rotor: centre of
            // mass on the axis, equal transverse moments, no products of inertia) exerts the same force
            // on its parent and the same joint torque at every joint angle: with R the joint rotation,
            // R I = I R and R s = s, hence v = R v', a = R a', f = R f' and X^T f = Xtree^T f', where the
            // primed quantities are computed with the angle held at zero. Dynamics programs (ID, FD, H)
            // therefore evaluate such bodies at angle zero: no sin/cos, constant transforms. Forward
            // kinematics, whose outputs are the body poses themselves, keeps the angles.
            void setFreezeAxisymmetricLeaves(bool on) { freeze_leaves_ = on; }
            bool isAxisymmetricLeaf(int body) const { return axisym_leaf_[body] != 0; }

            // Gyrostat reduction (ID, H and the L^T D L forward dynamics): such a body r with parent p,
            // axis z (in p's frame) and axial moment J obeys, with I_r s = [J z; 0] and s x* I_r = I_r s x,
            //     f_r = [I_r a_p' + v_p' x* I_r v_p']  +  [J (qdd_r z + qd_r w_p x z); 0],
            //     tau_r = J (z . wdot_p + qdd_r),
            // so its inertia is merged into its parent's once, at compile time (X0^T I_r X0 with the
            // constant Xtree), and what remains per rotor is a couple on the parent and one dot product.
            // In the mass matrix it contributes J G_k G_l on its own dofs and the couple [J z G_k; 0]
            // on p for the coupling with every dof that moves p.
            void setGyrostatReduction(bool on) { gyrostats_ = on; }
            bool isGyrostat(int body) const
            {
                return gyrostats_ && freeze_leaves_ && axisym_leaf_[body] && m_.bodies()[body].parent_index_ >= 0;
            }
            int jointAxisOfBody(int body) const
            {
                const ClusterTreeNode &c = m_.clusters()[m_.getIndexOfClusterContainingBody(body)];
                return (int)c.joint_.axes[body - c.first_body_];
            }
            V3 gyrostatAxis(int body) const // joint axis of the rotor in its parent's frame
            {
                V3 e;
                e[jointAxisOfBody(body)] = Sym(1.0);
                return mulT(constM3(m_.bodies()[body].Xtree_.E), e);
            }
            Sym gyrostatInertia(int body) const
            {
                const int a = jointAxisOfBody(body);
                return Sym(m_.bodies()[body].inertia_.getMatrix()[6 * a + a]);
            }
            // rigid inertia of a body, with the inertias of its gyrostat children merged in
            RigidInertia bodyInertia(int body) const
            {
                RigidInertia I = RigidInertia::fromMatrix(m_.bodies()[body].inertia_.getMatrix());
                for (const Body &r : m_.bodies())
                    if (r.parent_index_ == body && isGyrostat(r.index_))
                    {
                        Xf X0;
                        X0.E = constM3(r.Xtree_.E);
                        X0.r = constV3(r.Xtree_.r);
                        I = I + RigidInertia::fromMatrix(r.inertia_.getMatrix()).toParent(X0);
                    }
                return I;
            }

            // ---------------------------------------------------------------------------------
            // per-cluster constraint quantities
            // ---------------------------------------------------------------------------------
            struct ClusterKin
            {
                std::vector<Sym> q_s, qd_s, g; // spanning position / velocity, bias g (N)
                std::vector<Sym> G;            // N x n
                std::vector<Sym> K, k;         // nc x N, nc (implicit only)
            };
            struct BodyKin
            {
                Xf Xl;        // from the parent body (any cluster) to this body
                Xf Xup;       // from the cluster-ancestor body to this body
                int anc = -1; // global index of the cluster-ancestor body
                SV v, vJ, cJ, avp;
                std::vector<SV> S; // n columns of the cluster motion subspace rows of this body
                Sym qd;            // spanning velocity of this body's joint (revolute)
            };

            // phi, K (nc x N) and optionally k for an implicit cluster at spanning position q_s
            void implicitJacobian(const ClusterDesc &d, const std::vector<Sym> &q_s,
                                  const std::vector<Sym> *qd_s, std::vector<Sym> &phi,
                                  std::vector<Sym> &K, std::vector<Sym> *k) const
            {
                const int N = d.num_bodies, nc = d.num_constraints;
                K.assign(nc * N, Sym(0.0));
                for (int j = 0; j < N; j++)
                {
                    std::vector<Taylor2> qs(N);
                    for (int i = 0; i < N; i++)
                        qs[i] = Taylor2(q_s[i], Sym(i == j ? 1.0 : 0.0), Sym(0.0));
                    const std::vector<Taylor2> p = d.phi.evaluate(qs);
                    for (int i = 0; i < nc; i++)
                        K[i * N + j] = p[i].c1;
                    if (j == 0)
                    {
                        phi.resize(nc);
                        for (int i = 0; i < nc; i++)
                            phi[i] = p[i].c0;
                    }
                }
                if (k && qd_s)
                {
                    std::vector<Taylor2> qs(N);
                    for (int i = 0; i < N; i++)
                        qs[i] = Taylor2(q_s[i], (*qd_s)[i], Sym(0.0));
                    const std::vector<Taylor2> p = d.phi.evaluate(qs);
                    k->resize(nc);
                    for (int i = 0; i < nc; i++)
                        (*k)[i] = -(Sym(2.0) * p[i].c2);
                }
            }

            ClusterKin clusterConstraint(const ClusterTreeNode &c, bool with_velocity) const
            {
                const ClusterDesc &d = c.joint_;
                const int N = d.num_bodies, n = d.num_velocities;
                ClusterKin ck;
                std::vector<Sym> y(d.num_positions), yd(n);
                for (int i = 0; i < d.num_positions; i++)
                    y[i] = Sym::input(IN_Q, c.position_index_ + i);
                for (int i = 0; i < n; i++)
                    yd[i] = with_velocity ? inYd(c.velocity_index_ + i) : Sym(0.0);
                ck.G.assign(N * n, Sym(0.0));
                ck.g.assign(N, Sym(0.0));
                if (d.type == ClusterType::Explicit)
                {
                    // q_span = gamma(y) = G y   (LoopConstraint.cpp:48-52)
                    for (int i = 0; i < N * n; i++)
                        ck.G[i] = Sym(d.G[i]);
                    ck.q_s.assign(N, Sym(0.0));
                    for (int i = 0; i < N; i++)
                        for (int j = 0; j < n; j++)
                            ck.q_s[i] = ck.q_s[i] + ck.G[i * n + j] * y[j];
                }
                else
                {
                    ck.q_s = y;
                    std::vector<int> ind, dep;
                    for (int i = 0; i < N; i++)
                        (d.independent[i] ? ind : dep).push_back(i);
                    const int nc = d.num_constraints;
                    std::vector<Sym> phi;
                    implicitJacobian(d, ck.q_s, nullptr, phi, ck.K, nullptr);
                    std::vector<Sym> Kd(nc * nc);
                    for (int i = 0; i < nc; i++)
                        for (int j = 0; j < nc; j++)
                            Kd[i * nc + j] = ck.K[i * N + dep[j]];
                    const std::vector<Sym> Kd_inv = smallInverse(Kd, nc);
                    // G = P [1; -Kd^-1 Ki]   (GenericJoint.cpp:70-85)
                    for (int j = 0; j < n; j++)
                        ck.G[ind[j] * n + j] = Sym(1.0);
                    for (int i = 0; i < nc; i++)
                        for (int j = 0; j < n; j++)
                        {
                            Sym s(0.0);
                            for (int l = 0; l < nc; l++)
                                s = s + Kd_inv[i * nc + l] * ck.K[l * N + ind[j]];
                            ck.G[dep[i] * n + j] = -s;
                        }
                    if (with_velocity)
                    {
                        ck.qd_s.assign(N, Sym(0.0));
                        for (int i = 0; i < N; i++)
                            for (int j = 0; j < n; j++)
                                ck.qd_s[i] = ck.qd_s[i] + ck.G[i * n + j] * yd[j];
                        // k = -Kdot qd, g = P [0; Kd^-1 k]   (GenericJoint.cpp:60-68,87-91)
                        std::vector<Sym> K2;
                        implicitJacobian(d, ck.q_s, &ck.qd_s, phi, K2, &ck.k);
                        for (int i = 0; i < nc; i++)
                        {
                            Sym s(0.0);
                            for (int l = 0; l < nc; l++)
                                s = s + Kd_inv[i * nc + l] * ck.k[l];
                            ck.g[dep[i]] = s;
                        }
                    }
                }
                if (ck.qd_s.empty())
                {
                    ck.qd_s.assign(N, Sym(0.0));
                    for (int i = 0; i < N; i++)
                        for (int j = 0; j < n; j++)
                            ck.qd_s[i] = ck.qd_s[i] + ck.G[i * n + j] * yd[j];
                }
                return ck;
            }

            // ---------------------------------------------------------------------------------
            // kinematics of every body (forward pass)
            // ---------------------------------------------------------------------------------
            // children lists and the depth-first cluster order. The emitted program follows the
            // order in which expressions are created, so every sweep below visits the tree depth
            // first (finish one limb before starting the next): the values that must stay live across
            // the downward and upward sweep of a limb are then few enough to stay in registers.
            void buildTraversal()
            {
                const int Nc = m_.getNumClusters();
                children_.assign(Nc, std::vector<int>());
                roots_.clear();
                for (const ClusterTreeNode &c : m_.clusters())
                    (c.parent_index_ >= 0 ? children_[c.parent_index_] : roots_).push_back(c.index_);
            }

            void beginKinematics()
            {
                bk_.assign(m_.getNumBodies(), BodyKin());
                ck_.assign(m_.getNumClusters(), ClusterKin());
                buildTraversal();
            }

            // all clusters, depth first
            void kinematics(bool with_velocity, bool with_subspace)
            {
                beginKinematics();
                std::function<void(int)> visit = [&](int ci) {
                    kinematicsCluster(ci, with_velocity, with_subspace);
                    for (int ch : children_[ci])
                        visit(ch);
                };
                for (int r : roots_)
                    visit(r);
            }

            // kinematics of the bodies of one cluster (its parent cluster must have been processed)
            void kinematicsCluster(int ci, bool with_velocity, bool with_subspace)
            {
                {
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    const ClusterDesc &d = c.joint_;
                    const int n = d.num_velocities;
                    if (d.type == ClusterType::FreeQuaternion || d.type == ClusterType::FreeRollPitchYaw)
                    {
                        // Joints::Free (Joint.h:61-68); Xtree ignored (FreeJoint.cpp:45)
                        BodyKin &b = bk_[c.first_body_];
                        const int pi = c.position_index_;
                        V3 p{{Sym::input(IN_Q, pi), Sym::input(IN_Q, pi + 1), Sym::input(IN_Q, pi + 2)}};
                        M3 E;
                        if (d.type == ClusterType::FreeQuaternion)
                            E = quaternionToRotationMatrix(Sym::input(IN_Q, pi + 3), Sym::input(IN_Q, pi + 4),
                                                           Sym::input(IN_Q, pi + 5), Sym::input(IN_Q, pi + 6));
                        else
                        {
                            const Sym r = Sym::input(IN_Q, pi + 3), pt = Sym::input(IN_Q, pi + 4),
                                      yw = Sym::input(IN_Q, pi + 5);
                            E = mul(mul(coordinateRotation(ori::CoordinateAxis::X, sym::sin(r), sym::cos(r)),
                                        coordinateRotation(ori::CoordinateAxis::Y, sym::sin(pt), sym::cos(pt))),
                                    coordinateRotation(ori::CoordinateAxis::Z, sym::sin(yw), sym::cos(yw)));
                        }
                        b.Xl.E = E;
                        b.Xl.r = p;
                        b.Xup = b.Xl;
                        b.anc = -1;
                        for (int i = 0; i < 6; i++)
                            b.v[i] = with_velocity ? inYd(c.velocity_index_ + i) : Sym(0.0);
                        b.vJ = b.v;
                        if (with_subspace)
                        {
                            b.S.assign(6, SV());
                            for (int k = 0; k < 6; k++)
                                b.S[k][k] = Sym(1.0);
                        }
                        return;
                    }

                    const long n0 = (long)Sym::G().nodes.size();
                    ClusterKin ck = clusterConstraint(c, with_velocity);
                    if (std::getenv("GRBDA_LTL_TRACE"))
                        std::fprintf(stderr, "constraint nodes cluster %d type %d: %ld\n", ci, (int)d.type,
                                     (long)Sym::G().nodes.size() - n0);
                    for (int i = 0; i < d.num_bodies; i++)
                    {
                        const Body &body = c.bodies_[i];
                        BodyKin &b = bk_[body.index_];
                        const int axis = (int)d.axes[i];
                        const bool frozen = freeze_leaves_ && axisym_leaf_[body.index_];
                        const Sym s = frozen ? Sym(0.0) : sym::sin(ck.q_s[i]);
                        const Sym co = frozen ? Sym(1.0) : sym::cos(ck.q_s[i]);
                        // XJ * Xtree  (Joint.h:94-97)
                        b.Xl.E = mul(coordinateRotation(d.axes[i], s, co), constM3(body.Xtree_.E));
                        b.Xl.r = constV3(body.Xtree_.r);
                        b.qd = ck.qd_s[i];
                        SV sq; // s_i * qd_i
                        sq[axis] = b.qd;
                        const int p = body.parent_index_;
                        const bool parent_in_cluster = p >= c.first_body_ && p >= 0 &&
                                                       m_.getIndexOfClusterContainingBody(p) == c.index_;
                        if (parent_in_cluster)
                        {
                            const BodyKin &pb = bk_[p];
                            b.Xup = b.Xl * pb.Xup;
                            b.anc = pb.anc;
                            b.vJ = b.Xl.applyMotion(pb.vJ) + sq;
                            // cJ_i = Xl cJ_p + vJ_i x (s_i qd_i) + s_i g_i  (GenericJoint.cpp:427-451)
                            b.cJ = b.Xl.applyMotion(pb.cJ) + motionCross(b.vJ, sq);
                        }
                        else
                        {
                            b.Xup = b.Xl;
                            b.anc = p;
                            b.vJ = sq;
                        }
                        b.cJ[axis] = b.cJ[axis] + ck.g[i];
                        b.v = (p >= 0 ? b.Xl.applyMotion(bk_[p].v) : SV()) + sq;
                        b.avp = motionCross(b.v, b.vJ);
                        if (with_subspace)
                        {
                            b.S.assign(n, SV());
                            for (int k = 0; k < n; k++)
                            {
                                if (parent_in_cluster)
                                    b.S[k] = b.Xl.applyMotion(bk_[p].S[k]);
                                b.S[k][axis] = b.S[k][axis] + ck.G[i * n + k];
                            }
                        }
                    }
                    ck_[ci] = ck;
                }
            }

            // couple of a gyrostat on its parent (added to f_parent) and its own spanning joint torque
            Sym gyrostatForces(int body, const Sym &qd, const Sym &qdd, const SV &a_parent, SV &f_parent) const
            {
                const int p = m_.bodies()[body].parent_index_;
                const V3 z = gyrostatAxis(body);
                const Sym J = gyrostatInertia(body);
                const V3 n = J * (qdd * z + qd * cross(bk_[p].v.ang(), z));
                f_parent = f_parent + SV::make(n, V3());
                return J * (dot(z, a_parent.ang()) + qdd);
            }

            SV minusGravity() const
            {
                SV a;
                if (!zero_gravity_)
                    for (int i = 0; i < 3; i++)
                        a[3 + i] = Sym(-m_.getGravity()[i]);
                return a;
            }

            // ---------------------------------------------------------------------------------
            // forward kinematics outputs: per body p(3), R(9), [w_world; v_world](6)
            // ---------------------------------------------------------------------------------
            void forwardKinematics(std::vector<Sym> &p_out, std::vector<Sym> &R_out, std::vector<Sym> &v_out)
            {
                // cluster by cluster, depth first: the absolute transform and the outputs of a body are
                // formed right after its joint transform, so only the transforms along the current path
                // are alive (forming all joint transforms first kept 37 x 18 values alive, i.e. in local
                // memory, until the output loop reached them)
                beginKinematics();
                const int Nb = m_.getNumBodies();
                std::vector<Xf> Xa(Nb);
                p_out.assign(3 * Nb, Sym(0.0));
                R_out.assign(9 * Nb, Sym(0.0));
                v_out.assign(6 * Nb, Sym(0.0));
                std::function<void(int)> visit = [&](int ci) {
                    kinematicsCluster(ci, true, false);
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    for (int i = c.first_body_; i < c.first_body_ + c.joint_.num_bodies; i++)
                    {
                        const int p = m_.bodies()[i].parent_index_;
                        Xa[i] = p >= 0 ? bk_[i].Xl * Xa[p] : bk_[i].Xl;
                        for (int k = 0; k < 3; k++)
                            p_out[3 * i + k] = Xa[i].r[k];
                        for (int r = 0; r < 3; r++)
                            for (int cc = 0; cc < 3; cc++)
                                R_out[9 * i + 3 * r + cc] = Xa[i].E(cc, r);
                        const V3 w = mulT(Xa[i].E, bk_[i].v.ang()), vl = mulT(Xa[i].E, bk_[i].v.lin());
                        for (int k = 0; k < 3; k++)
                            v_out[6 * i + k] = w[k];
                        for (int k = 0; k < 3; k++)
                            v_out[6 * i + 3 + k] = vl[k];
                    }
                    for (int ch : children_[ci])
                        visit(ch);
                };
                for (int r : roots_)
                    visit(r);
            }

            // ---------------------------------------------------------------------------------
            // external forces (TreeModel::setExternalForces, TreeModel.cpp:189-193, ClusterTreeDynamics.cpp
            // :100-105): a world-frame spatial force f on body i enters RNEA and ABA as f_i -= Xa_i^* f. Both
            // recursions are linear in it, so  ID_ext = ID - J^T f  and  FD_ext(tau) = FD(tau + J^T f)  with
            // J^T f = the backward force pass over the transformed forces alone. This program evaluates
            // tau_in + sign J^T f for forces on the model's terminal links (feet, hands, chain tips).
            // ---------------------------------------------------------------------------------
            static std::vector<int> externalForceBodies(const ClusterTreeModel &model)
            {
                if (!model.externalForceBodies().empty())
                    return model.externalForceBodies(); // chosen by the caller (any bodies, rotors included)
                ModelCompiler probe(model);
                std::vector<char> has_child(model.getNumBodies(), 0);
                for (const Body &b : model.bodies())
                    if (b.parent_index_ >= 0)
                        has_child[b.parent_index_] = 1;
                std::vector<int> out;
                for (const Body &b : model.bodies())
                    if (!has_child[b.index_] && !probe.isAxisymmetricLeaf(b.index_))
                        out.push_back(b.index_);
                return out;
            }
            std::vector<Sym> generalizedExternalForce(int sign)
            {
                beginKinematics();
                const int Nb = m_.getNumBodies(), nv = m_.getNumDegreesOfFreedom();
                const std::vector<int> force_bodies = externalForceBodies(m_);
                std::vector<int> slot(Nb, -1);
                for (size_t k = 0; k < force_bodies.size(); k++)
                    slot[force_bodies[k]] = (int)k;
                std::vector<Xf> Xa(Nb);
                std::vector<SV> f(Nb);
                std::vector<Sym> tau(nv, Sym(0.0));
                auto isFree = [](const ClusterDesc &d) {
                    return d.type == ClusterType::FreeQuaternion || d.type == ClusterType::FreeRollPitchYaw;
                };
                std::function<void(int)> visit = [&](int ci) {
                    kinematicsCluster(ci, false, false);
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    const ClusterDesc &d = c.joint_;
                    const int N = d.num_bodies, n = d.num_velocities, b0 = c.first_body_;
                    for (int i = b0; i < b0 + N; i++)
                    {
                        const int p = m_.bodies()[i].parent_index_;
                        Xa[i] = p >= 0 ? bk_[i].Xl * Xa[p] : bk_[i].Xl;
                        if (slot[i] >= 0)
                        {
                            SV fw;
                            for (int k = 0; k < 6; k++)
                                fw[k] = Sym::input(IN_YD, 6 * slot[i] + k); // the force array travels in the velocity slot
                            f[i] = Xa[i].applyForce(fw);
                        }
                    }
                    for (int ch : children_[ci])
                        visit(ch);
                    for (int i = b0 + N - 1; i >= b0; i--)
                    {
                        const int p = m_.bodies()[i].parent_index_;
                        if (isFree(d))
                            for (int k = 0; k < 6; k++)
                                tau[c.velocity_index_ + k] = f[i][k];
                        else
                        {
                            const Sym tau_s = f[i][(int)d.axes[i - b0]];
                            for (int k = 0; k < n; k++)
                                tau[c.velocity_index_ + k] = tau[c.velocity_index_ + k] + ck_[ci].G[(i - b0) * n + k] * tau_s;
                        }
                        if (p >= 0)
                            f[p] = f[p] + bk_[i].Xl.applyForceTranspose(f[i]);
                    }
                };
                for (int r : roots_)
                    visit(r);
                std::vector<Sym> out(nv);
                for (int k = 0; k < nv; k++)
                {
                    const Sym t = Sym::input(IN_AUX, k);
                    out[k] = sign > 0 ? t + tau[k] : t - tau[k];
                }
                return out;
            }

            // ---------------------------------------------------------------------------------
            // inverse dynamics: spanning-tree RNEA + projection tau = G^T tau_s
            // ---------------------------------------------------------------------------------
            std::vector<Sym> inverseDynamics()
            {
                beginKinematics();
                const int Nb = m_.getNumBodies(), nv = m_.getNumDegreesOfFreedom();
                std::vector<SV> a(Nb), f(Nb);
                std::vector<Sym> tau(nv, Sym(0.0)), gyro_tau(Nb);

                auto downward = [&](int ci) {
                    kinematicsCluster(ci, true, false);
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    const ClusterDesc &d = c.joint_;
                    const int n = d.num_velocities;
                    std::vector<Sym> ydd(n);
                    for (int k = 0; k < n; k++)
                        ydd[k] = inAux(c.velocity_index_ + k);
                    const bool is_free = d.type == ClusterType::FreeQuaternion ||
                                         d.type == ClusterType::FreeRollPitchYaw;
                    for (int i = 0; i < d.num_bodies; i++)
                    {
                        const int bi = c.first_body_ + i;
                        const Body &body = m_.bodies()[bi];
                        const BodyKin &b = bk_[bi];
                        const int p = body.parent_index_;
                        if (isGyrostat(bi))
                        {
                            const ClusterKin &ck = ck_[c.index_];
                            Sym qdd = ck.g[i];
                            for (int k = 0; k < n; k++)
                                qdd = qdd + ck.G[i * n + k] * ydd[k];
                            gyro_tau[bi] = gyrostatForces(bi, b.qd, qdd, a[p], f[p]);
                            continue;
                        }
                        SV ai = b.Xl.applyMotion(p >= 0 ? a[p] : minusGravity());
                        if (is_free)
                        {
                            for (int k = 0; k < 6; k++)
                                ai[k] = ai[k] + ydd[k];
                        }
                        else
                        {
                            // qdd_s = G ydd + g
                            const ClusterKin &ck = ck_[c.index_];
                            Sym qdd = ck.g[i];
                            for (int k = 0; k < n; k++)
                                qdd = qdd + ck.G[i * n + k] * ydd[k];
                            const int axis = (int)d.axes[i];
                            SV sq;
                            sq[axis] = b.qd;
                            ai[axis] = ai[axis] + qdd;
                            ai = ai + motionCross(b.v, sq);
                        }
                        a[bi] = ai;
                        const RigidInertia I = bodyInertia(bi);
                        f[bi] = I.apply(ai) + forceCross(b.v, I.apply(b.v));
                    }
                };
                auto upward = [&](int ci) {
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    const ClusterDesc &d = c.joint_;
                    const int n = d.num_velocities;
                    const bool is_free = d.type == ClusterType::FreeQuaternion ||
                                         d.type == ClusterType::FreeRollPitchYaw;
                    std::map<int, SV> to_parent;
                    for (int i = d.num_bodies - 1; i >= 0; i--)
                    {
                        const int bi = c.first_body_ + i;
                        const int p = m_.bodies()[bi].parent_index_;
                        if (is_free)
                            for (int k = 0; k < 6; k++)
                                tau[c.velocity_index_ + k] = f[bi][k];
                        else
                        {
                            const ClusterKin &ck = ck_[c.index_];
                            const Sym tau_s = isGyrostat(bi) ? gyro_tau[bi] : f[bi][(int)d.axes[i]];
                            for (int k = 0; k < n; k++)
                                tau[c.velocity_index_ + k] = tau[c.velocity_index_ + k] + ck.G[i * n + k] * tau_s;
                        }
                        if (p >= 0 && !isGyrostat(bi))
                        {
                            const SV fp = bk_[bi].Xl.applyForceTranspose(f[bi]);
                            if (m_.getIndexOfClusterContainingBody(p) == ci)
                                f[p] = f[p] + fp; // in-cluster parent
                            else if (to_parent.count(p))
                                to_parent[p] = to_parent[p] + fp;
                            else
                                to_parent[p] = fp;
                        }
                    }
                    // one sum per parent body: the limb hands a single 6-vector to the trunk
                    for (auto &kv : to_parent)
                        f[kv.first] = f[kv.first] + kv.second;
                };
                std::function<void(int)> visit = [&](int ci) {
                    downward(ci);
                    for (int ch : children_[ci])
                        visit(ch);
                    upward(ci);
                };
                for (int r : roots_)
                    visit(r);
                return tau;
            }

            // ---------------------------------------------------------------------------------
            // derivatives of the inverse dynamics (SURVEY 8 f4): d tau / d dq and d tau / d yd, both nv x nv,
            // COLUMN-major (as Eigen and CasADi store the reference's Jacobians): element [j * nv + i] = d tau_i / d x_j;
            // a column is one tangent sweep, so the outputs of the program complete column by column.
            // (d tau / d ydd is the mass matrix.)
            // dq is the tangent-space perturbation of the reference's derivative test
            // (UnitTests/testHelpers.hpp:50-112, `plus`): q + dq for every one-dof coordinate; floating base
            // [p; quat] (+) [dw; dp] = [p + R^T dp; quat + 1/2 quat (x) (0, dw)] with R the rotation of
            // quaternionToRotationMatrix(quat). The reference test leaves implicit clusters out (its TODO at
            // testRigidBodyDynamicsAlgosDerivatives.cpp:166); here their spanning coordinates move along the
            // constraint manifold, dq_span = G(q) dy, the derivative with respect to the independent coordinates.
            // ---------------------------------------------------------------------------------
            std::vector<std::vector<std::pair<int, Sym>>> positionTangentMap()
            {
                const int nv = m_.getNumDegreesOfFreedom();
                std::vector<std::vector<std::pair<int, Sym>>> T(nv); // per direction: (position index, d q / d dq_j)
                for (const ClusterTreeNode &c : m_.clusters())
                {
                    const ClusterDesc &d = c.joint_;
                    const int pi = c.position_index_, vi = c.velocity_index_, n = d.num_velocities;
                    if (d.type == ClusterType::FreeQuaternion)
                    {
                        const Sym e0 = Sym::input(IN_Q, pi + 3), e1 = Sym::input(IN_Q, pi + 4), e2 = Sym::input(IN_Q, pi + 5),
                                  e3 = Sym::input(IN_Q, pi + 6);
                        const M3 E = quaternionToRotationMatrix(e0, e1, e2, e3);
                        const Sym h(0.5);
                        // 1/2 quat (x) (0, w): [-qv . w; e0 w + qv x w] / 2, columns = unit vectors w
                        const Sym dq4[4][3] = {{-(h * e1), -(h * e2), -(h * e3)},
                                               {h * e0, -(h * e3), h * e2},
                                               {h * e3, h * e0, -(h * e1)},
                                               {-(h * e2), h * e1, h * e0}};
                        for (int k = 0; k < 3; k++)
                        {
                            for (int r = 0; r < 4; r++)
                                T[vi + k].push_back({pi + 3 + r, dq4[r][k]});
                            for (int r = 0; r < 3; r++)
                                T[vi + 3 + k].push_back({pi + r, E(k, r)}); // (E^T)_{r k}
                        }
                    }
                    else if (d.type == ClusterType::FreeRollPitchYaw || d.type == ClusterType::Explicit)
                        for (int k = 0; k < n; k++)
                            T[vi + k].push_back({pi + k, Sym(1.0)});
                    else
                    {
                        const ClusterKin ck = clusterConstraint(c, false);
                        for (int k = 0; k < n; k++)
                            for (int i = 0; i < d.num_bodies; i++)
                                T[vi + k].push_back({pi + i, ck.G[i * n + k]});
                    }
                }
                return T;
            }
            void inverseDynamicsDerivatives(std::vector<Sym> &dtau_dq, std::vector<Sym> &dtau_dyd)
            {
                const int nv = m_.getNumDegreesOfFreedom();
                const std::vector<Sym> tau = inverseDynamics(); // ydd = inAux(): inputs, or placeholders (below)
                const auto T = positionTangentMap();
                dtau_dq.assign(nv * nv, Sym(0.0));
                dtau_dyd.assign(nv * nv, Sym(0.0));
                for (int j = 0; j < nv; j++)
                {
                    std::unordered_map<int32_t, Sym> seed;
                    for (auto &kv : T[j])
                        seed[Sym::input(IN_Q, kv.first).id] = kv.second;
                    const std::vector<Sym> col = tangentSweep(tau, seed);
                    for (int i = 0; i < nv; i++)
                        dtau_dq[j * nv + i] = col[i];
                    seed.clear();
                    seed[inYd(j).id] = Sym(1.0);
                    const std::vector<Sym> col_v = tangentSweep(tau, seed);
                    for (int i = 0; i < nv; i++)
                        dtau_dyd[j * nv + i] = col_v[i];
                }
            }

            // Derivatives of the forward dynamics by the implicit function theorem, tau = ID(q, yd, ydd):
            //   d ydd / d x = -H^-1 (d ID / d x) at ydd = FD(q, yd, tau),   d ydd / d tau = H^-1.
            // (The reference differentiates the forward dynamics the same way it does everything: CasADi's
            // jacobian() of the symbolic program, testRigidBodyDynamicsAlgosDerivatives.cpp:141-151 - there named
            // `inverseDynamics(tau)` but bound to the argument of forwardDynamics in the test's finite differences.)
            // The partial derivatives of ID are taken with placeholder accelerations (input array 3), which are then
            // replaced by the forward-dynamics expressions; every H^-1 column solve shares the one factorisation.
            void forwardDynamicsDerivatives(std::vector<Sym> &dydd_dq, std::vector<Sym> &dydd_dyd, std::vector<Sym> &dydd_dtau)
            {
                const int nv = m_.getNumDegreesOfFreedom();
                std::vector<Sym> placeholder(nv);
                for (int i = 0; i < nv; i++)
                    placeholder[i] = Sym::input(3, i);
                std::vector<Sym> d_q, d_yd;
                aux_override_ = &placeholder;
                inverseDynamicsDerivatives(d_q, d_yd);
                aux_override_ = nullptr;
                const std::vector<Sym> ydd = forwardDynamicsLTL();
                std::unordered_map<int32_t, Sym> values;
                for (int i = 0; i < nv; i++)
                    values[placeholder[i].id] = ydd[i];
                std::vector<Sym> all = d_q;
                all.insert(all.end(), d_yd.begin(), d_yd.end());
                all = substituteInputs(all, values);
                dydd_dq.assign(nv * nv, Sym(0.0));
                dydd_dyd.assign(nv * nv, Sym(0.0));
                dydd_dtau.assign(nv * nv, Sym(0.0));
                for (int j = 0; j < nv; j++)
                {
                    std::vector<Sym> bq(nv), bv(nv), e(nv, Sym(0.0));
                    for (int i = 0; i < nv; i++)
                        bq[i] = -all[j * nv + i], bv[i] = -all[nv * nv + j * nv + i];
                    e[j] = Sym(1.0);
                    const std::vector<Sym> xq = solveMassMatrix(bq), xv = solveMassMatrix(bv), xe = solveMassMatrix(e);
                    for (int i = 0; i < nv; i++)
                        dydd_dq[j * nv + i] = xq[i], dydd_dyd[j * nv + i] = xv[i], dydd_dtau[j * nv + i] = xe[i];
                }
            }

            // ---------------------------------------------------------------------------------
            // reverse mode: vector-Jacobian products of the dynamics. The cotangent w travels in input array 2
            // behind the third argument, [aux (nv); w (nv)]. q_bar is the gradient with respect to the STORED
            // position entries (nq of them, what torch.autograd needs): q_bar[k] = sum_i w_i d out_i / d q[k].
            // ---------------------------------------------------------------------------------
            std::vector<Sym> vjpPositions() const
            {
                std::vector<Sym> x(m_.getNumPositions());
                for (int k = 0; k < (int)x.size(); k++)
                    x[k] = Sym::input(IN_Q, k);
                return x;
            }
            // the n cotangent entries at input array 2, [first, first + n)
            std::vector<Sym> vjpCotangent(int n, int first) const
            {
                std::vector<Sym> w(n);
                for (int i = 0; i < n; i++)
                    w[i] = Sym::input(IN_AUX, first + i);
                return w;
            }

            // in2 = [ydd; tau_bar]: (q_bar, yd_bar, ydd_bar = H tau_bar), one reverse sweep of the inverse dynamics.
            // q_bar is the exact derivative of the inverse-dynamics program for every position entry, also off the
            // unit quaternion and off phi = 0.
            void inverseDynamicsVJP(std::vector<Sym> &q_bar, std::vector<Sym> &yd_bar, std::vector<Sym> &ydd_bar)
            {
                const int nq = m_.getNumPositions(), nv = m_.getNumDegreesOfFreedom();
                const std::vector<Sym> tau = inverseDynamics();
                std::vector<Sym> wrt = vjpPositions();
                for (int i = 0; i < nv; i++)
                    wrt.push_back(inYd(i));
                for (int i = 0; i < nv; i++)
                    wrt.push_back(inAux(i));
                const std::vector<Sym> bar = adjointSweep(tau, vjpCotangent(nv, nv), wrt);
                q_bar.assign(bar.begin(), bar.begin() + nq);
                yd_bar.assign(bar.begin() + nq, bar.begin() + nq + nv);
                ydd_bar.assign(bar.begin() + nq + nv, bar.end());
            }

            // in2 = [tau; ydd_bar]: (q_bar, yd_bar, tau_bar) by the implicit function theorem, as
            // forwardDynamicsDerivatives: with mu = H^-1 ydd_bar, tau_bar = mu and x_bar = -mu^T d ID / d x at
            // ydd = FD(q, yd, tau) - one reverse sweep of the inverse dynamics with placeholder accelerations (input
            // array 3), which are then replaced by the forward-dynamics expressions; the solve shares the one
            // factorisation. Contracted with a direction that keeps quaternions unit and implicit clusters on
            // phi = 0, q_bar equals w^T times the tangent Jacobian of forwardDynamicsDerivatives. Its component
            // normal to that set (quaternion norm, constraint violation) is the one of -H^-1 d ID / d q: it is not
            // the derivative of one particular forward-dynamics program off the set. A caller that normalises its
            // quaternion in its own graph drops that component anyway.
            void forwardDynamicsVJP(std::vector<Sym> &q_bar, std::vector<Sym> &yd_bar, std::vector<Sym> &tau_bar)
            {
                const int nq = m_.getNumPositions(), nv = m_.getNumDegreesOfFreedom();
                std::vector<Sym> placeholder(nv);
                for (int i = 0; i < nv; i++)
                    placeholder[i] = Sym::input(3, i);
                aux_override_ = &placeholder;
                const std::vector<Sym> id = inverseDynamics();
                aux_override_ = nullptr;
                tau_bar = solveMassMatrix(vjpCotangent(nv, nv));
                std::vector<Sym> neg_mu(nv);
                for (int i = 0; i < nv; i++)
                    neg_mu[i] = -tau_bar[i];
                std::vector<Sym> wrt = vjpPositions();
                for (int i = 0; i < nv; i++)
                    wrt.push_back(inYd(i));
                std::vector<Sym> bar = adjointSweep(id, neg_mu, wrt);
                const std::vector<Sym> ydd = forwardDynamicsLTL();
                std::unordered_map<int32_t, Sym> values;
                for (int i = 0; i < nv; i++)
                    values[placeholder[i].id] = ydd[i];
                bar = substituteInputs(bar, values);
                q_bar.assign(bar.begin(), bar.begin() + nq);
                yd_bar.assign(bar.begin() + nq, bar.end());
            }

            // in1 = f_ext [6 nf], in2 = w [nv]: (q_bar, f_bar) of tau_out = tau_in + sign J^T f, one reverse sweep of
            // generalizedExternalForce. The program is linear in tau_in and in f: tau_in_bar = w (left to the
            // caller), f_bar = sign J w. The cotangent sits where tau_in does (input array 2, entries 0..nv-1); it
            // only enters the sweep as the adjoint of the roots. q_bar is the exact derivative of the program for
            // every stored position entry.
            void externalForceVJP(int sign, std::vector<Sym> &q_bar, std::vector<Sym> &f_bar)
            {
                const int nq = m_.getNumPositions(), nv = m_.getNumDegreesOfFreedom();
                const int nf = (int)externalForceBodies(m_).size();
                const std::vector<Sym> tau = generalizedExternalForce(sign);
                std::vector<Sym> wrt = vjpPositions();
                for (int k = 0; k < 6 * nf; k++)
                    wrt.push_back(Sym::input(IN_YD, k));
                const std::vector<Sym> bar = adjointSweep(tau, vjpCotangent(nv, 0), wrt);
                q_bar.assign(bar.begin(), bar.begin() + nq);
                f_bar.assign(bar.begin() + nq, bar.end());
            }

            // in1 = yd, in2 = [p_bar (3 n_cp); v_bar (3 n_cp)]: (q_bar, yd_bar), one reverse sweep of
            // contactKinematics. yd_bar = J_lin^T v_bar (the contact velocities are linear in yd); q_bar is the exact
            // derivative of the program for every stored position entry, as for inverseDynamicsVJP.
            void contactKinematicsVJP(std::vector<Sym> &q_bar, std::vector<Sym> &yd_bar)
            {
                const int nq = m_.getNumPositions(), nv = m_.getNumDegreesOfFreedom();
                std::vector<Sym> roots, vel;
                contactKinematics(roots, vel);
                roots.insert(roots.end(), vel.begin(), vel.end());
                std::vector<Sym> wrt = vjpPositions();
                for (int i = 0; i < nv; i++)
                    wrt.push_back(inYd(i));
                const std::vector<Sym> bar = adjointSweep(roots, vjpCotangent((int)roots.size(), 0), wrt);
                q_bar.assign(bar.begin(), bar.begin() + nq);
                yd_bar.assign(bar.begin() + nq, bar.end());
            }

            // ---------------------------------------------------------------------------------
            // mass matrix: spanning-tree CRBA + projection H = G^T H_s G   (row-major nv x nv)
            // ---------------------------------------------------------------------------------
            std::vector<Sym> massMatrix()
            {
                kinematics(false, false);
                const int Nb = m_.getNumBodies(), nv = m_.getNumDegreesOfFreedom();
                std::vector<RigidInertia> Ic(Nb);
                for (int i = 0; i < Nb; i++)
                    Ic[i] = bodyInertia(i);
                for (int i = Nb - 1; i >= 0; i--)
                {
                    const int p = m_.bodies()[i].parent_index_;
                    if (p >= 0 && !isGyrostat(i))
                        Ic[p] = Ic[p] + Ic[i].toParent(bk_[i].Xl);
                }
                // spanning dofs: body i owns dof columns sdof[i] .. (+6 for the free body, +1 else)
                std::vector<int> sdof(Nb), sn(Nb);
                int ns = 0;
                for (const ClusterTreeNode &c : m_.clusters())
                    for (int i = 0; i < c.joint_.num_bodies; i++)
                    {
                        const bool is_free = c.joint_.type == ClusterType::FreeQuaternion ||
                                             c.joint_.type == ClusterType::FreeRollPitchYaw;
                        sdof[c.first_body_ + i] = ns;
                        sn[c.first_body_ + i] = is_free ? 6 : 1;
                        ns += sn[c.first_body_ + i];
                    }
                auto axisOf = [&](int body) {
                    const int ci = m_.getIndexOfClusterContainingBody(body);
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    return (int)c.joint_.axes[body - c.first_body_];
                };
                std::vector<Sym> Hs(ns * ns, Sym(0.0));
                for (int i = 0; i < Nb; i++)
                    for (int k = 0; k < sn[i]; k++)
                    {
                        const int col = sdof[i] + k;
                        SV F;
                        int j = i;
                        auto record = [&]() {
                            for (int l = 0; l < sn[j]; l++)
                            {
                                const Sym h = F[sn[j] == 6 ? l : axisOf(j)];
                                Hs[(sdof[j] + l) * ns + col] = h;
                                Hs[col * ns + sdof[j] + l] = h;
                            }
                        };
                        if (isGyrostat(i))
                        {
                            // own entry J, then the couple [J z; 0] on the parent
                            Hs[col * ns + col] = gyrostatInertia(i);
                            F = SV::make(gyrostatInertia(i) * gyrostatAxis(i), V3());
                            j = m_.bodies()[i].parent_index_;
                            record();
                        }
                        else
                        {
                            SV s;
                            s[sn[i] == 6 ? k : axisOf(i)] = Sym(1.0);
                            F = Ic[i].apply(s);
                            for (int l = 0; l < sn[i]; l++)
                                Hs[(sdof[i] + l) * ns + col] = F[sn[i] == 6 ? l : axisOf(i)];
                        }
                        while (m_.bodies()[j].parent_index_ >= 0)
                        {
                            F = bk_[j].Xl.applyForceTranspose(F);
                            j = m_.bodies()[j].parent_index_;
                            record();
                        }
                    }
                // projection with the block-diagonal G
                std::vector<std::vector<std::pair<int, Sym>>> Gcol(nv); // independent dof -> (spanning dof, G)
                for (const ClusterTreeNode &c : m_.clusters())
                {
                    const ClusterDesc &d = c.joint_;
                    const bool is_free = d.type == ClusterType::FreeQuaternion ||
                                         d.type == ClusterType::FreeRollPitchYaw;
                    if (is_free)
                    {
                        for (int k = 0; k < 6; k++)
                            Gcol[c.velocity_index_ + k].push_back({sdof[c.first_body_] + k, Sym(1.0)});
                        continue;
                    }
                    const ClusterKin &ck = ck_[c.index_];
                    for (int i = 0; i < d.num_bodies; i++)
                        for (int k = 0; k < d.num_velocities; k++)
                            if (!ck.G[i * d.num_velocities + k].isZero())
                                Gcol[c.velocity_index_ + k].push_back(
                                    {sdof[c.first_body_ + i], ck.G[i * d.num_velocities + k]});
                }
                std::vector<Sym> H(nv * nv, Sym(0.0));
                // columns from last to first: row b of H (entries to its ancestors from this step, to its
                // descendants from earlier steps) is then complete at step b, so the emitter can hand
                // finished 16-value chunks of the row-major output to the coalesced store path early
                for (int b = nv - 1; b >= 0; b--)
                {
                    // t = H_s G[:, b]
                    std::vector<Sym> t(ns, Sym(0.0));
                    for (auto &e : Gcol[b])
                        for (int r = 0; r < ns; r++)
                            t[r] = t[r] + Hs[r * ns + e.first] * e.second;
                    for (int a = 0; a <= b; a++)
                    {
                        Sym s(0.0);
                        for (auto &e : Gcol[a])
                            s = s + e.second * t[e.first];
                        H[a * nv + b] = s;
                        H[b * nv + a] = s;
                    }
                }
                return H;
            }

            // ---------------------------------------------------------------------------------
            // forward dynamics: constraint-embedded (cluster) articulated-body algorithm
            // ---------------------------------------------------------------------------------
            std::vector<Sym> forwardDynamics()
            {
                beginKinematics();
                const int Nb = m_.getNumBodies(), nv = m_.getNumDegreesOfFreedom(), Nc = m_.getNumClusters();

                // articulated inertia: rigid accumulator + general symmetric accumulator on the
                // diagonal; general blocks (i < j) off the diagonal within a cluster
                std::vector<RigidInertia> rigid(Nb);
                std::vector<SymInertia> gen(Nb);
                std::vector<char> has_gen(Nb, 0);
                std::map<std::pair<int, int>, M6> offdiag;
                std::vector<SV> pA(Nb);
                // downward sweep of one cluster: kinematics, rigid inertias, pA = v x* (I v)
                // (ClusterTreeDynamics.cpp:95-98)
                auto downward = [&](int ci) {
                    kinematicsCluster(ci, true, true);
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    for (int i = c.first_body_; i < c.first_body_ + c.joint_.num_bodies; i++)
                    {
                        rigid[i] = RigidInertia::fromMatrix(m_.bodies()[i].inertia_.getMatrix());
                        pA[i] = forceCross(bk_[i].v, rigid[i].apply(bk_[i].v));
                    }
                };
                auto applyIA = [&](int i, const SV &x) {
                    SV y = rigid[i].apply(x);
                    if (has_gen[i])
                        y = y + gen[i].apply(x);
                    return y;
                };

                struct ClusterABA
                {
                    std::vector<std::vector<SV>> U; // [body][column]
                    LDLT ldl;
                    std::vector<Sym> u;
                };
                std::vector<ClusterABA> aba(Nc);

                // upward sweep of one cluster (ClusterTreeDynamics.cpp:108-129,157-191)
                auto upward = [&](int ci) {
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    const int N = c.joint_.num_bodies, n = c.joint_.num_velocities, b0 = c.first_body_;
                    ClusterABA &A = aba[ci];
                    // c_i = cJ + avp
                    std::vector<SV> cb(N);
                    for (int i = 0; i < N; i++)
                        cb[i] = bk_[b0 + i].cJ + bk_[b0 + i].avp;
                    // U = IA S
                    A.U.assign(N, std::vector<SV>(n));
                    for (int i = 0; i < N; i++)
                        for (int k = 0; k < n; k++)
                        {
                            SV y = applyIA(b0 + i, bk_[b0 + i].S[k]);
                            for (int j = 0; j < N; j++)
                            {
                                if (j == i)
                                    continue;
                                auto it = offdiag.find({b0 + std::min(i, j), b0 + std::max(i, j)});
                                if (it == offdiag.end())
                                    continue;
                                y = y + (i < j ? it->second.apply(bk_[b0 + j].S[k])
                                               : it->second.applyTranspose(bk_[b0 + j].S[k]));
                            }
                            A.U[i][k] = y;
                        }
                    // D = S^T U, u = tau - S^T pA
                    std::vector<Sym> D(n * n);
                    A.u.assign(n, Sym(0.0));
                    for (int k = 0; k < n; k++)
                    {
                        for (int l = k; l < n; l++)
                        {
                            Sym s(0.0);
                            for (int i = 0; i < N; i++)
                                s = s + dot(bk_[b0 + i].S[k], A.U[i][l]);
                            D[k * n + l] = s;
                            D[l * n + k] = s;
                        }
                        Sym s = inAux(c.velocity_index_ + k);
                        for (int i = 0; i < N; i++)
                            s = s - dot(bk_[b0 + i].S[k], pA[b0 + i]);
                        A.u[k] = s;
                    }
                    A.ldl.factor(D, n);

                    if (c.parent_index_ < 0)
                        return;

                    // z = D^-1 (u - U^T c)
                    std::vector<Sym> t = A.u;
                    for (int k = 0; k < n; k++)
                        for (int i = 0; i < N; i++)
                            t[k] = t[k] - dot(A.U[i][k], cb[i]);
                    const std::vector<Sym> z = A.ldl.solve(t);
                    // pa_i = pA_i + sum_j IA_ij c_j + U_i z ; parent pA += X_i^T pa_i
                    // Everything this cluster hands to an ancestor body is summed first (one symmetric
                    // 6x6 + one 6-vector per ancestor), so a limb crosses the trunk cut with 27 values.
                    std::map<int, SV> pA_to;
                    std::map<int, SymInertia> IA_to;
                    auto addInertiaTo = [&](int anc, const SymInertia &I) {
                        auto it = IA_to.find(anc);
                        if (it == IA_to.end())
                            IA_to[anc] = I;
                        else
                            it->second = it->second + I;
                    };
                    for (int i = 0; i < N; i++)
                    {
                        SV pa = pA[b0 + i] + applyIA(b0 + i, cb[i]);
                        for (int j = 0; j < N; j++)
                        {
                            if (j == i)
                                continue;
                            auto it = offdiag.find({b0 + std::min(i, j), b0 + std::max(i, j)});
                            if (it == offdiag.end())
                                continue;
                            pa = pa + (i < j ? it->second.apply(cb[j]) : it->second.applyTranspose(cb[j]));
                        }
                        for (int k = 0; k < n; k++)
                            pa = pa + z[k] * A.U[i][k];
                        const int anc = bk_[b0 + i].anc;
                        const SV pa_p = bk_[b0 + i].Xup.applyForceTranspose(pa);
                        if (pA_to.count(anc))
                            pA_to[anc] = pA_to[anc] + pa_p;
                        else
                            pA_to[anc] = pa_p;
                    }
                    // parent IA += X^T IA X - W D^-1 W^T,   W_a = sum_{i -> a} X_i^T U_i
                    std::map<int, std::vector<SV>> W;
                    for (int i = 0; i < N; i++)
                    {
                        const int anc = bk_[b0 + i].anc;
                        auto &Wa = W[anc];
                        if (Wa.empty())
                            Wa.assign(n, SV());
                        for (int k = 0; k < n; k++)
                            Wa[k] = Wa[k] + bk_[b0 + i].Xup.applyForceTranspose(A.U[i][k]);
                        // diagonal blocks: rigid part transformed in 10-parameter form
                        addInertiaTo(anc, SymInertia::fromRigid(rigid[b0 + i].toParent(bk_[b0 + i].Xup)));
                        if (has_gen[b0 + i])
                            addInertiaTo(anc, gen[b0 + i].toParent(bk_[b0 + i].Xup));
                    }
                    // off-diagonal blocks of this cluster
                    for (auto &kv : offdiag)
                    {
                        const int i = kv.first.first, j = kv.first.second;
                        if (i < b0 || i >= b0 + N)
                            continue;
                        const int a = bk_[i].anc, b = bk_[j].anc;
                        const M6 M = transformBlock(bk_[i].Xup, kv.second, bk_[j].Xup);
                        addBlock(a, b, M, gen, has_gen, offdiag);
                    }
                    // V_a = W_a D^-1 (columns), then -(V_a W_b^T)
                    std::map<int, std::vector<SV>> V;
                    for (auto &kv : W)
                    {
                        std::vector<SV> Va(n);
                        for (int r = 0; r < 6; r++)
                        {
                            std::vector<Sym> row(n);
                            for (int k = 0; k < n; k++)
                                row[k] = kv.second[k][r];
                            const std::vector<Sym> x = A.ldl.solve(row);
                            for (int k = 0; k < n; k++)
                                Va[k][r] = x[k];
                        }
                        V[kv.first] = Va;
                    }
                    for (auto &ka : W)
                        for (auto &kb : W)
                        {
                            const int a = ka.first, b = kb.first;
                            if (a > b)
                                continue;
                            M6 M;
                            for (int r = 0; r < 6; r++)
                                for (int s = (a == b ? r : 0); s < 6; s++)
                                {
                                    Sym e(0.0);
                                    for (int k = 0; k < n; k++)
                                        e = e + V[a][k][r] * kb.second[k][s];
                                    M(r, s) = -e;
                                    if (a == b)
                                        M(s, r) = -e;
                                }
                            if (a == b)
                                addInertiaTo(a, symFromM6(M));
                            else
                                addBlock(a, b, M, gen, has_gen, offdiag);
                        }
                    for (auto &kv : IA_to)
                    {
                        gen[kv.first] = has_gen[kv.first] ? gen[kv.first] + kv.second : kv.second;
                        has_gen[kv.first] = 1;
                    }
                    for (auto &kv : pA_to)
                        pA[kv.first] = pA[kv.first] + kv.second;
                };
                std::function<void(int)> visit = [&](int ci) {
                    downward(ci);
                    for (int ch : children_[ci])
                        visit(ch);
                    upward(ci);
                };
                for (int r : roots_)
                    visit(r);

                // forward pass: accelerations (ClusterTreeDynamics.cpp:132-152), depth first as well
                std::vector<Sym> ydd_out(nv);
                std::vector<SV> a(Nb);
                std::vector<int> order;
                std::function<void(int)> collect = [&](int ci) {
                    order.push_back(ci);
                    for (int ch : children_[ci])
                        collect(ch);
                };
                for (int r : roots_)
                    collect(r);
                for (int ci : order)
                {
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    const int N = c.joint_.num_bodies, n = c.joint_.num_velocities, b0 = c.first_body_;
                    const ClusterABA &A = aba[ci];
                    const bool is_free = c.joint_.type == ClusterType::FreeQuaternion ||
                                         c.joint_.type == ClusterType::FreeRollPitchYaw;
                    std::vector<SV> at(N);
                    for (int i = 0; i < N; i++)
                    {
                        const BodyKin &b = bk_[b0 + i];
                        at[i] = b.Xup.applyMotion(b.anc >= 0 ? a[b.anc] : minusGravity()) + b.cJ + b.avp;
                    }
                    std::vector<Sym> ydd;
                    if (is_free)
                    {
                        // S = 1: ydd = D^-1 (u - D a') = D^-1 u - a'
                        ydd = A.ldl.solve(A.u);
                        for (int k = 0; k < 6; k++)
                            ydd[k] = ydd[k] - at[0][k];
                    }
                    else
                    {
                        std::vector<Sym> t = A.u;
                        for (int k = 0; k < n; k++)
                            for (int i = 0; i < N; i++)
                                t[k] = t[k] - dot(A.U[i][k], at[i]);
                        ydd = A.ldl.solve(t);
                    }
                    for (int k = 0; k < n; k++)
                        ydd_out[c.velocity_index_ + k] = ydd[k];
                    for (int i = 0; i < N; i++)
                    {
                        SV ai = at[i];
                        for (int k = 0; k < n; k++)
                            ai = ai + ydd[k] * bk_[b0 + i].S[k];
                        a[b0 + i] = ai;
                    }
                }
                return ydd_out;
            }

            // ---------------------------------------------------------------------------------
            // forward dynamics, second method: ydd = H^-1 (tau - C) with the cluster CRBA, the cluster
            // RNEA bias and a branch-sparse L^T D L factorisation, all inside ONE depth-first sweep.
            // Same result as forwardDynamics() (ClusterTreeModel::forwardDynamics,
            // ClusterTreeDynamics.cpp:10-19) up to rounding; the operands it must keep between the
            // upward and the final downward sweep are only the factor L (one value per
            // (dof, ancestor dof) pair) and z, about half of what the articulated-body sweep keeps
            // (U, D^-1, S, Xup, c per cluster), and composite inertias stay in 10-parameter form.
            //   upward step of cluster c (children finished):
            //     C_c      = G^T f                      (RNEA with ydd = 0, as inverseDynamics())
            //     H[c, a]  = S_a^T X^T (Ic S_c)         for every ancestor-or-self cluster a (cluster CRBA,
            //                                           ClusterTreeModel.cpp massMatrix)
            //     pivots k in c, last to first: row = H[k,:] - Acc[k,:], d = row[k], L[k,a] = row[a]/d,
            //     Acc[a,a'] += L[k,a] row[a'],  accb[a] += L[k,a] w_k,  w_k = tau_k - C_k - accb[k],  z_k = w_k/d
            //   final downward sweep: ydd_k = z_k - sum_a L[k,a] ydd_a
            // ---------------------------------------------------------------------------------
            std::vector<Sym> forwardDynamicsLTL()
            {
                beginKinematics();
                const int Nb = m_.getNumBodies(), nv = m_.getNumDegreesOfFreedom();
                std::vector<SV> a(Nb), f(Nb);
                std::vector<RigidInertia> Ic(Nb);
                std::vector<Sym> bias(nv, Sym(0.0)), z(nv), ydd_out(nv), gyro_tau(Nb);
                std::vector<std::vector<int>> anc_dofs(nv); // ancestor dofs of a dof, ascending
                std::vector<std::map<int, Sym>> L(nv);
                std::map<std::pair<int, int>, Sym> Acc;
                std::vector<Sym> accb(nv, Sym(0.0));
                auto accumulate = [](std::map<std::pair<int, int>, Sym> &M, int r, int c, const Sym &x) {
                    auto it = M.find({r, c});
                    if (it == M.end())
                        M[{r, c}] = x;
                    else
                        it->second = it->second + x;
                };
                auto isFree = [](const ClusterDesc &d) {
                    return d.type == ClusterType::FreeQuaternion || d.type == ClusterType::FreeRollPitchYaw;
                };

                std::map<std::string, long> trace;
                long mark = (long)Sym::G().nodes.size();
                auto phase = [&](const char *name) {
                    const long now = (long)Sym::G().nodes.size();
                    trace[name] += now - mark;
                    mark = now;
                };
                auto downward = [&](int ci) {
                    phase("other");
                    kinematicsCluster(ci, true, true);
                    phase("kinematics");
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    const ClusterDesc &d = c.joint_;
                    // dof ancestry: the parent cluster's last dof and its ancestors, then own earlier dofs
                    std::vector<int> path;
                    if (c.parent_index_ >= 0)
                    {
                        const ClusterTreeNode &pc = m_.clusters()[c.parent_index_];
                        const int last = pc.velocity_index_ + pc.joint_.num_velocities - 1;
                        path = anc_dofs[last];
                        path.push_back(last);
                    }
                    for (int k = 0; k < d.num_velocities; k++)
                    {
                        anc_dofs[c.velocity_index_ + k] = path;
                        path.push_back(c.velocity_index_ + k);
                    }
                    for (int i = 0; i < d.num_bodies; i++)
                    {
                        const int bi = c.first_body_ + i;
                        const Body &body = m_.bodies()[bi];
                        const BodyKin &b = bk_[bi];
                        const int p = body.parent_index_;
                        if (isGyrostat(bi))
                        {
                            gyro_tau[bi] = gyrostatForces(bi, b.qd, ck_[ci].g[i], a[p], f[p]);
                            continue;
                        }
                        SV ai = b.Xl.applyMotion(p >= 0 ? a[p] : minusGravity());
                        if (!isFree(d))
                        {
                            // ydd = 0: qdd_s = g
                            const int axis = (int)d.axes[i];
                            SV sq;
                            sq[axis] = b.qd;
                            ai[axis] = ai[axis] + ck_[ci].g[i];
                            ai = ai + motionCross(b.v, sq);
                        }
                        a[bi] = ai;
                        Ic[bi] = bodyInertia(bi);
                        f[bi] = Ic[bi].apply(ai) + forceCross(b.v, Ic[bi].apply(b.v));
                    }
                    phase("bias_down");
                };

                auto upward = [&](int ci) {
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    const ClusterDesc &d = c.joint_;
                    const int N = d.num_bodies, n = d.num_velocities, b0 = c.first_body_, v0 = c.velocity_index_;
                    // ---- bias force of this cluster (spanning-tree RNEA, projected with G) ----
                    {
                        std::map<int, SV> to_parent;
                        for (int i = N - 1; i >= 0; i--)
                        {
                            const int bi = b0 + i;
                            const int p = m_.bodies()[bi].parent_index_;
                            if (isFree(d))
                                for (int k = 0; k < 6; k++)
                                    bias[v0 + k] = f[bi][k];
                            else
                            {
                                const Sym tau_s = isGyrostat(bi) ? gyro_tau[bi] : f[bi][(int)d.axes[i]];
                                for (int k = 0; k < n; k++)
                                    bias[v0 + k] = bias[v0 + k] + ck_[ci].G[i * n + k] * tau_s;
                            }
                            if (p >= 0 && !isGyrostat(bi))
                            {
                                const SV fp = bk_[bi].Xl.applyForceTranspose(f[bi]);
                                if (m_.getIndexOfClusterContainingBody(p) == ci)
                                    f[p] = f[p] + fp;
                                else if (to_parent.count(p))
                                    to_parent[p] = to_parent[p] + fp;
                                else
                                    to_parent[p] = fp;
                            }
                        }
                        for (auto &kv : to_parent)
                            f[kv.first] = f[kv.first] + kv.second;
                    }
                    phase("bias_up");
                    // ---- rows of H owned by this cluster (cluster CRBA) ----
                    std::map<std::pair<int, int>, Sym> H; // (own dof, ancestor-or-own dof <= it)
                    for (int k = 0; k < n; k++)
                    {
                        std::map<int, SV> F_anc;
                        for (int i = 0; i < N; i++)
                        {
                            const BodyKin &b = bk_[b0 + i];
                            if (isGyrostat(b0 + i))
                            {
                                // J G_k G_l on the own dofs; the couple [J z G_k; 0] on the parent body
                                const Sym Gk = ck_[ci].G[i * n + k];
                                if (Gk.isZero())
                                    continue;
                                const Sym JG = gyrostatInertia(b0 + i) * Gk;
                                const int p = m_.bodies()[b0 + i].parent_index_;
                                const SV Fc = SV::make(JG * gyrostatAxis(b0 + i), V3());
                                for (int l = 0; l <= k; l++)
                                    accumulate(H, v0 + k, v0 + l, JG * ck_[ci].G[i * n + l]);
                                int target = p;
                                SV Ft = Fc;
                                if (p >= b0 && p < b0 + N)
                                {
                                    // parent inside this cluster: it moves with the own dofs as well
                                    for (int l = 0; l < n; l++)
                                    {
                                        const Sym h = dot(bk_[p].S[l], Fc);
                                        if (l <= k)
                                            accumulate(H, v0 + k, v0 + l, h);
                                        if (l >= k)
                                            accumulate(H, v0 + l, v0 + k, h);
                                    }
                                    target = bk_[p].anc;
                                    if (target >= 0)
                                        Ft = bk_[p].Xup.applyForceTranspose(Fc);
                                }
                                if (target >= 0)
                                {
                                    if (F_anc.count(target))
                                        F_anc[target] = F_anc[target] + Ft;
                                    else
                                        F_anc[target] = Ft;
                                }
                                continue;
                            }
                            const SV Fi = Ic[b0 + i].apply(b.S[k]);
                            for (int l = 0; l <= k; l++)
                                accumulate(H, v0 + k, v0 + l, dot(b.S[l], Fi));
                            if (b.anc < 0)
                                continue;
                            const SV Fp = b.Xup.applyForceTranspose(Fi);
                            if (F_anc.count(b.anc))
                                F_anc[b.anc] = F_anc[b.anc] + Fp;
                            else
                                F_anc[b.anc] = Fp;
                        }
                        for (auto &kv : F_anc)
                        {
                            int j = kv.first;
                            SV F = kv.second;
                            while (true)
                            {
                                const ClusterTreeNode &ac = m_.clusters()[m_.getIndexOfClusterContainingBody(j)];
                                for (int l = 0; l < ac.joint_.num_velocities; l++)
                                    accumulate(H, v0 + k, ac.velocity_index_ + l, dot(bk_[j].S[l], F));
                                if (bk_[j].anc < 0)
                                    break;
                                F = bk_[j].Xup.applyForceTranspose(F);
                                j = bk_[j].anc;
                            }
                        }
                    }
                    phase("crba_rows");
                    // ---- composite inertia handed to the ancestor bodies ----
                    {
                        std::map<int, RigidInertia> Ic_to;
                        for (int i = 0; i < N; i++)
                        {
                            const BodyKin &b = bk_[b0 + i];
                            if (b.anc < 0 || isGyrostat(b0 + i))
                                continue;
                            const RigidInertia Ip = Ic[b0 + i].toParent(b.Xup);
                            auto it = Ic_to.find(b.anc);
                            if (it == Ic_to.end())
                                Ic_to[b.anc] = Ip;
                            else
                                it->second = it->second + Ip;
                        }
                        for (auto &kv : Ic_to)
                            Ic[kv.first] = Ic[kv.first] + kv.second;
                    }
                    phase("crba_inertia");
                    // ---- pivots of this cluster, last to first ----
                    for (int k = v0 + n - 1; k >= v0; k--)
                    {
                        const std::vector<int> &anc = anc_dofs[k];
                        auto reduced = [&](int col) {
                            Sym h(0.0);
                            auto it = H.find({k, col});
                            if (it != H.end())
                                h = it->second;
                            auto ia = Acc.find({k, col});
                            if (ia != Acc.end())
                            {
                                h = h - ia->second;
                                Acc.erase(ia);
                            }
                            return h;
                        };
                        const Sym dk = reduced(k);
                        if (dk.isZero())
                            throw std::runtime_error("mass matrix has a structurally zero pivot");
                        const Sym dinv = Sym(1.0) / dk;
                        std::vector<Sym> row(anc.size());
                        for (size_t x = 0; x < anc.size(); x++)
                            row[x] = reduced(anc[x]);
                        const Sym w = inAux(k) - bias[k] - accb[k];
                        z[k] = w * dinv;
                        for (size_t x = 0; x < anc.size(); x++)
                        {
                            if (row[x].isZero())
                                continue;
                            const Sym l = row[x] * dinv;
                            L[k][anc[x]] = l;
                            for (size_t y = 0; y <= x; y++)
                                if (!row[y].isZero())
                                    accumulate(Acc, anc[x], anc[y], l * row[y]);
                            accb[anc[x]] = accb[anc[x]] + l * w;
                        }
                    }
                    phase("pivots");
                };
                // final downward sweep (ancestors first)
                auto solve = [&](int ci) {
                    const ClusterTreeNode &c = m_.clusters()[ci];
                    for (int k = c.velocity_index_; k < c.velocity_index_ + c.joint_.num_velocities; k++)
                    {
                        Sym x = z[k];
                        for (auto &kv : L[k])
                            x = x - kv.second * ydd_out[kv.first];
                        ydd_out[k] = x;
                    }
                };
                std::function<void(int)> visit = [&](int ci) {
                    downward(ci);
                    for (int ch : children_[ci])
                        visit(ch);
                    upward(ci);
                };
                // last limb first: its factor entries were produced last and are still in registers
                std::function<void(int)> visit2 = [&](int ci) {
                    solve(ci);
                    for (auto it = children_[ci].rbegin(); it != children_[ci].rend(); ++it)
                        visit2(*it);
                };
                for (int r : roots_)
                    visit(r);
                for (int r : roots_)
                    visit2(r);
                phase("solve");
                if (std::getenv("GRBDA_LTL_TRACE"))
                    for (auto &kv : trace)
                        std::fprintf(stderr, "ltl nodes %-14s %ld\n", kv.first.c_str(), kv.second);
                return ydd_out;
            }

            // ---------------------------------------------------------------------------------
            // operational space (SURVEY 8 f1): contact points, their Jacobians, apply-test-force, inverse OSIM
            // ---------------------------------------------------------------------------------
            // H^-1 b: the factorisation program with zero velocities and zero gravity (the bias vanishes
            // structurally) and b in the place of tau. Called once per right-hand side inside ONE graph scope:
            // hash-consing makes the kinematics, the mass matrix rows and the factor common to all of them.
            std::vector<Sym> solveMassMatrix(const std::vector<Sym> &b)
            {
                const std::vector<Sym> zeros(m_.getNumDegreesOfFreedom(), Sym(0.0));
                yd_override_ = &zeros;
                aux_override_ = &b;
                zero_gravity_ = true;
                std::vector<Sym> x = forwardDynamicsLTL();
                yd_override_ = aux_override_ = nullptr;
                zero_gravity_ = false;
                return x;
            }

            // absolute transform (world -> body) of every body and the kinematics the contact programs need
            void contactSetup(bool with_velocity, std::vector<Xf> &Xa)
            {
                const bool fr = freeze_leaves_;
                freeze_leaves_ = false; // a contact point may sit on any body: true poses everywhere
                kinematics(with_velocity, true);
                freeze_leaves_ = fr;
                Xa.assign(m_.getNumBodies(), Xf());
                for (int i = 0; i < m_.getNumBodies(); i++)
                {
                    const int p = m_.bodies()[i].parent_index_;
                    Xa[i] = p >= 0 ? bk_[i].Xl * Xa[p] : bk_[i].Xl;
                }
            }
            // TreeModel::contactPointForwardKinematics (TreeModel.cpp:60-78): world position and world linear
            // velocity of every contact point
            void contactKinematics(std::vector<Sym> &p_out, std::vector<Sym> &v_out)
            {
                std::vector<Xf> Xa;
                contactSetup(true, Xa);
                for (const ContactPoint &cp : m_.contactPoints())
                {
                    const Xf &X = Xa[cp.body_index_];
                    const V3 d = mulT(X.E, constV3(cp.local_offset_)); // offset in world orientation
                    const V3 pos = X.r + d;
                    const V3 w = mulT(X.E, bk_[cp.body_index_].v.ang()), vo = mulT(X.E, bk_[cp.body_index_].v.lin());
                    const V3 vel = vo + cross(w, d);
                    for (int k = 0; k < 3; k++)
                    {
                        p_out.push_back(pos[k]);
                        v_out.push_back(vel[k]);
                    }
                }
            }
            // contactJacobianWorldFrame (ClusterTreeDynamics.cpp:10-45): 6 x nv, [angular; linear] rows, world
            // orientation, at the contact point. Column of dof k of an ancestor cluster: the motion S_k of the
            // ancestor body (its own coordinates) seen at the contact point.
            std::vector<std::vector<Sym>> contactJacobianWorld(const ContactPoint &cp, const std::vector<Xf> &Xa) const
            {
                const int nv = m_.getNumDegreesOfFreedom();
                std::vector<std::vector<Sym>> J(6, std::vector<Sym>(nv, Sym(0.0)));
                const V3 pc = Xa[cp.body_index_].r + mulT(Xa[cp.body_index_].E, constV3(cp.local_offset_));
                for (int j = cp.body_index_; j >= 0; j = bk_[j].anc)
                {
                    const ClusterTreeNode &c = m_.clusters()[m_.getIndexOfClusterContainingBody(j)];
                    const V3 arm = pc - Xa[j].r;
                    for (int k = 0; k < c.joint_.num_velocities; k++)
                    {
                        const V3 w = mulT(Xa[j].E, bk_[j].S[k].ang()), v = mulT(Xa[j].E, bk_[j].S[k].lin()) + cross(w, arm);
                        for (int r = 0; r < 3; r++)
                        {
                            J[r][c.velocity_index_ + k] = w[r];
                            J[3 + r][c.velocity_index_ + k] = v[r];
                        }
                    }
                }
                return J;
            }
            // all contact points: [n_cp][6][nv], row-major
            std::vector<Sym> contactJacobians()
            {
                std::vector<Xf> Xa;
                contactSetup(false, Xa);
                std::vector<Sym> out;
                for (const ContactPoint &cp : m_.contactPoints())
                    for (auto &row : contactJacobianWorld(cp, Xa))
                        out.insert(out.end(), row.begin(), row.end());
                return out;
            }
            // applyTestForce (ClusterTreeDynamics.cpp:193-234): a world-frame force f on contact point c changes
            // the accelerations by dstate = H^-1 J_lin^T f; lambda_inv = f^T J_lin H^-1 J_lin^T f. f[3 n_cp] travels
            // in the velocity slot. out: dstate [n_cp][nv], lambda_inv [n_cp].
            void applyTestForce(std::vector<Sym> &dstate, std::vector<Sym> &lambda_inv)
            {
                const int nv = m_.getNumDegreesOfFreedom();
                std::vector<std::vector<Sym>> rhs;
                {
                    std::vector<Xf> Xa;
                    contactSetup(false, Xa);
                    int c = 0;
                    for (const ContactPoint &cp : m_.contactPoints())
                    {
                        const auto J = contactJacobianWorld(cp, Xa);
                        std::vector<Sym> t(nv, Sym(0.0));
                        for (int k = 0; k < nv; k++)
                            for (int r = 0; r < 3; r++)
                                t[k] = t[k] + J[3 + r][k] * Sym::input(IN_YD, 3 * c + r);
                        rhs.push_back(t);
                        c++;
                    }
                }
                for (const auto &t : rhs)
                {
                    const std::vector<Sym> x = solveMassMatrix(t);
                    Sym l(0.0);
                    for (int k = 0; k < nv; k++)
                        l = l + t[k] * x[k];
                    dstate.insert(dstate.end(), x.begin(), x.end());
                    lambda_inv.push_back(l);
                }
            }
            // inverseOperationalSpaceInertiaMatrix (ClusterTreeDynamics.cpp:292-435, the EFPA): Lambda^-1 =
            // J H^-1 J^T over the end-effectors, J = their 6 x nv Jacobians in the orientation of their own body
            // (the reference's X_offset = createSXform(1, local_offset)), [6 n_ee][6 n_ee] row-major.
            std::vector<Sym> inverseOperationalSpaceInertiaMatrix()
            {
                const int nv = m_.getNumDegreesOfFreedom();
                std::vector<std::vector<Sym>> Jb; // 6 n_ee rows
                {
                    std::vector<Xf> Xa;
                    contactSetup(false, Xa);
                    for (const ContactPoint &cp : m_.contactPoints())
                    {
                        if (!cp.is_end_effector_)
                            continue;
                        const auto Jw = contactJacobianWorld(cp, Xa);
                        const M3 &E = Xa[cp.body_index_].E;
                        for (int half = 0; half < 2; half++)
                            for (int r = 0; r < 3; r++)
                            {
                                std::vector<Sym> row(nv, Sym(0.0));
                                for (int k = 0; k < nv; k++)
                                    for (int cidx = 0; cidx < 3; cidx++)
                                        row[k] = row[k] + E(r, cidx) * Jw[3 * half + cidx][k];
                                Jb.push_back(row);
                            }
                    }
                }
                const int m = (int)Jb.size();
                std::vector<std::vector<Sym>> X(m); // H^-1 J^T, column by column
                for (int i = 0; i < m; i++)
                    X[i] = solveMassMatrix(Jb[i]);
                std::vector<Sym> out(m * m, Sym(0.0));
                for (int i = 0; i < m; i++)
                    for (int j = 0; j <= i; j++)
                    {
                        Sym s(0.0);
                        for (int k = 0; k < nv; k++)
                            s = s + Jb[i][k] * X[j][k];
                        out[i * m + j] = s;
                        out[j * m + i] = s;
                    }
                return out;
            }

            const std::vector<BodyKin> &bodyKinematics() const { return bk_; }
            const std::vector<ClusterKin> &clusterKinematics() const { return ck_; }

        private:
            static SymInertia symFromM6(const M6 &M)
            {
                SymInertia I;
                int k = 0;
                for (int i = 0; i < 3; i++)
                    for (int j = i; j < 3; j++)
                    {
                        I.A.a[k] = M(i, j);
                        I.C.a[k] = M(3 + i, 3 + j);
                        k++;
                    }
                for (int i = 0; i < 3; i++)
                    for (int j = 0; j < 3; j++)
                        I.B(i, j) = M(i, 3 + j);
                return I;
            }
            static void addSymmetric(int a, const M6 &M, std::vector<SymInertia> &gen, std::vector<char> &has_gen)
            {
                const SymInertia I = symFromM6(M);
                gen[a] = has_gen[a] ? gen[a] + I : I;
                has_gen[a] = 1;
            }
            // add block M at (a, b) of the articulated inertia (a != b: off-diagonal, stored for a < b;
            // a == b: M + M^T because both (i, j) and (j, i) land on the same diagonal block)
            static void addBlock(int a, int b, const M6 &M, std::vector<SymInertia> &gen,
                                 std::vector<char> &has_gen, std::map<std::pair<int, int>, M6> &offdiag)
            {
                if (a == b)
                {
                    addSymmetric(a, M + M.transposed(), gen, has_gen);
                    return;
                }
                const std::pair<int, int> key{std::min(a, b), std::max(a, b)};
                const M6 Mk = a < b ? M : M.transposed();
                auto it = offdiag.find(key);
                if (it == offdiag.end())
                    offdiag[key] = Mk;
                else
                    it->second = it->second + Mk;
            }

            void findAxisymmetricLeaves()
            {
                const int Nb = m_.getNumBodies();
                axisym_leaf_.assign(Nb, 0);
                std::vector<char> has_child(Nb, 0);
                for (const Body &b : m_.bodies())
                    if (b.parent_index_ >= 0)
                        has_child[b.parent_index_] = 1;
                for (const ClusterTreeNode &c : m_.clusters())
                {
                    const ClusterDesc &d = c.joint_;
                    if (d.type == ClusterType::FreeQuaternion || d.type == ClusterType::FreeRollPitchYaw)
                        continue;
                    for (int i = 0; i < d.num_bodies; i++)
                    {
                        const int bi = c.first_body_ + i;
                        if (has_child[bi])
                            continue;
                        const Mat6 &I = m_.bodies()[bi].inertia_.getMatrix();
                        const int a = (int)d.axes[i], o1 = (a + 1) % 3, o2 = (a + 2) % 3;
                        const double h[3] = {0.5 * (I[6 * 2 + 4] - I[6 * 1 + 5]), 0.5 * (I[6 * 0 + 5] - I[6 * 2 + 3]),
                                             0.5 * (I[6 * 1 + 3] - I[6 * 0 + 4])};
                        double scale = 0.0;
                        for (int r = 0; r < 3; r++)
                            for (int cc = 0; cc < 3; cc++)
                                scale = std::max(scale, std::fabs(I[6 * r + cc]));
                        const double tol = 1e-12 * scale, htol = 1e-12 * std::max(scale, std::fabs(I[35]));
                        const bool ok = std::fabs(h[o1]) <= htol && std::fabs(h[o2]) <= htol &&
                                        std::fabs(I[6 * a + o1]) <= tol && std::fabs(I[6 * a + o2]) <= tol &&
                                        std::fabs(I[6 * o1 + o2]) <= tol &&
                                        std::fabs(I[6 * o1 + o1] - I[6 * o2 + o2]) <= tol;
                        axisym_leaf_[bi] = ok ? 1 : 0;
                    }
                }
            }

            const ClusterTreeModel &m_;
            const std::vector<Sym> *yd_override_ = nullptr, *aux_override_ = nullptr;
            bool zero_gravity_ = false;
            bool freeze_leaves_ = true, gyrostats_ = true;
            std::vector<char> axisym_leaf_;
            std::vector<BodyKin> bk_;
            std::vector<ClusterKin> ck_;
            std::vector<std::vector<int>> children_;
            std::vector<int> roots_;
        };

    } // namespace compiler
} // namespace grbda
