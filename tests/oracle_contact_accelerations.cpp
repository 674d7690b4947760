// Test infrastructure: the oracle's classical contact-point accelerations, for tests/test_contact_dynamics.py.
// Compiled by that test into a library of its own together with the oracle's C API (the oracle itself is unchanged),
// it reads the handles of oracle/liboracle.so (same source, same layout of Handle).
#include "oracle_capi.cpp"

extern "C"
{
    // acc: [batch][n_cp][3], the classical world acceleration of every contact point at (q, yd, ydd) WITHOUT gravity:
    // forwardAccelerationKinematics with the gravity set to zero, then, with the body's world-frame spatial velocity
    // (w, v0) and acceleration (wd, a0) at the world origin and the point's world position p,
    // a0 + wd x p + w x (v0 + w x p)
    int oracle_contact_accelerations(void *hv, const double *q, const double *yd, const double *ydd, double *acc,
                                     int64_t batch, int threads)
    {
        Handle *h = (Handle *)hv;
        const int nq = h->model->getNumPositions(), nv = h->model->getNumDegreesOfFreedom();
        const int nc = (int)h->model->contact_points.size();
        return runBatch(h, batch, threads, [&](ClusterTreeModel<double> &m, int64_t b)
                        {
                            m.setState(toVec(q + b * nq, nq), toVec(yd + b * nv, nv));
                            const Mat<double> gravity = m.gravity;
                            m.gravity = Mat<double>(6, 1);
                            m.forwardAccelerationKinematics(toVec(ydd + b * nv, nv));
                            m.gravity = gravity;
                            auto cross = [](const double *x, const double *y, double *z) {
                                z[0] = x[1] * y[2] - x[2] * y[1], z[1] = x[2] * y[0] - x[0] * y[2], z[2] = x[0] * y[1] - x[1] * y[0];
                            };
                            for (int c = 0; c < nc; c++)
                            {
                                const auto &cp = m.contact_points[c];
                                const int sub = m.bodies[cp.body_index].sub_index_within_cluster;
                                auto &node = m.nodes[m.clusterContainingBody(cp.body_index)];
                                const auto &Xa = node->Xa[sub];
                                const Mat<double> vw = Xa.inverseTransformMotionVector(node->v.segment(6 * sub, 6));
                                const Mat<double> aw = Xa.inverseTransformMotionVector(node->a.segment(6 * sub, 6));
                                const Mat<double> p = Xa.inverseTransformPoint(cp.local_offset);
                                const double w[3] = {vw[0], vw[1], vw[2]}, wd[3] = {aw[0], aw[1], aw[2]}, pp[3] = {p[0], p[1], p[2]};
                                double wxp[3], wdxp[3], vp[3], wxvp[3];
                                cross(w, pp, wxp);
                                cross(wd, pp, wdxp);
                                for (int i = 0; i < 3; i++)
                                    vp[i] = vw[3 + i] + wxp[i];
                                cross(w, vp, wxvp);
                                for (int i = 0; i < 3; i++)
                                    acc[(b * nc + c) * 3 + i] = aw[3 + i] + wdxp[i] + wxvp[i];
                            } });
    }
}
