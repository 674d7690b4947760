// Device-side model compiler, part 3: driver. Model + algorithm -> emitted CUDA body, tape, counts.
#pragma once
#include <fstream>
#include <ostream>
#include <sstream>
#include "algorithms.h"
#include "emit.h"

namespace grbda
{
    namespace compiler
    {
        enum Algo
        {
            ALGO_ID = 0,      // in: q, yd, ydd   out: tau[nv]
            ALGO_FD = 1,      // in: q, yd, tau   out: ydd[nv]
            ALGO_FK = 2,      // in: q, yd        out: p[3 Nb], R[9 Nb], v[6 Nb]
            ALGO_H = 3,       // in: q            out: H[nv nv]
            ALGO_PHI = 4,     // in: q            out: phi[sum nc], Kd (row-major per implicit cluster)
            // generalized force of external forces on the model's terminal links (ModelCompiler::
            // externalForceBodies): in: q, f_ext[6 nf] (world frame, TreeModel::setExternalForces), tau_in
            ALGO_GFA = 5,     // out: tau_in + J^T f_ext   (forward dynamics with external forces: FD(.., tau + J^T f))
            ALGO_GFS = 6,     // out: tau_in - J^T f_ext   (inverse dynamics with external forces: ID(..) - J^T f)
            ALGO_COUNT = 7,   // entry points / registry slots
            // alternative programs of an entry point (selected per kernel variant, same I/O as the entry)
            PROGRAM_FD_LTL = 7, // forward dynamics as H^-1 (tau - C): CRBA + RNEA bias + sparse L^T D L
            // operational space (model.contactPoints()); always compiled at run time for the contact set
            ALGO_CONTACT_KIN = 8,  // in: q, yd          out: p_c[3 n_cp], v_c[3 n_cp] (world)
            ALGO_CONTACT_JAC = 9,  // in: q              out: J[n_cp][6][nv] (world frame, [angular; linear])
            ALGO_TEST_FORCE = 10,  // in: q, f[3 n_cp]   out: dstate[n_cp][nv], lambda_inv[n_cp]
            ALGO_OSIM = 11,        // in: q              out: Lambda^-1 [6 n_ee][6 n_ee]
            // derivatives (SURVEY 8 f4; compiled at run time when first used): column-major, [j nv + i] = d out_i / d x_j,
            // dq = tangent-space perturbation of the positions (ModelCompiler::positionTangentMap)
            ALGO_ID_DERIV = 12,    // in: q, yd, ydd     out: dtau/ddq [nv nv], dtau/dyd [nv nv]
            ALGO_FD_DERIV = 13,    // in: q, yd, tau     out: dydd/ddq [nv nv], dydd/dyd [nv nv], dydd/dtau = H^-1 [nv nv]
            // reverse mode (compiled at run time when first used): the cotangent w travels behind the third argument
            // in input array 2; q_bar is the gradient with respect to the nq stored position entries
            ALGO_ID_VJP = 14,      // in: q, yd, [ydd; w]  out: q_bar [nq], yd_bar [nv], ydd_bar = H w [nv]
            ALGO_FD_VJP = 15,      // in: q, yd, [tau; w]  out: q_bar [nq], yd_bar [nv], tau_bar = H^-1 w [nv]
            // reverse mode of the external-force programs 5 / 6 (tau_in_bar = w is left to the caller) and of the
            // contact kinematics 8: the cotangent is input array 2 itself
            ALGO_GFA_VJP = 16,     // in: q, f_ext [6 nf], w [nv]   out: q_bar [nq], f_bar = J w [6 nf]
            ALGO_GFS_VJP = 17,     // in: q, f_ext [6 nf], w [nv]   out: q_bar [nq], f_bar = -J w [6 nf]
            ALGO_CONTACT_KIN_VJP = 18, // in: q, yd, [p_bar; v_bar] [6 n_cp]   out: q_bar [nq], yd_bar = J_lin^T v_bar [nv]
            PROGRAM_COUNT = 19
        };
        // registry slot a program belongs to
        inline int algoOfProgram(int program) { return program == PROGRAM_FD_LTL ? ALGO_FD : program; }
        inline const char *algoName(int a)
        {
            static const char *names[] = {"id", "fd", "fk", "h", "phi", "gfa", "gfs", "fd_ltl", "contact_kin", "contact_jac",
                                          "test_force", "osim", "id_deriv", "fd_deriv", "id_vjp", "fd_vjp", "gfa_vjp", "gfs_vjp",
                                          "contact_kin_vjp"};
            return names[a];
        }

        struct CompiledAlgo
        {
            std::string name;
            int n_in[3] = {0, 0, 0};
            int n_out[3] = {0, 0, 0};
            std::string body;
            std::string range_check; // expression: may the fast sin/cos forms be used for this state
            bool parked = false;     // body parks long-lived values in the thread's shared-memory row
            int num_parked = 0;
            int park_extra = 0;      // slots per thread of the park area behind the tiles (parked bodies)
            bool direct_out = false; // output 0 is stored straight to global memory although it is small (no output tile)
            int stage_buffers = 1;   // chunked outputs: staging buffers per warp (1, or one per output array)
            bool vector_stores = false; // large outputs leave as 256-bit stores of the thread's own row (emit.h)
            bool ring_stores = false;   // ... assembled in per-thread shared-memory rings (emit.h, row_stores = 2)
            ProgramStats stats;
            Tape tape;
        };

        // Input / output sizes of one program without building it (launch-shape decisions need them first).
        inline void algoSizes(const ClusterTreeModel &model, int program, int n_in[3], int n_out[3])
        {
            const int nq = model.getNumPositions(), nv = model.getNumDegreesOfFreedom(), nb = model.getNumBodies();
            n_in[0] = nq, n_in[1] = n_in[2] = 0;
            n_out[0] = n_out[1] = n_out[2] = 0;
            switch (program)
            {
            case ALGO_ID:
            case ALGO_FD:
            case PROGRAM_FD_LTL:
                n_in[1] = n_in[2] = nv, n_out[0] = nv;
                break;
            case ALGO_GFA:
            case ALGO_GFS:
                n_in[1] = 6 * (int)ModelCompiler::externalForceBodies(model).size(), n_in[2] = nv, n_out[0] = nv;
                break;
            case ALGO_FK:
                n_in[1] = nv, n_out[0] = 3 * nb, n_out[1] = 9 * nb, n_out[2] = 6 * nb;
                break;
            case ALGO_H:
                n_out[0] = nv * nv;
                break;
            case ALGO_PHI:
                for (const ClusterTreeNode &c : model.clusters())
                    if (c.joint_.type == ClusterType::Implicit)
                    {
                        n_out[0] += c.joint_.num_constraints;
                        n_out[1] += c.joint_.num_constraints * (c.joint_.num_bodies - c.joint_.num_velocities);
                    }
                break;
            case ALGO_CONTACT_KIN:
                n_in[1] = nv, n_out[0] = n_out[1] = 3 * (int)model.contactPoints().size();
                break;
            case ALGO_CONTACT_JAC:
                n_out[0] = 6 * nv * (int)model.contactPoints().size();
                break;
            case ALGO_TEST_FORCE:
                n_in[1] = 3 * (int)model.contactPoints().size();
                n_out[0] = nv * (int)model.contactPoints().size(), n_out[1] = (int)model.contactPoints().size();
                break;
            case ALGO_OSIM:
                n_out[0] = 36 * model.getNumEndEffectors() * model.getNumEndEffectors();
                break;
            case ALGO_ID_DERIV:
                n_in[1] = n_in[2] = nv, n_out[0] = n_out[1] = nv * nv;
                break;
            case ALGO_FD_DERIV:
                n_in[1] = n_in[2] = nv, n_out[0] = n_out[1] = n_out[2] = nv * nv;
                break;
            case ALGO_ID_VJP:
            case ALGO_FD_VJP:
                n_in[1] = nv, n_in[2] = 2 * nv, n_out[0] = nq, n_out[1] = n_out[2] = nv;
                break;
            case ALGO_GFA_VJP:
            case ALGO_GFS_VJP:
                n_in[1] = 6 * (int)ModelCompiler::externalForceBodies(model).size(), n_in[2] = nv;
                n_out[0] = nq, n_out[1] = n_in[1];
                break;
            case ALGO_CONTACT_KIN_VJP:
                n_in[1] = nv, n_in[2] = 6 * (int)model.contactPoints().size(), n_out[0] = nq, n_out[1] = nv;
                break;
            default:
                throw std::runtime_error("algoSizes: unknown program");
            }
        }

        // Build the symbolic program of one algorithm in the CURRENT graph scope.
        inline Program buildProgram(const ClusterTreeModel &model, int algo)
        {
            ModelCompiler mc(model);
            Program p;
            p.name = algoName(algo);
            const int nq = model.getNumPositions(), nv = model.getNumDegreesOfFreedom();
            switch (algo)
            {
            case ALGO_ID:
                p.n_in[0] = nq, p.n_in[1] = nv, p.n_in[2] = nv;
                p.outputs.push_back(mc.inverseDynamics());
                break;
            case ALGO_FD:
                p.n_in[0] = nq, p.n_in[1] = nv, p.n_in[2] = nv;
                p.outputs.push_back(mc.forwardDynamics());
                break;
            case PROGRAM_FD_LTL:
                p.n_in[0] = nq, p.n_in[1] = nv, p.n_in[2] = nv;
                p.outputs.push_back(mc.forwardDynamicsLTL());
                break;
            case ALGO_GFA:
            case ALGO_GFS:
                p.n_in[0] = nq, p.n_in[1] = 6 * (int)ModelCompiler::externalForceBodies(model).size(), p.n_in[2] = nv;
                p.outputs.push_back(mc.generalizedExternalForce(algo == ALGO_GFA ? 1 : -1));
                break;
            case ALGO_FK:
            {
                p.n_in[0] = nq, p.n_in[1] = nv;
                std::vector<sym::Sym> pp, R, v;
                mc.setFreezeAxisymmetricLeaves(false); // the outputs are the poses themselves
                mc.forwardKinematics(pp, R, v);
                p.outputs = {pp, R, v};
                break;
            }
            case ALGO_H:
                p.n_in[0] = nq;
                p.outputs.push_back(mc.massMatrix());
                break;
            case ALGO_PHI:
            {
                // constraint violation and K_d of every implicit cluster (state generation / validity)
                p.n_in[0] = nq;
                std::vector<sym::Sym> phi_all, Kd_all;
                for (const ClusterTreeNode &c : model.clusters())
                {
                    if (c.joint_.type != ClusterType::Implicit)
                        continue;
                    const ClusterDesc &d = c.joint_;
                    std::vector<sym::Sym> q(d.num_bodies), phi, K;
                    for (int i = 0; i < d.num_bodies; i++)
                        q[i] = sym::Sym::input(IN_Q, c.position_index_ + i);
                    mc.implicitJacobian(d, q, nullptr, phi, K, nullptr);
                    for (auto &x : phi)
                        phi_all.push_back(x);
                    for (int i = 0; i < d.num_constraints; i++)
                        for (int j = 0; j < d.num_bodies; j++)
                            if (!d.independent[j])
                                Kd_all.push_back(K[i * d.num_bodies + j]);
                }
                p.outputs = {phi_all, Kd_all};
                break;
            }
            case ALGO_CONTACT_KIN:
            {
                p.n_in[0] = nq, p.n_in[1] = nv;
                std::vector<sym::Sym> pos, vel;
                mc.contactKinematics(pos, vel);
                p.outputs = {pos, vel};
                break;
            }
            case ALGO_CONTACT_JAC:
                p.n_in[0] = nq;
                p.outputs.push_back(mc.contactJacobians());
                break;
            case ALGO_TEST_FORCE:
            {
                p.n_in[0] = nq, p.n_in[1] = 3 * (int)model.contactPoints().size();
                std::vector<sym::Sym> dstate, lambda_inv;
                mc.applyTestForce(dstate, lambda_inv);
                p.outputs = {dstate, lambda_inv};
                break;
            }
            case ALGO_OSIM:
                p.n_in[0] = nq;
                p.outputs.push_back(mc.inverseOperationalSpaceInertiaMatrix());
                break;
            case ALGO_ID_DERIV:
            {
                p.n_in[0] = nq, p.n_in[1] = nv, p.n_in[2] = nv;
                std::vector<sym::Sym> dq, dyd;
                mc.inverseDynamicsDerivatives(dq, dyd);
                p.outputs = {dq, dyd};
                break;
            }
            case ALGO_FD_DERIV:
            {
                p.n_in[0] = nq, p.n_in[1] = nv, p.n_in[2] = nv;
                std::vector<sym::Sym> dq, dyd, dtau;
                mc.forwardDynamicsDerivatives(dq, dyd, dtau);
                p.outputs = {dq, dyd, dtau};
                break;
            }
            case ALGO_ID_VJP:
            case ALGO_FD_VJP:
            {
                p.n_in[0] = nq, p.n_in[1] = nv, p.n_in[2] = 2 * nv;
                std::vector<sym::Sym> q_bar, yd_bar, aux_bar;
                if (algo == ALGO_ID_VJP)
                    mc.inverseDynamicsVJP(q_bar, yd_bar, aux_bar);
                else
                    mc.forwardDynamicsVJP(q_bar, yd_bar, aux_bar);
                p.outputs = {q_bar, yd_bar, aux_bar};
                break;
            }
            case ALGO_GFA_VJP:
            case ALGO_GFS_VJP:
            {
                p.n_in[0] = nq, p.n_in[1] = 6 * (int)ModelCompiler::externalForceBodies(model).size(), p.n_in[2] = nv;
                std::vector<sym::Sym> q_bar, f_bar;
                mc.externalForceVJP(algo == ALGO_GFA_VJP ? 1 : -1, q_bar, f_bar);
                p.outputs = {q_bar, f_bar};
                break;
            }
            case ALGO_CONTACT_KIN_VJP:
            {
                p.n_in[0] = nq, p.n_in[1] = nv, p.n_in[2] = 6 * (int)model.contactPoints().size();
                std::vector<sym::Sym> q_bar, yd_bar;
                mc.contactKinematicsVJP(q_bar, yd_bar);
                p.outputs = {q_bar, yd_bar};
                break;
            }
            default:
                throw std::runtime_error("compileAlgo: unknown algorithm");
            }
            return p;
        }

        inline CompiledAlgo compileAlgo(const ClusterTreeModel &model, int algo, bool want_body = true,
                                        int sync_every = 0, ConstTable *consts = nullptr, int out_chunk = 0,
                                        bool park = false, bool allow_vector_stores = true, int park_extra = 0,
                                        bool direct_out = false)
        {
            sym::Graph graph;
            sym::GraphScope scope(graph);
            const Program p = buildProgram(model, algo);
            CompiledAlgo out;
            out.name = p.name;
            for (int i = 0; i < 3; i++)
                out.n_in[i] = p.n_in[i];
            for (size_t i = 0; i < p.outputs.size(); i++)
                out.n_out[i] = (int)p.outputs[i].size();
            Emitter em(graph, p, consts);
            out.stats = em.stats();
            out.tape = em.tape();
            if (want_body)
            {
                ParkConfig pc;
                for (int i = 0; i < 3; i++)
                    pc.n_slots[i] = p.n_in[i];
                pc.n_slots[3] = out.n_out[0] <= 64 && !direct_out ? out.n_out[0] : 0; // the shells stage output 0 when it is small
                pc.n_slots[4] = park_extra;                            // park area behind the tiles
                // Programs with large outputs (mass matrix) hold their results until a 16-value chunk is complete: many
                // values that wait a few hundred statements each, not a few that wait for half the program. Measured
                // on B200 (TelloWithArms / MIT humanoid mass matrix, 2^18 states, unparked 0.278 / 0.279 ms): gap 300 ->
                // 0.263 / 0.265, 100 -> 0.247 / 0.256, 50 -> 0.248 / 0.259, 20 -> 0.260 / 0.276 ms
                if (grbda_kernels::shapeChunkStageBytes(out.n_out, 1, 32, 8) > 0)
                    pc.min_gap = 100;
                if (const char *gap = std::getenv("GRBDA_PARK_GAP")) // tuning experiments
                    pc.min_gap = std::atoi(gap);
                out.parked = park && sync_every == 0;
                // how large in-order outputs (forward kinematics) leave: rings (default), predicated register quads
                // ("pred": needs CTAs of four warps - the caller says whether its launch shape has them) or the chunk
                // staging every other large output uses ("chunk"); GRBDA_ROW_STORES selects, for A/B timing
                const char *rs = std::getenv("GRBDA_ROW_STORES");
                int row_stores = 2;
                if (rs && std::string(rs) == "pred")
                    row_stores = allow_vector_stores ? 1 : 0;
                else if (rs && std::string(rs) == "chunk")
                    row_stores = 0;
                if (std::getenv("GRBDA_NO_VECTOR_STORES") && std::getenv("GRBDA_NO_VECTOR_STORES")[0] == '1')
                    row_stores = 0;
                out.body = em.cudaBody(sync_every, out_chunk, out.parked ? &pc : nullptr, row_stores);
                out.num_parked = em.numParked();
                out.park_extra = out.parked ? park_extra : 0;
                out.direct_out = direct_out && out.n_out[0] <= 64;
                out.stage_buffers = em.stageBuffers();
                out.vector_stores = em.vectorStores();
                out.ring_stores = em.ringStores();
                out.range_check = em.cudaRangeCheck();
            }
            return out;
        }

        // Which program runs forwardDynamics by default. Both are ClusterTreeModel::forwardDynamics; the
        // factorisation (cluster CRBA + bias + branch-sparse L^T D L) keeps far fewer values alive between its two
        // sweeps and wins on floating-base robots with short limbs, the articulated-body sweep is O(depth) and
        // wins on deep chains. Measured on B200 (profiles/r2_fd_program_sweep.jsonl, 15 models): the
        // factorisation is the faster kernel exactly when it executes fewer than ~0.85 x the operations of the
        // sweep (Tello 0.77 -> 2.3x faster; 8-link chain 0.91 -> 1.7x slower; 24-link chain 2.85 -> 6x slower).
        inline int chooseForwardDynamicsProgram(const ClusterTreeModel &model)
        {
            if (const char *force = std::getenv("GRBDA_FD_PROGRAM")) // "aba" / "ltl": experiments
                return std::string(force) == "aba" ? (int)ALGO_FD : (int)PROGRAM_FD_LTL;
            auto flops = [&](int program) {
                sym::Graph graph;
                sym::GraphScope scope(graph);
                const Program p = buildProgram(model, program);
                return (double)Emitter(graph, p).stats().flops();
            };
            return flops(PROGRAM_FD_LTL) < 0.85 * flops(ALGO_FD) ? (int)PROGRAM_FD_LTL : (int)ALGO_FD;
        }

        // The generated `struct Body` of one program: sizes, range check, run<real, FAST>(). Shared by the
        // build-time tool (tools/modelc.cpp) and grbda_cuda_emit_source (host-compiled emitter self test).
        inline void emitBodyStruct(std::ostream &os, const std::string &struct_name, const CompiledAlgo &c)
        {
            os << "struct " << struct_name << "\n{\n";
            os << "    static constexpr int N_IN0 = " << c.n_in[0] << ", N_IN1 = " << c.n_in[1]
               << ", N_IN2 = " << c.n_in[2] << ";\n";
            os << "    static constexpr int N_OUT0 = " << c.n_out[0] << ", N_OUT1 = " << c.n_out[1]
               << ", N_OUT2 = " << c.n_out[2] << ";\n";
            os << "    static constexpr bool RANGE_CHECKED = " << (c.range_check == "true" ? "false" : "true") << ";\n";
            os << "    static constexpr int STAGE_BUFFERS = " << c.stage_buffers << ";\n";
            os << "    static constexpr bool VECTOR_STORES = " << (c.vector_stores ? "true" : "false") << ";\n";
            os << "    static constexpr bool RING_STORES = " << (c.ring_stores ? "true" : "false") << ";\n";
            os << "    static constexpr bool PARKED = " << (c.parked ? "true" : "false") << "; // " << c.num_parked
               << " values parked in the thread's tile row\n";
            os << "    static constexpr int PARK_EXTRA = " << c.park_extra << ";\n";
            os << "    static constexpr bool DIRECT_OUT0 = " << (c.direct_out ? "true" : "false") << ";\n";
            os << "    template <typename real>\n    static __device__ __forceinline__ bool inRange(const real "
                  "*__restrict__ in0, const real *__restrict__ in1,\n        const real *__restrict__ in2)\n    {\n"
                  "#define KC(x) ((real)(x))\n#define IN0(i) in0[i]\n#define IN1(i) in1[i]\n#define IN2(i) in2[i]\n"
                  "        return " << c.range_check << ";\n#undef KC\n#undef IN0\n#undef IN1\n#undef IN2\n    }\n";
            os << "    template <typename real, bool FAST>\n";
            if (c.parked)
                // the thread's rows are read AND written (parking): no __restrict__, one pointer per row
                os << "    static __device__ __forceinline__ void run(const real *in0, const real *in1, const real *in2,\n"
                      "        real *out0, real *out1, real *out2, const OutStage<real> &stage)\n    {\n"
                      "        real *const row0 = const_cast<real *>(in0), *const row1 = const_cast<real *>(in1),\n"
                      "                   *const row2 = const_cast<real *>(in2), *const row3 = out0, *const row4 = stage.park;\n"
                      "#define IN0(i) row0[i]\n#define IN1(i) row1[i]\n#define IN2(i) row2[i]\n#define OUT0(i, x) row3[i] = (x)\n"
                      // volatile: otherwise the compiler forwards the stored value to the load and keeps (spills) it itself
                      "#define PARK_ST(t, i, x) *(volatile real *)(row##t + (i)) = (x)\n"
                      "#define PARK_LD(t, i) (*(volatile real *)(row##t + (i)))\n";
            else
                os << "    static __device__ __forceinline__ void run(const real *__restrict__ in0, const real "
                      "*__restrict__ in1,\n"
                      "        const real *__restrict__ in2, real *__restrict__ out0, real *__restrict__ out1, "
                      "real *__restrict__ out2,\n        const OutStage<real> &stage)\n    {\n"
                      "#define IN0(i) in0[i]\n#define IN1(i) in1[i]\n#define IN2(i) in2[i]\n#define OUT0(i, x) out0[i] = (x)\n"
                      "#define PARK_ST(t, i, x)\n#define PARK_LD(t, i) KC(0.0)\n";
            os << "#define KC(x) ((real)(x))\n#define KT(i) kc_table<real>(i)\n"
                  "#define OUT1(i, x) out1[i] = (x)\n#define OUT2(i, x) out2[i] = (x)\n"
                  "#define GRBDA_ALIGN() " << (std::getenv("GRBDA_ALIGN_CTA") ? "__syncthreads()" : "__syncwarp()") << "\n#define GRBDA_PIN(x, late) GRBDA_PIN_IMPL(x, late, stage.zero)\n"
                  "#define STGV4(k, m, base, a, b, c, d) if (stage.cls[k] == (m)) storeRow4(out##k + (base), a, b, c, d)\n"
                  "#define STGV1(k, m, base, a) if (stage.cls[k] == (m)) storeRow1(out##k + (base), a)\n"
                  "#define RING_PUT(k, e, x) ringPut<e>(stage.ring[k], x)\n"
                  "#define RING_HEAD(k) ringHead<real>(stage.ring[k], out##k)\n"
                  "#define RING_FLUSH(k, n) ringFlush<real, n>(stage.ring[k], out##k)\n"
                  "#define RING_TAIL(k) ringTail<real, N_OUT##k>(stage.ring[k], out##k)\n"
                  "#define STG_PUT(j, x) stage.lane[j] = (x)\n"
                  "#define STG_PUTK(k, j, x) stage.lane[(k) * stage.buf_stride + (j)] = (x)\n"
                  "#define STG_FLUSHI0(base, count) flushChunk<real, N_OUT0, count>(stage.g[0], base, stage.warp, stage.valid)\n"
                  "#define STG_FLUSHI1(base, count) flushChunk<real, N_OUT1, count>(stage.g[1], base, stage.warp + stage.buf_stride, stage.valid)\n"
                  "#define STG_FLUSHI2(base, count) flushChunk<real, N_OUT2, count>(stage.g[2], base, stage.warp + 2 * stage.buf_stride, stage.valid)\n"
                  "#define STG_FLUSH0(base, count) flushChunk<real, N_OUT0, count>(stage.g[0], base, stage.warp, stage.valid)\n"
                  "#define STG_FLUSH1(base, count) flushChunk<real, N_OUT1, count>(stage.g[1], base, stage.warp, stage.valid)\n"
                  "#define STG_FLUSH2(base, count) flushChunk<real, N_OUT2, count>(stage.g[2], base, stage.warp, stage.valid)\n";
            os << c.body;
            os << "#undef KC\n#undef KT\n#undef IN0\n#undef IN1\n#undef IN2\n#undef OUT0\n#undef OUT1\n#undef OUT2\n#undef GRBDA_ALIGN\n#undef GRBDA_PIN\n#undef PARK_ST\n#undef PARK_LD\n#undef STGV4\n#undef STGV1\n#undef RING_PUT\n#undef RING_HEAD\n#undef RING_FLUSH\n#undef RING_TAIL\n#undef STG_PUT\n#undef STG_PUTK\n#undef STG_FLUSHI0\n#undef STG_FLUSHI1\n#undef STG_FLUSHI2\n#undef STG_FLUSH0\n#undef STG_FLUSH1\n#undef STG_FLUSH2\n";
            os << "    }\n};\n";
        }


        // State generator of one model (kernels/stategen.cuh): one (phi, K_d) evaluator per implicit cluster and
        // `struct Gen` that fills one random valid state. Shared by tools/modelc.cpp and the run-time compiler.
        inline void emitGenerator(std::ostream &os, const ClusterTreeModel &model)
        {
            const int nq = model.getNumPositions(), nv = model.getNumDegreesOfFreedom();
            // one (phi, Kd) evaluator per implicit cluster
            for (const ClusterTreeNode &c : model.clusters())
            {
                if (c.joint_.type != ClusterType::Implicit)
                    continue;
                const ClusterDesc &d = c.joint_;
                sym::Graph graph;
                sym::GraphScope scope(graph);
                ModelCompiler mc(model);
                std::vector<sym::Sym> q(d.num_bodies), phi, K, Kd;
                for (int i = 0; i < d.num_bodies; i++)
                    q[i] = sym::Sym::input(0, i);
                mc.implicitJacobian(d, q, nullptr, phi, K, nullptr);
                std::vector<int> ind, dep;
                for (int i = 0; i < d.num_bodies; i++)
                    (d.independent[i] ? ind : dep).push_back(i);
                for (int i = 0; i < d.num_constraints; i++)
                    for (int j : dep)
                        Kd.push_back(K[i * d.num_bodies + j]);
                Program p;
                p.outputs = {phi, Kd};
                Emitter em(graph, p);
                os << "struct Cluster" << c.index_ << "\n{\n    static constexpr int N = " << d.num_bodies
                   << ", NC = " << d.num_constraints << ";\n";
                os << "    static __device__ __forceinline__ int ind(int i) { const int t[] = {";
                for (size_t i = 0; i < ind.size(); i++)
                    os << ind[i] << (i + 1 < ind.size() ? ", " : "");
                os << "}; return t[i]; }\n";
                os << "    static __device__ __forceinline__ int dep(int i) { const int t[] = {";
                for (size_t i = 0; i < dep.size(); i++)
                    os << dep[i] << (i + 1 < dep.size() ? ", " : "");
                os << "}; return t[i]; }\n";
                os << "    static __device__ __noinline__ void eval(const double *q, double *phi, double *Kd)\n    {\n"
                      "        typedef double real;\n        constexpr bool FAST = false;\n"
                      "#define KC(x) ((real)(x))\n#define GRBDA_PIN(x, late) (x)\n#define GRBDA_DIV(a, b) ((a) / (b))\n#define IN0(i) q[i]\n#define OUT0(i, x) phi[i] = (x)\n"
                      "#define OUT1(i, x) Kd[i] = (x)\n";
                os << em.cudaBody();
                os << "#undef KC\n#undef KT\n#undef GRBDA_PIN\n#undef GRBDA_DIV\n#undef IN0\n#undef OUT0\n#undef OUT1\n    }\n};\n\n";
            }
            os << "struct Gen\n{\n    static constexpr int NQ = " << nq << ", NV = " << nv << ";\n";
            os << "    static __device__ bool run(Philox &rng, double *q, double *yd, double *aux)\n    {\n"
                  "        bool ok = true;\n";
            for (const ClusterTreeNode &c : model.clusters())
            {
                const ClusterDesc &d = c.joint_;
                const int pi = c.position_index_;
                if (d.type == ClusterType::FreeQuaternion || d.type == ClusterType::FreeRollPitchYaw)
                {
                    os << "        for (int i = 0; i < 3; i++) q[" << pi << " + i] = rng.uniform();\n";
                    os << "        { double rpy[3]; for (int i = 0; i < 3; i++) rpy[i] = rng.uniform();\n";
                    if (d.type == ClusterType::FreeQuaternion)
                        os << "          rpyToQuat(rpy, q + " << pi + 3 << "); }\n";
                    else
                        os << "          for (int i = 0; i < 3; i++) q[" << pi + 3 << " + i] = rpy[i]; }\n";
                }
                else if (d.type == ClusterType::Explicit)
                    os << "        for (int i = 0; i < " << d.num_positions << "; i++) q[" << pi
                       << " + i] = rng.uniform();\n";
                else
                    os << "        ok = randomImplicitPosition<Cluster" << c.index_ << ">(rng, q + " << pi
                       << ") && ok;\n";
            }
            os << "        for (int i = 0; i < NV; i++) yd[i] = rng.uniform();\n"
                  "        for (int i = 0; i < NV; i++) aux[i] = rng.uniform();\n        return ok;\n    }\n};\n";
            // integration step: positions from the NEW velocities (semi-implicit Euler), cluster by cluster
            os << "struct Step\n{\n    static constexpr int NQ = " << nq << ", NV = " << nv << ";\n";
            os << "    static __device__ bool run(const double *q, const double *yd, double dt, double *qn)\n    {\n"
                  "        bool ok = true;\n";
            for (const ClusterTreeNode &c : model.clusters())
            {
                const ClusterDesc &d = c.joint_;
                const int pi = c.position_index_, vi = c.velocity_index_;
                if (d.type == ClusterType::FreeQuaternion)
                    os << "        integrateFreeQuaternion(q + " << pi << ", yd + " << vi << ", dt, qn + " << pi << ");\n";
                else if (d.type == ClusterType::FreeRollPitchYaw) // no reference counterpart (integrateQuat only): refused per state
                    os << "        for (int i = 0; i < 6; i++) qn[" << pi << " + i] = q[" << pi << " + i];\n        ok = false;\n";
                else if (d.type == ClusterType::Explicit)
                    os << "        for (int i = 0; i < " << d.num_positions << "; i++) qn[" << pi << " + i] = q[" << pi
                       << " + i] + dt * yd[" << vi << " + i];\n";
                else
                {
                    // independent spanning coordinates advance with their velocities, dependent ones start from
                    // their old values and are projected back onto phi = 0
                    os << "        for (int i = 0; i < " << d.num_bodies << "; i++) qn[" << pi << " + i] = q[" << pi << " + i];\n";
                    int k = 0;
                    for (int i = 0; i < d.num_bodies; i++)
                        if (d.independent[i])
                            os << "        qn[" << pi + i << "] += dt * yd[" << vi + k++ << "];\n";
                    os << "        ok = projectImplicitPosition<Cluster" << c.index_ << ">(qn + " << pi << ") && ok;\n";
                }
            }
            os << "        return ok;\n    }\n};\n";
        }

        // Binary tape: int32 header {magic, n_ops, n_arrays, n_in0, n_in1, n_in2}, then op,a,b,c,e
        // (int32 each, n_ops), val (float64 n_ops), then per output array: int32 count + indices.
        inline void writeTape(const CompiledAlgo &c, const std::string &path)
        {
            std::ofstream f(path, std::ios::binary);
            if (!f)
                throw std::runtime_error("cannot write " + path);
            const Tape &t = c.tape;
            const int32_t hdr[6] = {0x47524244, (int32_t)t.op.size(), (int32_t)t.outputs.size(), c.n_in[0],
                                    c.n_in[1], c.n_in[2]};
            f.write((const char *)hdr, sizeof(hdr));
            auto wi = [&](const std::vector<int32_t> &v) { f.write((const char *)v.data(), v.size() * 4); };
            wi(t.op), wi(t.a), wi(t.b), wi(t.c), wi(t.e);
            f.write((const char *)t.val.data(), t.val.size() * 8);
            for (auto &o : t.outputs)
            {
                const int32_t n = (int32_t)o.size();
                f.write((const char *)&n, 4);
                wi(o);
            }
        }

    } // namespace compiler
} // namespace grbda
