// Device-side model compiler: forward- and reverse-mode differentiation of an expression DAG (SURVEY 8 f4).
//
// The reference has no hand-written derivative algorithms: its "analytical derivatives" are CasADi's
// jacobian() of the symbolic inverse dynamics with respect to a tangent-space perturbation dq, the velocities
// and the third argument (reference: UnitTests/testRigidBodyDynamicsAlgosDerivatives.cpp:126-155, perturbation
// q (+) dq: UnitTests/testHelpers.hpp:50-112). The compiler already holds the same symbolic program, so the
// derivative programs are produced the same way: one tangent sweep per input direction over the DAG, through
// the Sym operators - constant folding and hash-consing remove every term whose tangent is structurally zero
// (a joint only moves its own subtree; a force only travels to its ancestors), which is the sparsity the
// published O(N d) derivative algorithms exploit by hand.
#pragma once
#include <unordered_map>
#include <vector>
#include "sym.h"

namespace grbda
{
    namespace compiler
    {
        // Tangents of `roots` along ONE direction. `seed`: tangent of input nodes (node id -> expression);
        // inputs that are not listed have tangent zero. Nodes created by the sweep are appended to the
        // current graph; only nodes that existed before the call are differentiated.
        inline std::vector<sym::Sym> tangentSweep(const std::vector<sym::Sym> &roots,
                                                  const std::unordered_map<int32_t, sym::Sym> &seed)
        {
            using sym::Sym;
            sym::Graph &g = Sym::G();
            const int32_t n0 = (int32_t)g.nodes.size();
            // nodes the roots depend on (ids are topologically ordered: operands precede their users)
            std::vector<char> live(n0, 0);
            for (const Sym &r : roots)
                live[r.id] = 1;
            for (int32_t i = n0 - 1; i >= 0; i--)
            {
                if (!live[i])
                    continue;
                const sym::Node n = g.nodes[i];
                if (n.op == sym::OP_CONST || n.op == sym::OP_INPUT)
                    continue;
                for (int32_t o : {n.a, n.b, n.c, n.e})
                    if (o >= 0)
                        live[o] = 1;
            }
            const int32_t zero = g.constant(0.0);
            std::vector<int32_t> tan(n0, zero);
            auto T = [&](int32_t id) { return Sym::fromId(tan[id]); };
            auto V = [&](int32_t id) { return Sym::fromId(id); };
            for (int32_t i = 0; i < n0; i++)
            {
                if (!live[i])
                    continue;
                const sym::Node n = g.nodes[i]; // copy: the vector grows below
                Sym t(0.0);
                switch (n.op)
                {
                case sym::OP_CONST:
                    break;
                case sym::OP_INPUT:
                {
                    auto it = seed.find(i);
                    if (it != seed.end())
                        t = it->second;
                    break;
                }
                case sym::OP_ADD:
                    t = T(n.a) + T(n.b);
                    break;
                case sym::OP_SUB:
                    t = T(n.a) - T(n.b);
                    break;
                case sym::OP_NEG:
                    t = -T(n.a);
                    break;
                case sym::OP_MUL:
                    t = T(n.a) * V(n.b) + V(n.a) * T(n.b);
                    break;
                case sym::OP_DIV: // x = a / b: dx = (da - x db) / b
                    if (!(T(n.a).isZero() && T(n.b).isZero()))
                        t = (T(n.a) - V(i) * T(n.b)) / V(n.b);
                    break;
                case sym::OP_SIN:
                    if (!T(n.a).isZero())
                        t = sym::cos(V(n.a)) * T(n.a);
                    break;
                case sym::OP_COS:
                    if (!T(n.a).isZero())
                        t = -(sym::sin(V(n.a)) * T(n.a));
                    break;
                case sym::OP_SQRT: // x = sqrt(a): dx = da / (2 x)
                    if (!T(n.a).isZero())
                        t = T(n.a) / (Sym(2.0) * V(i));
                    break;
                case sym::OP_SELECT_GT: // the condition is piecewise constant
                    t = sym::selectGt(V(n.a), V(n.b), T(n.c), T(n.e));
                    break;
                }
                tan[i] = t.id;
            }
            std::vector<Sym> out;
            out.reserve(roots.size());
            for (const Sym &r : roots)
                out.push_back(T(r.id));
            return out;
        }

        // Reverse mode: sum_k root_adjoints[k] * d roots[k] / d x for every input node x of `wrt`, one expression
        // per entry. The adjoints are expressions (a cotangent read from an input array, or an H^-1 solve), not
        // constants. Only nodes that are live (the roots depend on them) and active (they depend on a `wrt` input)
        // carry adjoints, so constant sub-graphs (inertias, gravity, joint-axis structure) get no adjoint code; the
        // contributions of a node used several times are summed with `+`, and constant folding / hash-consing drop
        // the structurally zero terms as in tangentSweep. Nodes created by the sweep are appended to the current
        // graph; only nodes that existed before the call are differentiated.
        inline std::vector<sym::Sym> adjointSweep(const std::vector<sym::Sym> &roots,
                                                  const std::vector<sym::Sym> &root_adjoints,
                                                  const std::vector<sym::Sym> &wrt)
        {
            using sym::Sym;
            if (roots.size() != root_adjoints.size())
                throw std::runtime_error("adjointSweep: one adjoint per root is required");
            sym::Graph &g = Sym::G();
            const int32_t n0 = (int32_t)g.nodes.size();
            std::vector<char> live(n0, 0), active(n0, 0);
            for (const Sym &r : roots)
                live[r.id] = 1;
            for (int32_t i = n0 - 1; i >= 0; i--)
            {
                if (!live[i])
                    continue;
                const sym::Node n = g.nodes[i];
                if (n.op == sym::OP_CONST || n.op == sym::OP_INPUT)
                    continue;
                for (int32_t o : {n.a, n.b, n.c, n.e})
                    if (o >= 0)
                        live[o] = 1;
            }
            for (const Sym &x : wrt)
                if (x.id < n0 && g.nodes[x.id].op == sym::OP_INPUT)
                    active[x.id] = 1;
            for (int32_t i = 0; i < n0; i++)
            {
                const sym::Node &n = g.nodes[i];
                if (!live[i] || n.op == sym::OP_CONST || n.op == sym::OP_INPUT)
                    continue;
                if (n.op == sym::OP_SELECT_GT) // the condition is piecewise constant
                    active[i] = active[n.c] || active[n.e];
                else
                    active[i] = active[n.a] || (n.b >= 0 && active[n.b]);
            }
            const int32_t zero = g.constant(0.0);
            std::vector<int32_t> adj(n0, zero);
            auto A = [&](int32_t id) { return Sym::fromId(adj[id]); };
            auto V = [&](int32_t id) { return Sym::fromId(id); };
            auto acc = [&](int32_t id, const Sym &x) {
                if (active[id])
                    adj[id] = (A(id) + x).id;
            };
            for (size_t k = 0; k < roots.size(); k++)
                acc(roots[k].id, root_adjoints[k]);
            for (int32_t i = n0 - 1; i >= 0; i--)
            {
                if (!live[i] || !active[i] || A(i).isZero())
                    continue;
                const sym::Node n = g.nodes[i]; // copy: the vector grows below
                const Sym a = A(i);
                switch (n.op)
                {
                case sym::OP_CONST:
                case sym::OP_INPUT:
                    break;
                case sym::OP_ADD:
                    acc(n.a, a);
                    acc(n.b, a);
                    break;
                case sym::OP_SUB:
                    acc(n.a, a);
                    acc(n.b, -a);
                    break;
                case sym::OP_NEG:
                    acc(n.a, -a);
                    break;
                case sym::OP_MUL:
                    if (active[n.a])
                        acc(n.a, a * V(n.b));
                    if (active[n.b])
                        acc(n.b, a * V(n.a));
                    break;
                case sym::OP_DIV: // x = a / b: da = adj / b, db = -(adj / b) x
                {
                    const Sym t = a / V(n.b);
                    acc(n.a, t);
                    if (active[n.b])
                        acc(n.b, -(t * V(i)));
                    break;
                }
                case sym::OP_SIN: // cos of the same argument: hash-conses with the primal sin/cos pair
                    acc(n.a, a * sym::cos(V(n.a)));
                    break;
                case sym::OP_COS:
                    acc(n.a, -(a * sym::sin(V(n.a))));
                    break;
                case sym::OP_SQRT: // x = sqrt(a): da = adj / (2 x)
                    acc(n.a, a / (Sym(2.0) * V(i)));
                    break;
                case sym::OP_SELECT_GT:
                    acc(n.c, sym::selectGt(V(n.a), V(n.b), a, Sym(0.0)));
                    acc(n.e, sym::selectGt(V(n.a), V(n.b), Sym(0.0), a));
                    break;
                }
            }
            std::vector<Sym> out;
            out.reserve(wrt.size());
            for (const Sym &x : wrt)
                out.push_back(x.id < n0 ? A(x.id) : Sym(0.0));
            return out;
        }

        // `roots` with some input nodes replaced by expressions (node id -> expression): the partial derivatives of
        // a program are taken with placeholder inputs held fixed, which are then given their values.
        inline std::vector<sym::Sym> substituteInputs(const std::vector<sym::Sym> &roots,
                                                      const std::unordered_map<int32_t, sym::Sym> &values)
        {
            using sym::Sym;
            sym::Graph &g = Sym::G();
            const int32_t n0 = (int32_t)g.nodes.size();
            std::vector<char> live(n0, 0);
            for (const Sym &r : roots)
                live[r.id] = 1;
            for (int32_t i = n0 - 1; i >= 0; i--)
            {
                if (!live[i])
                    continue;
                const sym::Node n = g.nodes[i];
                if (n.op == sym::OP_CONST || n.op == sym::OP_INPUT)
                    continue;
                for (int32_t o : {n.a, n.b, n.c, n.e})
                    if (o >= 0)
                        live[o] = 1;
            }
            std::vector<int32_t> sub(n0, -1);
            auto S = [&](int32_t id) { return Sym::fromId(sub[id]); };
            for (int32_t i = 0; i < n0; i++)
            {
                if (!live[i])
                    continue;
                const sym::Node n = g.nodes[i];
                Sym x = Sym::fromId(i);
                switch (n.op)
                {
                case sym::OP_CONST:
                    break;
                case sym::OP_INPUT:
                {
                    auto it = values.find(i);
                    if (it != values.end())
                        x = it->second;
                    break;
                }
                case sym::OP_ADD:
                    x = S(n.a) + S(n.b);
                    break;
                case sym::OP_SUB:
                    x = S(n.a) - S(n.b);
                    break;
                case sym::OP_NEG:
                    x = -S(n.a);
                    break;
                case sym::OP_MUL:
                    x = S(n.a) * S(n.b);
                    break;
                case sym::OP_DIV:
                    x = S(n.a) / S(n.b);
                    break;
                case sym::OP_SIN:
                    x = sym::sin(S(n.a));
                    break;
                case sym::OP_COS:
                    x = sym::cos(S(n.a));
                    break;
                case sym::OP_SQRT:
                    x = sym::sqrt(S(n.a));
                    break;
                case sym::OP_SELECT_GT:
                    x = sym::selectGt(S(n.a), S(n.b), S(n.c), S(n.e));
                    break;
                }
                sub[i] = x.id;
            }
            std::vector<Sym> out;
            out.reserve(roots.size());
            for (const Sym &r : roots)
                out.push_back(S(r.id));
            return out;
        }
    } // namespace compiler
} // namespace grbda
