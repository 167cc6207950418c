// StageCodegen: local system -> CUDA stage functions.
//
// What is generated (north_star subsystem 1).  The SQP local system
//   H = hess_w f, grad = grad_w f, J = dc/dw, l - c, u - c,   w = [p; x], c = [p; x; g]
// (SQPOptimizationSolver.cpp:58-71) is split by COLUMN GROUP: one group for the p columns
// and one per stage frame of x.  For a group with variables V the generator builds, with
// symbolic seeds s (one per variable of V), the forward-mode tangent program
//   T_r(s) = sum_{j in V} d g_r / d w_j * s_j      for every g row touching V
//   U_i(s) = sum_{j in V} d grad_i / d w_j * s_j   for every gradient entry touching V
// plus the primal values the group owns (its g rows, its gradient entries, its share of
// f).  On the device ONE WARP evaluates the program for one (instance, group): lane j runs
// it with s = e_j, so lane j ends up holding column j of the Jacobian / Hessian block --
// the same straight-line code on every lane, no divergence.  Lanes scatter their column
// into a shared-memory image of the group's CONTIGUOUS CSC value range and the warp then
// streams that range to HBM with coalesced 16-byte stores.  A group whose image exceeds a
// fixed budget (the p group at long horizons: its Hessian range holds one entry per stage
// and parameter) skips the image and stores straight into the instance's rows, so the
// kernel's static shared memory does not depend on the horizon.  Programs that are textually
// identical after making variable indices stage-relative are emitted once (all interior
// stages of an OCP share one template).
#include "optimal_control_problem/codegen/StageCodegen.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <filesystem>
#include <fstream>
#include <sstream>
#include <unordered_map>

#include <unistd.h>

#ifndef OCP_B200_INCLUDE_DIR_DEFAULT
#define OCP_B200_INCLUDE_DIR_DEFAULT "/root/repo/include"
#endif

namespace ocp_codegen {
using namespace casadi;

namespace {

std::string literal(double v) {
  if (std::isnan(v)) return "OCP_NAN";
  if (std::isinf(v)) return v > 0 ? "OCP_INF" : "(-OCP_INF)";
  char buf[64];
  std::snprintf(buf, sizeof(buf), "%.17g", v);
  std::string s(buf);
  if (s.find_first_of(".eEn") == std::string::npos) s += ".0";
  if (v < 0) s = "(" + s + ")";
  return s;
}

// Emits straight-line code for a set of roots; temporaries are numbered in DFS post-order
// from the roots so that isomorphic stage graphs give identical text.
struct Emitter {
  std::unordered_map<int, std::string> leaf;   // symbol node id -> C expression
  std::unordered_map<int, std::string> name;   // op node id -> temp name
  std::ostringstream body;
  int ntemp = 0;
  size_t nstmt = 0;

  std::string ref(const SXElem& e) {
    if (e.is_constant()) return literal(e.to_double());
    if (e.is_symbolic()) {
      auto it = leaf.find(e.id());
      casadi_assert(it != leaf.end(), "codegen: free symbol '" + e.name() + "'");
      return it->second;
    }
    auto it = name.find(e.id());
    casadi_assert(it != name.end(), "codegen: node was not emitted");
    return it->second;
  }

  void emit_node(const SXElem& e) {
    const int op = e.op();
    std::string a = ref(e.dep(0));
    std::string b = op_is_binary(op) ? ref(e.dep(1)) : "";
    std::string rhs;
    switch (op) {
      case OP_ADD: rhs = a + " + " + b; break;
      case OP_SUB: rhs = a + " - " + b; break;
      case OP_MUL: rhs = a + " * " + b; break;
      case OP_DIV: rhs = a + " / " + b; break;
      case OP_POW: rhs = "pow(" + a + ", " + b + ")"; break;
      case OP_ATAN2: rhs = "atan2(" + a + ", " + b + ")"; break;
      case OP_FMIN: rhs = "fmin(" + a + ", " + b + ")"; break;
      case OP_FMAX: rhs = "fmax(" + a + ", " + b + ")"; break;
      case OP_LT: rhs = "(" + a + " < " + b + " ? 1.0 : 0.0)"; break;
      case OP_NEG: rhs = "-" + a; break;
      case OP_SQ: rhs = a + " * " + a; break;
      case OP_SQRT: rhs = "sqrt(" + a + ")"; break;
      case OP_SIN: rhs = "sin(" + a + ")"; break;
      case OP_COS: rhs = "cos(" + a + ")"; break;
      case OP_TAN: rhs = "tan(" + a + ")"; break;
      case OP_ASIN: rhs = "asin(" + a + ")"; break;
      case OP_ACOS: rhs = "acos(" + a + ")"; break;
      case OP_ATAN: rhs = "atan(" + a + ")"; break;
      case OP_EXP: rhs = "exp(" + a + ")"; break;
      case OP_LOG: rhs = "log(" + a + ")"; break;
      case OP_FABS: rhs = "fabs(" + a + ")"; break;
      case OP_SIGN: rhs = "ocp_sign(" + a + ")"; break;
      case OP_TANH: rhs = "tanh(" + a + ")"; break;
      case OP_SINH: rhs = "sinh(" + a + ")"; break;
      case OP_COSH: rhs = "cosh(" + a + ")"; break;
      default: throw CasadiException("codegen: unsupported op");
    }
    std::string nm = "t" + std::to_string(ntemp++);
    body << "  const double " << nm << " = " << rhs << ";\n";
    name[e.id()] = nm;
    ++nstmt;
  }

  // make sure every op node under `root` has a temp
  void require(const SXElem& root) {
    if (root.is_constant() || root.is_symbolic() || name.count(root.id())) return;
    std::vector<std::pair<SXElem, int>> stack;  // node, next child
    stack.push_back({root, 0});
    while (!stack.empty()) {
      SXElem e = stack.back().first;
      int& next = stack.back().second;
      const int nchild = op_is_binary(e.op()) ? 2 : 1;
      if (next < nchild) {
        SXElem c = e.dep(next++);
        if (!c.is_constant() && !c.is_symbolic() && !name.count(c.id())) stack.push_back({c, 0});
      } else {
        if (!name.count(e.id())) emit_node(e);
        stack.pop_back();
      }
    }
  }
};

unsigned long long fnv1a(const std::string& s) {
  unsigned long long h = 1469598103934665603ULL;
  for (unsigned char c : s) { h ^= c; h *= 1099511628211ULL; }
  return h;
}

struct GroupPlan {
  int first_col = 0, ncols = 0, xoff = 0;  // xoff: offset of the X base pointer into x
  bool is_p = false;
  bool staged = true;   // image in shared memory + copy_out; false: lanes store straight to global memory
  int tmpl = -1, otmpl = -1;
  int a_base = 0, a_len = 0, h_base = 0, h_len = 0;
  int atab_off = 0, htab_off = 0, ctab_off = 0;
  int n_tg = 0, n_th = 0, n_cown = 0;
};

// Largest per-unit image (A range + H range of a group, doubles) that is staged in shared memory.  It holds every
// group of the three benchmark models at H = 20; a block's images then stay under 4 units x 2 x 640 doubles = 40 KB.
constexpr int kStageBudget = 640;
// c_groups (12 ints per group, 13 with the `staged` flag) lives in the 64 KB __constant__ bank
constexpr size_t kConstantBank = 64 * 1024;

void int_array(std::ostringstream& os, const char* decl, const std::vector<int>& v) {
  os << decl << "[" << std::max<size_t>(v.size(), 1) << "] = {";
  for (size_t i = 0; i < v.size(); ++i) {
    if (i % 24 == 0) os << "\n  ";
    os << v[i] << (i + 1 < v.size() ? "," : "");
  }
  if (v.empty()) os << "0";
  os << "};\n";
}

}  // namespace

std::string include_dir() {
  if (const char* e = std::getenv("OCP_B200_INCLUDE_DIR")) return e;
  return OCP_B200_INCLUDE_DIR_DEFAULT;
}

ModelSource generate(const ModelSpec& spec) {
  const int np = static_cast<int>(spec.p.numel());
  const int N = static_cast<int>(spec.x.numel());
  const int ng = static_cast<int>(spec.g.numel());
  const int n = np + N, m = n + ng;
  const int nf = spec.nf, H = spec.horizon;
  casadi_assert(nf > 0 && H > 0 && nf * H == N, "codegen: stage layout does not match x");
  casadi_assert(spec.grad.numel() == n && spec.grad.is_dense(), "codegen: gradient must be dense n-by-1");
  casadi_assert(spec.hess.size1() == n && spec.hess.size2() == n, "codegen: Hessian must be n-by-n");
  casadi_assert(spec.jac.size1() == m && spec.jac.size2() == n, "codegen: Jacobian must be m-by-n");
  casadi_assert(ng == 0 || spec.g.is_dense(), "codegen: constraints must be a dense column");

  std::vector<SXElem> w;
  w.insert(w.end(), spec.p.nonzeros().begin(), spec.p.nonzeros().end());
  w.insert(w.end(), spec.x.nonzeros().begin(), spec.x.nonzeros().end());
  std::vector<int> hc(spec.hess.sparsity().get_colind().begin(), spec.hess.sparsity().get_colind().end());
  std::vector<int> hr(spec.hess.sparsity().get_row().begin(), spec.hess.sparsity().get_row().end());
  std::vector<int> ac(spec.jac.sparsity().get_colind().begin(), spec.jac.sparsity().get_colind().end());
  std::vector<int> ar(spec.jac.sparsity().get_row().begin(), spec.jac.sparsity().get_row().end());
  for (int j = 0; j < n; ++j) {
    casadi_assert(ac[j + 1] > ac[j] && ar[ac[j]] == j, "codegen: J must start every column with its identity row");
    casadi_assert(ac[j + 1] - ac[j] == 1 || ar[ac[j] + 1] >= n, "codegen: unexpected entry in the identity block of J");
  }

  // ---- groups ---------------------------------------------------------------------------
  const int G = (np > 0 ? 1 : 0) + H;
  std::vector<GroupPlan> groups(G);
  std::vector<int> group_of(n);
  {
    int gi = 0;
    if (np > 0) {
      groups[gi].first_col = 0; groups[gi].ncols = np; groups[gi].xoff = 0; groups[gi].is_p = true;
      for (int j = 0; j < np; ++j) group_of[j] = gi;
      ++gi;
    }
    for (int k = 0; k < H; ++k, ++gi) {
      groups[gi].first_col = np + k * nf; groups[gi].ncols = nf; groups[gi].xoff = k * nf;
      for (int j = 0; j < nf; ++j) group_of[np + k * nf + j] = gi;
    }
  }
  for (GroupPlan& g : groups) {
    g.a_base = ac[g.first_col]; g.a_len = ac[g.first_col + g.ncols] - g.a_base;
    g.h_base = hc[g.first_col]; g.h_len = hc[g.first_col + g.ncols] - g.h_base;
    g.staged = g.a_len + g.h_len <= kStageBudget;
  }
  const bool any_direct = std::any_of(groups.begin(), groups.end(), [](const GroupPlan& g) { return !g.staged; });
  const size_t group_info_bytes = (any_direct ? 13 : 12) * sizeof(int);
  casadi_assert(G * group_info_bytes <= kConstantBank,
                "codegen: " + std::to_string(G) + " column groups (horizon " + std::to_string(H) +
                    ") overflow the 64 KB constant bank that holds the group table (" +
                    std::to_string(group_info_bytes) + " bytes per group, at most " +
                    std::to_string(kConstantBank / group_info_bytes) + " groups)");

  // ---- dependencies of g rows and gradient entries on w --------------------------------------
  std::vector<SXElem> roots;
  roots.insert(roots.end(), spec.g.nonzeros().begin(), spec.g.nonzeros().end());
  roots.insert(roots.end(), spec.grad.nonzeros().begin(), spec.grad.nonzeros().end());
  dag::DepSets deps = dag::dependency_sets(roots, w);
  // group -> rows of g / entries of grad that touch it; owner group of every g row
  std::vector<std::vector<int>> tg(G), th(G), cown(G);
  auto groups_touched = [&](const std::vector<int>& vars) {
    std::vector<int> gs;
    for (int j : vars) if (gs.empty() || gs.back() != group_of[j]) gs.push_back(group_of[j]);
    gs.erase(std::unique(gs.begin(), gs.end()), gs.end());
    return gs;
  };
  size_t nnz_a_expected = static_cast<size_t>(n), nnz_h_expected = 0;
  for (int r = 0; r < ng; ++r) {
    const std::vector<int>& d = deps.of_root(r);
    nnz_a_expected += d.size();
    std::vector<int> gs = groups_touched(d);
    for (int gidx : gs) tg[gidx].push_back(r);
    cown[gs.empty() ? 0 : gs.front()].push_back(r);
  }
  for (int i = 0; i < n; ++i) {
    const std::vector<int>& d = deps.of_root(ng + i);
    nnz_h_expected += d.size();
    for (int gidx : groups_touched(d)) th[gidx].push_back(i);
  }
  casadi_assert(nnz_a_expected == ar.size(), "codegen: Jacobian pattern disagrees with the dependency analysis");
  casadi_assert(nnz_h_expected == hr.size(), "codegen: Hessian pattern disagrees with the dependency analysis");

  // ---- objective terms: flatten the top-level sum and hand every term to a group -------
  std::vector<std::vector<SXElem>> fterms(G);
  {
    std::vector<SXElem> terms, stack;
    if (!spec.f.is_empty()) stack.push_back(spec.f.scalar());
    while (!stack.empty()) {
      SXElem e = stack.back(); stack.pop_back();
      if (e.op() == OP_ADD) { stack.push_back(e.dep(1)); stack.push_back(e.dep(0)); }
      else terms.push_back(e);
    }
    dag::DepSets fd = dag::dependency_sets(terms, w);
    for (size_t t = 0; t < terms.size(); ++t) {
      const std::vector<int>& d = fd.of_root(t);
      fterms[d.empty() ? 0 : group_of[d.front()]].push_back(terms[t]);
    }
  }

  // ---- per group: tangent program, tables, text; de-duplicate text ---------------------
  std::vector<int> tab;                       // all int tables, concatenated
  std::vector<std::string> tmpl_text, otmpl_text;
  std::vector<bool> tmpl_staged;
  std::unordered_map<std::string, int> tmpl_index, otmpl_index;
  size_t nstmt_total = 0;
  int stage_a = 1, stage_h = 1;

  auto leaf_names = [&](Emitter& em, const GroupPlan& g, const std::vector<SXElem>* seeds) {
    for (int i = 0; i < np; ++i) em.leaf[w[i].id()] = "P[" + std::to_string(i) + "]";
    for (int i = 0; i < N; ++i) em.leaf[w[np + i].id()] = "X[" + std::to_string(i - g.xoff) + "]";
    if (seeds)
      for (size_t j = 0; j < seeds->size(); ++j) em.leaf[(*seeds)[j].id()] = "S" + std::to_string(j);
  };

  // lanes per (instance, group) unit: a group has at most `maxcols` tangent directions, so a warp of 32 lanes
  // carries 32 / L units of the SAME group (consecutive instances: same template, no divergence).  The H = 20
  // quadrotor has 16-column groups: one unit per warp leaves half the lanes idle.
  int maxcols = 1;
  for (const GroupPlan& gp : groups) maxcols = std::max(maxcols, gp.ncols);
  int max_image = 1;   // doubles of the per-unit shared-memory image (largest A range + H range of a staged group)
  for (const GroupPlan& gp : groups)
    if (gp.staged) { stage_a = std::max(stage_a, gp.a_len); stage_h = std::max(stage_h, gp.h_len); }
  max_image = stage_a + stage_h;
  int L = 32;
  // (4 warps per block, static shared memory: keep the images of a block under 40 KB)
  while (L > 8 && L / 2 >= maxcols && size_t(4) * (32 / (L / 2)) * max_image * sizeof(double) <= 40 * 1024) L /= 2;
  if (const char* e = std::getenv("OCP_B200_ASSEMBLE_LANES")) {
    const int v = std::atoi(e);
    if (v == 8 || v == 16 || v == 32) L = std::max(v, L);   // only wider than needed (diagnostics)
  }

  for (int gidx = 0; gidx < G; ++gidx) {
    GroupPlan& g = groups[gidx];
    const int nd = g.ncols;
    std::vector<SXElem> V(w.begin() + g.first_col, w.begin() + g.first_col + nd), seeds;
    for (int j = 0; j < nd; ++j) seeds.push_back(SXElem::sym("seed" + std::to_string(j)));
    std::vector<SXElem> troots;
    for (int r : tg[gidx]) troots.push_back(spec.g.nonzeros()[r]);
    for (int i : th[gidx]) troots.push_back(spec.grad.nonzeros()[i]);
    std::vector<SXElem> tang = dag::forward(troots, V, seeds);
    g.n_tg = static_cast<int>(tg[gidx].size());
    g.n_th = static_cast<int>(th[gidx].size());
    g.n_cown = static_cast<int>(cown[gidx].size());

    // destination tables (relative to the group's value range; -1 = not in the pattern)
    g.atab_off = static_cast<int>(tab.size());
    for (int r : tg[gidx])
      for (int j = 0; j < nd; ++j) {
        const int col = g.first_col + j;
        auto b = ar.begin() + ac[col], e = ar.begin() + ac[col + 1];
        auto it = std::lower_bound(b, e, n + r);
        tab.push_back((it != e && *it == n + r) ? static_cast<int>(it - ar.begin()) - g.a_base : -1);
      }
    g.htab_off = static_cast<int>(tab.size());
    for (int i : th[gidx])
      for (int j = 0; j < nd; ++j) {
        const int col = g.first_col + j;
        auto b = hr.begin() + hc[col], e = hr.begin() + hc[col + 1];
        auto it = std::lower_bound(b, e, i);
        tab.push_back((it != e && *it == i) ? static_cast<int>(it - hr.begin()) - g.h_base : -1);
      }
    g.ctab_off = static_cast<int>(tab.size());
    for (int r : cown[gidx]) tab.push_back(n + r);

    // ---- assembly template text
    Emitter em;
    leaf_names(em, g, &seeds);
    std::ostringstream t;
    if (!g.staged) t << "  // sA / sH point into global memory (the group's image exceeds the shared-memory budget)\n";
    t << "  // tangent directions: " << nd << ", g-row tangents: " << g.n_tg << ", gradient tangents: "
      << g.n_th << ", owned g rows: " << g.n_cown << "\n";
    t << "  const bool act = dir < " << nd << ";\n  const int dsel = act ? dir : 0;\n";
    for (int j = 0; j < nd; ++j) t << "  const double S" << j << " = (dir == " << j << ") ? 1.0 : 0.0;\n";
    std::ostringstream stores;
    // primal values first (they do not depend on the seeds)
    std::vector<SXElem> cvals, qvals;
    for (int r : cown[gidx]) cvals.push_back(spec.g.nonzeros()[r]);
    for (int j = 0; j < nd; ++j) qvals.push_back(spec.grad.nonzeros()[g.first_col + j]);
    for (const SXElem& e : cvals) em.require(e);
    for (const SXElem& e : qvals) em.require(e);
    for (const SXElem& e : tang) em.require(e);
    // lane-select stores of the primal outputs: output i lives on lane i % L of the unit
    auto lane_select = [&](const std::vector<SXElem>& vals, const char* var, int chunk) {
      std::ostringstream s;
      s << "    double " << var << " = 0.0;\n";
      for (int i = chunk * L; i < std::min<int>(vals.size(), chunk * L + L); ++i)
        s << "    if (lane == " << (i % L) << ") " << var << " = " << em.ref(vals[i]) << ";\n";
      return s.str();
    };
    for (int c = 0; c * L < static_cast<int>(cvals.size()); ++c) {
      stores << "  {\n" << lane_select(cvals, "cv", c);
      stores << "    const int i = " << c * L << " + lane;\n";
      stores << "    if (first_pass && i < " << cvals.size() << ") { const int r = ctab[i]; "
             << "l[r] = lbg[r - NVAR] - cv; u[r] = ubg[r - NVAR] - cv; }\n  }\n";
    }
    for (int c = 0; c * L < static_cast<int>(qvals.size()); ++c) {
      stores << "  {\n" << lane_select(qvals, "qv", c);
      stores << "    const int i = " << c * L << " + lane;\n";
      stores << "    if (first_pass && i < " << qvals.size() << ") q[firstcol + i] = qv;\n  }\n";
    }
    for (int k = 0; k < g.n_tg; ++k)
      stores << "  { const int d = atab[" << k * nd << " + dsel]; if (act && d >= 0) sA[d] = " << em.ref(tang[k])
             << "; }\n";
    for (int k = 0; k < g.n_th; ++k)
      stores << "  { const int d = htab[" << k * nd << " + dsel]; if (act && d >= 0) sH[d] = "
             << em.ref(tang[g.n_tg + k]) << "; }\n";
    std::string text = t.str() + em.body.str() + stores.str();
    auto it = tmpl_index.find(text);
    if (it == tmpl_index.end()) {
      g.tmpl = static_cast<int>(tmpl_text.size());
      tmpl_index[text] = g.tmpl;
      tmpl_text.push_back(text);
      tmpl_staged.push_back(g.staged);
      nstmt_total += em.nstmt;
    } else {
      g.tmpl = it->second;
    }

    // ---- objective template text
    if (!fterms[gidx].empty()) {
      Emitter eo;
      leaf_names(eo, g, nullptr);
      for (const SXElem& e : fterms[gidx]) eo.require(e);
      std::ostringstream o;
      o << eo.body.str() << "  double acc = 0.0;\n";
      for (const SXElem& e : fterms[gidx]) o << "  acc += " << eo.ref(e) << ";\n";
      o << "  return acc;\n";
      auto jt = otmpl_index.find(o.str());
      if (jt == otmpl_index.end()) {
        g.otmpl = static_cast<int>(otmpl_text.size());
        otmpl_index[o.str()] = g.otmpl;
        otmpl_text.push_back(o.str());
        nstmt_total += eo.nstmt;
      } else {
        g.otmpl = jt->second;
      }
    }
  }

  // ---- translation unit -------------------------------------------------------------------
  std::ostringstream s;
  s << "// Generated by ocp_codegen (optimal_control_problem_b200) -- do not edit.\n";
  s << "// model: " << spec.name << "  np=" << np << " nf=" << nf << " horizon=" << H << " ng=" << ng
    << "  n=" << n << " m=" << m << " nnz(H)=" << hr.size() << " nnz(A)=" << ar.size() << "\n";
  s << "// groups: " << G << ", stage templates: " << tmpl_text.size() << ", objective templates: "
    << otmpl_text.size() << "\n";
  const int num_direct = static_cast<int>(std::count_if(groups.begin(), groups.end(), [](const GroupPlan& g) { return !g.staged; }));
  s << "// unit lanes: " << L << ", groups storing straight to global memory: " << num_direct
    << ", static shared memory of assemble_kernel: " << 4 * (32 / L) * (stage_a + stage_h) * sizeof(double) << " bytes\n";
  s << "#include <cuda_runtime.h>\n#include <math_constants.h>\n#include \"ocp_b200_model.h\"\n\n";
  s << "#define OCP_INF CUDART_INF\n#define OCP_NAN CUDART_NAN\n\nnamespace {\n";
  s << "constexpr int NP = " << np << ", NF = " << nf << ", HORIZON = " << H << ", NG = " << ng << ";\n";
  s << "constexpr int NX = " << N << ", NVAR = " << n << ", NCON = " << m << ";\n";
  s << "constexpr int NNZ_H = " << hr.size() << ", NNZ_A = " << ar.size() << ";\n";
  s << "constexpr int NUM_GROUPS = " << G << ", STAGE_A = " << stage_a << ", STAGE_H = " << stage_h << ";\n";
  // resident blocks per SM the assembly kernel is compiled for (register cap = 65536 / (128 * blocks))
  int min_blocks = 4;   // measured on B200 (quadrotor, B=4096): 1.20 ms at 2, 0.94 at 3, 0.89 at 4
  if (const char* e = std::getenv("OCP_B200_ASSEMBLE_MIN_BLOCKS")) min_blocks = std::max(1, std::atoi(e));
  s << "constexpr int WARPS_PER_BLOCK = 4, MIN_BLOCKS = " << min_blocks << ";\n";
  s << "constexpr int UNIT_LANES = " << L << ", UNITS_PER_WARP = 32 / UNIT_LANES;   // lanes per (instance, group) unit\n\n";
  s << "struct GroupInfo { int tmpl, otmpl, first_col, ncols, xoff, a_base, a_len, h_base, h_len, atab_off, "
       "htab_off, ctab_off" << (any_direct ? ", staged" : "") << "; };\n";
  s << "__constant__ GroupInfo c_groups[NUM_GROUPS] = {\n";
  for (const GroupPlan& g : groups)
    s << "  {" << g.tmpl << "," << g.otmpl << "," << g.first_col << "," << g.ncols << "," << g.xoff << ","
      << g.a_base << "," << g.a_len << "," << g.h_base << "," << g.h_len << "," << g.atab_off << ","
      << g.htab_off << "," << g.ctab_off << (any_direct ? (g.staged ? ",1" : ",0") : "") << "},\n";
  s << "};\n";
  int_array(s, "__device__ const int d_tab", tab);
  int_array(s, "__device__ const int d_acol", ac);
  int_array(s, "const int h_hcolptr", hc);
  int_array(s, "const int h_hrowidx", hr);
  int_array(s, "const int h_acolptr", ac);
  int_array(s, "const int h_arowidx", ar);
  s << R"(
__device__ __forceinline__ double ocp_sign(double a) { return a > 0.0 ? 1.0 : (a < 0.0 ? -1.0 : 0.0); }

// shared -> global copy of one contiguous value range, 16-byte stores where aligned
// (by the UNIT_LANES lanes of one unit; lane = lane within the unit)
__device__ __forceinline__ void copy_out(double* __restrict__ dst, const double* __restrict__ src, int len, int lane) {
  int head = ((reinterpret_cast<unsigned long long>(dst) & 15ULL) != 0ULL && len > 0) ? 1 : 0;
  if (head && lane == 0) dst[0] = src[0];
  const int pairs = (len - head) >> 1;
  double2* d2 = reinterpret_cast<double2*>(dst + head);
  for (int i = lane; i < pairs; i += UNIT_LANES) d2[i] = make_double2(src[head + 2 * i], src[head + 2 * i + 1]);
  if (((len - head) & 1) && lane == UNIT_LANES - 1) dst[len - 1] = src[len - 1];
}

)";
  for (size_t t = 0; t < tmpl_text.size(); ++t) {
    s << "__device__ __forceinline__ void stage_tmpl_" << t
      << "(const double* __restrict__ X, const double* __restrict__ P, const int dir, const int lane,\n"
         "    const int firstcol, const int* __restrict__ atab, const int* __restrict__ htab, const int* __restrict__ ctab,\n"
         "    double* __restrict__ sA, double* __restrict__ sH, const double* __restrict__ lbg, const double* __restrict__ ubg,\n"
         "    double* __restrict__ l, double* __restrict__ u, double* __restrict__ q, const bool first_pass) {\n"
      << tmpl_text[t] << "}\n\n";
  }
  for (size_t t = 0; t < otmpl_text.size(); ++t) {
    s << "__device__ __forceinline__ double obj_tmpl_" << t
      << "(const double* __restrict__ X, const double* __restrict__ P) {\n" << otmpl_text[t] << "}\n\n";
  }
  s << R"(
// one warp per column group and UNITS_PER_WARP consecutive instances (UNIT_LANES lanes each)
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, MIN_BLOCKS)
assemble_kernel(const int B, const double* __restrict__ x, const double* __restrict__ p,
                const double* __restrict__ frames, const double* __restrict__ lbx, const double* __restrict__ ubx,
                const double* __restrict__ lbg, const double* __restrict__ ubg, double* __restrict__ hv, const int ldh,
                double* __restrict__ q, const int ldn, double* __restrict__ av, const int lda,
                double* __restrict__ l, double* __restrict__ u, const int ldm) {
  __shared__ double smem[WARPS_PER_BLOCK * UNITS_PER_WARP * (STAGE_A + STAGE_H)];
  const int wlane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int lane = wlane % UNIT_LANES, unit = wlane / UNIT_LANES;   // lane within the unit
  const long long gw = static_cast<long long>(blockIdx.x) * WARPS_PER_BLOCK + wib;
  const long long ngroups_inst = (static_cast<long long>(B) + UNITS_PER_WARP - 1) / UNITS_PER_WARP;
  if (gw >= ngroups_inst * NUM_GROUPS) return;
  const int grp = static_cast<int>(gw % NUM_GROUPS);
  const int inst_raw = static_cast<int>(gw / NUM_GROUPS) * UNITS_PER_WARP + unit;
  const bool valid = inst_raw < B;            // (a ragged last warp: its idle units run the code, store nothing)
  const int inst = valid ? inst_raw : B - 1;
  const GroupInfo gi = c_groups[grp];
  double* sA = smem + (wib * UNITS_PER_WARP + unit) * (STAGE_A + STAGE_H);
  double* sH = sA + STAGE_A;
  const double* xi = x + static_cast<size_t>(inst) * NX;
  const double* pi = p + static_cast<size_t>(inst) * NP;
  double* li = l + static_cast<size_t>(inst) * ldm;
  double* ui = u + static_cast<size_t>(inst) * ldm;
  double* qi = q + static_cast<size_t>(inst) * ldn;
)";
  if (any_direct)
    s << R"(  double* gA = av + static_cast<size_t>(inst) * lda + gi.a_base;   // groups that skip the shared-memory image
  double* gH = hv + static_cast<size_t>(inst) * ldh + gi.h_base;
)";
  s << R"(  // identity rows of c = [p; x; g]: A entry 1, bounds l - w, u - w (first frame pinned to `frames`)
  for (int j = lane; valid && j < gi.ncols; j += UNIT_LANES) {
    const int col = gi.first_col + j;
)" << (any_direct ? "    if (gi.staged) sA[d_acol[col] - gi.a_base] = 1.0;\n    else gA[d_acol[col] - gi.a_base] = 1.0;\n"
                  : "    sA[d_acol[col] - gi.a_base] = 1.0;\n")
    << R"(    double c, lo, hi;
    if (col < NP) {
      c = pi[col]; lo = c; hi = c;
    } else {
      const int k = col - NP;
      c = xi[k];
      if (frames != nullptr && k < NF) { lo = frames[static_cast<size_t>(inst) * NF + k]; hi = lo; }
      else { lo = lbx[k]; hi = ubx[k]; }
    }
    li[col] = lo - c;
    ui[col] = hi - c;
  }
  const int npass = (gi.ncols + UNIT_LANES - 1) / UNIT_LANES;
  for (int pass = 0; pass < npass; ++pass) {
    const int dir = valid ? pass * UNIT_LANES + lane : (1 << 20);   // no direction: no tangent stores
    switch (gi.tmpl) {
)";
  for (size_t t = 0; t < tmpl_text.size(); ++t)
    s << "      case " << t << ": stage_tmpl_" << t
      << "(xi + gi.xoff, pi, dir, lane, gi.first_col, d_tab + gi.atab_off, d_tab + gi.htab_off, d_tab + gi.ctab_off, "
      << (tmpl_staged[t] ? "sA, sH" : "gA, gH") << ", lbg, ubg, li, ui, qi, valid && pass == 0); break;\n";
  s << R"(      default: break;
    }
  }
  __syncwarp();
  if ()" << (any_direct ? "valid && gi.staged" : "valid") << R"() {
    copy_out(av + static_cast<size_t>(inst) * lda + gi.a_base, sA, gi.a_len, lane);
    copy_out(hv + static_cast<size_t>(inst) * ldh + gi.h_base, sH, gi.h_len, lane);
  }
}

// one warp per instance; lane g sums the objective terms of groups g, g+32, ...
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
objective_kernel(const int B, const double* __restrict__ x, const double* __restrict__ p, double* __restrict__ f) {
  const int lane = threadIdx.x & 31;
  const long long inst = static_cast<long long>(blockIdx.x) * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  if (inst >= B) return;
  const double* xi = x + static_cast<size_t>(inst) * NX;
  const double* pi = p + static_cast<size_t>(inst) * NP;
  double acc = 0.0;
  for (int grp = lane; grp < NUM_GROUPS; grp += 32) {
    const GroupInfo gi = c_groups[grp];
    switch (gi.otmpl) {
)";
  for (size_t t = 0; t < otmpl_text.size(); ++t)
    s << "      case " << t << ": acc += obj_tmpl_" << t << "(xi + gi.xoff, pi); break;\n";
  s << R"(      default: break;
    }
  }
  double total = 0.0;
  for (int src = 0; src < 32; ++src) total += __shfl_sync(0xffffffffu, acc, src);  // fixed order
  if (lane == 0) f[inst] = total;
}
}  // namespace

extern "C" const ocp_b200_model_info* ocp_b200_model_get_info(void) {
  static const ocp_b200_model_info info = {
      OCP_B200_MODEL_ABI_VERSION, NP, NF, HORIZON, NG, NVAR, NCON, NNZ_H, NNZ_A,
      h_hcolptr, h_hrowidx, h_acolptr, h_arowidx, NUM_GROUPS, NUM_TEMPLATES, MODEL_NAME, MODEL_HASH};
  return &info;
}

extern "C" int ocp_b200_model_assemble(int B, const double* x, const double* p, const double* frames,
                                       const double* lbx, const double* ubx, const double* lbg, const double* ubg,
                                       double* h_vals, int ld_h, double* q, int ld_n, double* a_vals, int ld_a,
                                       double* l, double* u, int ld_m, void* stream) {
  if (B <= 0) return 0;
  const long long warps = ((static_cast<long long>(B) + UNITS_PER_WARP - 1) / UNITS_PER_WARP) * NUM_GROUPS;
  const unsigned blocks = static_cast<unsigned>((warps + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK);
  assemble_kernel<<<blocks, WARPS_PER_BLOCK * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      B, x, p, frames, lbx, ubx, lbg, ubg, h_vals, ld_h, q, ld_n, a_vals, ld_a, l, u, ld_m);
  return static_cast<int>(cudaGetLastError());
}

extern "C" int ocp_b200_model_objective(int B, const double* x, const double* p, double* f, void* stream) {
  if (B <= 0) return 0;
  const unsigned blocks = static_cast<unsigned>((B + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK);
  objective_kernel<<<blocks, WARPS_PER_BLOCK * 32, 0, static_cast<cudaStream_t>(stream)>>>(B, x, p, f);
  return static_cast<int>(cudaGetLastError());
}
)";
  std::string body = s.str();
  ModelSource out;
  out.num_groups = G;
  out.num_templates = static_cast<int>(tmpl_text.size());
  out.num_statements = nstmt_total;
  out.hash = fnv1a(body);
  char hx[32];
  std::snprintf(hx, sizeof(hx), "0x%016llxULL", out.hash);
  std::string defs = "#define NUM_TEMPLATES " + std::to_string(tmpl_text.size()) + "\n#define MODEL_NAME \"" +
                     spec.name + "\"\n#define MODEL_HASH " + hx + "\n";
  out.source = defs + body;
  return out;
}

namespace {
// single-quoted for /bin/sh: the only character that needs care inside '...' is the quote itself
std::string sh_quote(const std::string& v) {
  std::string out = "'";
  for (char c : v) {
    if (c == '\'') out += "'\\''";
    else out += c;
  }
  return out + "'";
}
}  // namespace

// Several processes may build the same model at once (one rank per GPU, each calling genSolver() on a cold
// cache): every file a build writes carries the pid until it is complete and is then renamed into place, so no
// process ever reads a half-written source and nvcc never reads a file another rank is rewriting.  The model name
// becomes part of a file name and of a shell command line: it is restricted to [A-Za-z0-9_], paths are quoted.
std::string compile(const ModelSource& src, const std::string& name, const std::string& code_dir, bool verbose) {
  namespace fs = std::filesystem;
  if (name.empty() || name.size() > 64 ||
      name.find_first_not_of("ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789_") != std::string::npos)
    throw std::invalid_argument("codegen: problem name '" + name + "' must match [A-Za-z0-9_]{1,64}");
  fs::create_directories(code_dir);
  char hx[32];
  std::snprintf(hx, sizeof(hx), "%016llx", src.hash);
  const std::string stem = (fs::path(code_dir) / (name + "_" + hx)).string();
  const std::string cu = stem + ".cu", so = stem + ".so";
  if (fs::exists(so)) {
    if (verbose) std::cout << "stage library cached: " << so << std::endl;
    return so;
  }
  const std::string pid = std::to_string(static_cast<long>(::getpid()));
  const std::string cu_tmp = stem + ".tmp." + pid + ".cu", so_tmp = so + ".tmp." + pid;
  {
    std::ofstream f(cu_tmp);
    if (!f.good()) throw std::runtime_error("codegen: cannot write " + cu_tmp);
    f << src.source;
    f.close();
    if (!f.good()) throw std::runtime_error("codegen: short write to " + cu_tmp);
  }
  const char* nvcc_env = std::getenv("OCP_B200_NVCC");
  const std::string nvcc = nvcc_env ? nvcc_env : "nvcc";
  const char* extra_env = std::getenv("OCP_B200_NVCC_FLAGS");   // trusted: extra compiler flags, split by the shell
  const std::string extra = extra_env ? std::string(" ") + extra_env : std::string();
  const std::string cmd = sh_quote(nvcc) + " -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -shared "
                          "-Xcompiler -fPIC" + extra + " -I" + sh_quote(include_dir()) + " -o " + sh_quote(so_tmp) + " " +
                          sh_quote(cu_tmp) + " 2>&1";
  if (verbose) std::cout << "compiling stage library: " << cmd << std::endl;
  FILE* pipe = popen(cmd.c_str(), "r");
  if (!pipe) { std::error_code ec; fs::remove(cu_tmp, ec); throw std::runtime_error("codegen: cannot start nvcc"); }
  std::string log;
  char buf[512];
  while (fgets(buf, sizeof(buf), pipe)) log += buf;
  const int rc = pclose(pipe);
  std::error_code ec;
  if (rc != 0 || !fs::exists(so_tmp)) {
    fs::rename(cu_tmp, stem + ".failed.cu", ec);   // kept for inspection
    fs::remove(so_tmp, ec);
    throw std::runtime_error("codegen: nvcc failed for " + stem + ".failed.cu (exit " + std::to_string(rc) + ")\n" + log);
  }
  fs::rename(cu_tmp, cu, ec);      // the source next to the library (same content from every rank)
  fs::rename(so_tmp, so);          // atomic: a concurrent reader sees the old state or the complete file
  return so;
}

}  // namespace ocp_codegen
