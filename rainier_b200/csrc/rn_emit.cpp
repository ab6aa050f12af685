// rn_emit.cpp -- see rn_emit.hpp.
#include "rn_emit.hpp"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <set>
#include <sstream>

namespace rn {

extern const char* kPreludeSource;  // rn_prelude.cuh, embedded at build time
extern const char* kSamplerSource;     // rn_args.h + rn_sampler.cuh
extern const char* kSamplerWpcSource;  // rn_args.h + rn_sampler_wpc.cuh
extern const char* kFunctionSource;    // rn_function.cuh
extern const char* kOptimizerSource;   // rn_args.h + rn_optimizer.cuh

namespace {

std::string lit(double v) {
  if (std::isnan(v)) return "RN_NAN";
  if (std::isinf(v)) return v > 0 ? "RN_INF" : "(-RN_INF)";
  char buf[64];
  std::snprintf(buf, sizeof(buf), "%a", v);  // exact hex-float literal
  std::string s(buf);
  if (v < 0 || (v == 0 && std::signbit(v))) return "(" + s + ")";
  return s;
}

struct Emitter {
  const Program& P;
  const EmitOptions& opt;
  std::ostringstream os;
  bool wpc = false;
  std::vector<int> smem_slot;             // slot -> index in the shared accumulator block, or -1 (register)
  std::map<int, int> tab_off;             // large-lookup node id -> offset of its table in scratch
  std::vector<int> tab_fill;              // one representative lookup node per distinct table
  int red_off = 0, red_doubles = 0;       // cross-warp reduction scratch (K warps per chain)
  int n_smem_acc = 0, tab_doubles = 0;
  std::string col_suffix;                 // names of column values loaded in the current region of a row body
  std::string node_suffix;                // appended to the names of row-body values (the DMMA path emits one body per element)
  Emitter(const Program& p, const EmitOptions& o) : P(p), opt(o) {}

  // The body of one row of a streamed target.  Keeps live ranges short, because a "row" of the reference's
  // Model.observe is 8 unrolled observations over hundreds of columns (core/Model.scala:98-132):
  //   * a column value is loaded right before its first use (not hoisted to the top of the row),
  //   * the reverse sweep re-loads the columns it needs behind a compiler fence instead of keeping the forward
  //     sweep's copies alive (2 loads per element per row; the data sits in L1/L2/shared memory),
  //   * every accumulation / scatter is issued as soon as its operand exists (a_j += w * x_j contracts to one FMA in
  //     fast mode).  The order of the additions into any one slot is unchanged.
  int local_col(const TargetInfo& T, int k) const { return k - ((int)T.first_input - (int)P.n_params); }

  void operands(int id, std::vector<int>& out) const {
    const Node& n = P.nodes[id];
    out.clear();
    switch (n.kind) {
      case K_UNARY: out.push_back(n.a); break;
      case K_BINARY: out.push_back(n.a); out.push_back(n.b); break;
      case K_LOOKUP:
        out.push_back(n.a);
        for (int k = 0; k < n.c; k++) out.push_back(P.lookup_refs[n.b + k]);
        break;
      case K_SELEQ: out.push_back(n.a); out.push_back(n.b); out.push_back(n.c); break;
      default: break;
    }
  }

  // see row_body(): splits the row statements into independent dataflow components and merges them round-robin
  void interleave_components(const TargetInfo& T, const std::set<int>& body, std::vector<int>& order_fwd,
                             std::vector<int>& order_bwd) const {
    const int BIG = 4;  // two components of at least this many statements meeting in one statement = a joiner
    std::map<int, int> parent, size;  // union-find over statement ids
    std::set<int> tail;
    std::function<int(int)> find = [&](int x) {
      while (parent[x] != x) {
        parent[x] = parent[parent[x]];
        x = parent[x];
      }
      return x;
    };
    std::vector<int> ops;
    auto classify = [&](int s) {
      operands(s, ops);
      bool is_tail = false;
      std::set<int> comps;
      for (int o : ops) {
        if (!body.count(o)) continue;
        if (tail.count(o)) {
          is_tail = true;
          break;
        }
        comps.insert(find(o));
      }
      if (!is_tail && comps.size() >= 2) {
        int big = 0;
        for (int c : comps)
          if (size[c] >= BIG) big++;
        if (big >= 2) is_tail = true;
      }
      if (is_tail) {
        tail.insert(s);
        return;
      }
      parent[s] = s;
      size[s] = 1;
      for (int c : comps) {
        const int r = find(s), q = find(c);
        if (r == q) continue;
        parent[q] = r;
        size[r] += size[q];
      }
    };
    std::vector<int> fwd, bwd;
    for (int id : T.row_fwd)
      if (body.count(id)) {
        classify(id);
        fwd.push_back(id);
      }
    for (int id : T.row_bwd)
      if (body.count(id)) {
        classify(id);
        bwd.push_back(id);
      }
    auto schedule = [&](const std::vector<int>& region, std::vector<int>& out) {
      std::vector<int> comp_order;
      std::map<int, std::vector<int>> lists;
      std::vector<int> tails;
      for (int id : region) {
        if (tail.count(id)) {
          tails.push_back(id);
          continue;
        }
        const int c = find(id);
        if (!lists.count(c)) comp_order.push_back(c);
        lists[c].push_back(id);
      }
      // round-robin over at most `interleave` components at a time: every component in flight keeps its temporaries in
      // registers (8 observations of a Poisson row x ~16 registers did not fit the 128 of a 16-warp CTA: 1.4e9 spill
      // accesses and 244 GB of DRAM traffic per launch, profiles/r2_ncu_cfg5_v1.csv)
      const size_t W = (size_t)std::max(1, opt.interleave);
      std::vector<size_t> pos(comp_order.size(), 0);
      for (size_t g0 = 0; g0 < comp_order.size(); g0 += W)
        for (bool any = true; any;) {
          any = false;
          for (size_t k = g0; k < std::min(comp_order.size(), g0 + W); k++) {
            const std::vector<int>& l = lists[comp_order[k]];
            if (pos[k] < l.size()) {
              out.push_back(l[pos[k]++]);
              any = true;
            }
          }
        }
      out.insert(out.end(), tails.begin(), tails.end());
    };
    schedule(fwd, order_fwd);
    schedule(bwd, order_bwd);
  }

  template <class Load, class AccRef>
  void row_body(const TargetInfo& T, const char* ind, Load load, AccRef accref, bool atomic_scatter, int scatter_base_off) {
    std::set<int> body;
    for (int id : T.row_fwd)
      if (P.nodes[id].kind != K_CONST && P.nodes[id].kind != K_INPUT) body.insert(id);
    for (int id : T.row_bwd)
      if (P.nodes[id].kind != K_CONST && P.nodes[id].kind != K_INPUT) body.insert(id);
    std::map<int, std::vector<const AccStmt*>> acc_at;
    std::map<int, std::vector<const ScatterStmt*>> sc_at;
    std::vector<const AccStmt*> acc_tail;
    std::vector<const ScatterStmt*> sc_tail;
    for (const AccStmt& a : T.row_acc) (body.count(a.node) ? acc_at[a.node] : acc_tail).push_back(&a);
    for (const ScatterStmt& sc : T.row_scatter) (body.count(sc.node) ? sc_at[sc.node] : sc_tail).push_back(&sc);
    std::set<int> declared;
    auto need_col = [&](int o) {
      const Node& n = P.nodes[o];
      if (n.kind != K_INPUT || (uint32_t)n.a < P.n_params) return;
      const int k = n.a - (int)P.n_params;
      if (declared.insert(k).second) os << ind << "const double c" << k << col_suffix << " = " << load(k) << ";\n";
    };
    auto need_operands = [&](int id) {
      const Node& n = P.nodes[id];
      switch (n.kind) {
        case K_UNARY: need_col(n.a); break;
        case K_BINARY: need_col(n.a); need_col(n.b); break;
        case K_LOOKUP:
          need_col(n.a);
          for (int k = 0; k < n.c; k++) need_col(P.lookup_refs[n.b + k]);
          break;
        case K_SELEQ: need_col(n.a); need_col(n.b); need_col(n.c); break;
        default: break;
      }
    };
    auto emit_acc = [&](const AccStmt& a) { os << ind << accref(a.slot) << " += " << val(a.node) << ";\n"; };
    auto emit_scatter = [&](const ScatterStmt& sc) {
      if (atomic_scatter) {
        // branch-free (an index outside the table raises the flag and adds 0 to entry 0) and in the shared state space: the
        // generic atomicAdd carries one code path per address space behind a run-time test, 16 times per row body on cfg 5.
        // The index is converted again rather than kept from the forward Lookup: reusing it lost 3 % on cfg 5 (2.455e5 -> 2.374e5,
        // profiles/r2_bench_row_libm_ab_v2.txt) -- eight more values live across the reverse sweep's fence at 128 registers
        os << ind << "{ const int k = rn_d2i(" << val(sc.index_node) << ") - (" << sc.low << "); const bool bad = (unsigned)k >= " << sc.len
           << "u; err |= (int)bad; rn_scatter_add(&scr[" << (scatter_base_off + smem_slot[sc.slot_base]) << " + (bad ? 0 : k)], bad ? 0.0 : "
           << val(sc.node) << "); }\n";
        return;
      }
      os << ind << "{ const int k = rn_d2i(" << val(sc.index_node) << ") - (" << sc.low << "); if (k < 0 || k >= " << sc.len
         << ") err |= 1; else ";
      os << "acc[" << sc.slot_base << " + k] += " << val(sc.node) << "; }\n";
    };
    auto one = [&](int id) {
      if (!body.count(id)) return;
      need_operands(id);
      stmt(id, ind);
      auto ia = acc_at.find(id);
      if (ia != acc_at.end())
        for (const AccStmt* a : ia->second) emit_acc(*a);
      auto is = sc_at.find(id);
      if (is != sc_at.end())
        for (const ScatterStmt* sc : is->second) {
          need_col(sc->index_node);
          emit_scatter(*sc);
        }
    };
    // Instruction-level parallelism: the unrolled observations of a row are independent dataflow components whose
    // results only meet in a final sum.  Emitting them one after the other leaves each warp with a single serial
    // dependency chain (a 50-term dot product is 50 dependent FMAs; ncu: stall_wait dominates at 8 warps/SM), so the
    // statements of the components are interleaved round-robin; "joiner" statements (and everything downstream of
    // them) follow in their original order.  Values are unchanged (SSA); only the issue order moves.  The reverse sweep
    // follows the forward sweep of the whole row: issuing a group's reverse statements right after its forward statements
    // (no second read of the tile) measured cfg 5 -10 %, cfg 2s and rows-across-lanes cfg 3 +1 % (profiles/r2_bench_fused_sweeps_ab_v1.txt).
    std::vector<int> order_fwd, order_bwd;
    interleave_components(T, body, order_fwd, order_bwd);
    col_suffix.clear();
    for (int id : order_fwd) one(id);
    if (!order_bwd.empty()) {
      os << ind << "RN_FENCE();\n";
      declared.clear();
      col_suffix = "b";
      for (int id : order_bwd) one(id);
    }
    for (const AccStmt* a : acc_tail) {
      need_col(a->node);
      emit_acc(*a);
    }
    for (const ScatterStmt* sc : sc_tail) {
      need_col(sc->index_node);
      need_col(sc->node);
      emit_scatter(*sc);
    }
    col_suffix.clear();
  }

  std::string acc_ref(int slot) const {
    if (!wpc) return "acc[" + std::to_string(slot) + "]";
    if (smem_slot[slot] >= 0) return "scr[" + std::to_string(tab_doubles + smem_slot[slot]) + "]";
    return "a" + std::to_string(slot);
  }
  bool is_big_table(const Node& n) const {
    if (n.kind != K_LOOKUP || n.c <= 8) return false;
    for (int k = 0; k < n.c; k++)
      if (P.nodes[P.lookup_refs[n.b + k]].region != R_INV_FWD && P.nodes[P.lookup_refs[n.b + k]].region != R_INV_BWD) return false;
    return true;
  }

  std::string val(int id) const {
    if (!name_override.empty()) {
      auto it = name_override.find(id);
      if (it != name_override.end()) return it->second;
    }
    const Node& n = P.nodes[id];
    if (n.kind == K_CONST) return lit(n.value);
    if (n.kind == K_INPUT) {
      if ((uint32_t)n.a < P.n_params) return "q[" + std::to_string(n.a) + "]";
      return "c" + std::to_string(n.a - (int)P.n_params) + col_suffix;
    }
    if (!node_suffix.empty() && (n.region == R_ROW_FWD || n.region == R_ROW_BWD)) return "v" + std::to_string(id) + node_suffix;
    return "v" + std::to_string(id);
  }

  // `derived`: the node was created by the emitter's own reverse sweep (there is no reference operation to mirror), so
  // constant powers are strength-reduced in parity mode as well -- d/dx x^-1 = -x^-2 would otherwise cost one fdlibm
  // pow() per observation of a logistic regression
  // Row bodies of the warp-per-chain shape: total, branch-free exp / log / reciprocal (rn_prelude.cuh: rn_row_*) instead of CUDA's
  // exp(), log() and 1.0 / x, each of which ends a basic block with its range test -- and the statements of 4 or 8 observations
  // are interleaved precisely so that ptxas can overlap their chains.
  // Measured on B200 (profiles/r2_bench_row_libm_ab_v1.txt, ..._v2.txt): the rows-across-lanes body gains -- cfg 5: 2.22e5 -> 2.46e5
  // with two observations in flight where the arguments of exp are wild (every proposal rejected far from the mode: CUDA's exp
  // takes its out-of-line completion there), 2.41e5 -> 2.46e5 after an adaptive warmup --, the chain-batched DMMA kernel loses (cfg 3: 5.25e5 -> 4.66e5; at 128 registers the four elements
  // of its helper in one basic block spill: stack 976 -> 4776 bytes) -- so they are used in kernels without the DMMA path
  // and not in those with it (helper and its rows-across-lanes tail alike: that kernel stays exactly what round 2 validated).
  // ... and neither in row bodies that keep many accumulators in registers: the rows-across-lanes form of cfg 3 (RN_MMA=0: 51
  // accumulators) runs 5.4e4 with the row functions against 2.1e5 with CUDA's libm, the merged block spills.  So they are used
  // only where the registers have room: no DMMA path and at most 8 register accumulators (cfg 5: 2).  Set by density_wpc().
  bool row_functions = false;
  bool in_mma_helper = false;
  std::string recip(const std::string& x, bool row_variant) const {
    return (row_variant && row_functions) ? "rn_row_rcp(" + x + ")" : "(1.0 / " + x + ")";
  }
  std::string pow_expr(int a, int b, bool derived, bool row_variant = false) const {
    const Node& e = P.nodes[b];
    const std::string x = val(a);
    if (e.kind == K_CONST) {
      const double c = e.value;
      if (c == 1.0) return x;
      if (c == 2.0) return "(" + x + " * " + x + ")";
      if (c == -1.0) return recip(x, row_variant);
      if (derived && !opt.fast_math) {
        if (c == 3.0) return "(" + x + " * " + x + " * " + x + ")";
        if (c == 4.0) return "((" + x + " * " + x + ") * (" + x + " * " + x + "))";
        if (c == -2.0) return recip("(" + x + " * " + x + ")", row_variant);
        if (c == -3.0) return recip("(" + x + " * " + x + " * " + x + ")", row_variant);
        if (c == 0.5) return "sqrt(" + x + ")";
        if (c == -0.5) return recip("sqrt(" + x + ")", row_variant);
        if (c == 1.5) return "(" + x + " * sqrt(" + x + "))";
        if (c == -1.5) return recip("(" + x + " * sqrt(" + x + "))", row_variant);
      }
      if (opt.fast_math) {
        if (c == 3.0) return "(" + x + " * " + x + " * " + x + ")";
        if (c == 4.0) return "((" + x + " * " + x + ") * (" + x + " * " + x + "))";
        if (c == -2.0) return recip("(" + x + " * " + x + ")", row_variant);
        if (c == 0.5) return "sqrt(" + x + ")";
        if (c == -0.5) return "rsqrt(" + x + ")";
        if (c == 1.5) return "(" + x + " * sqrt(" + x + "))";
      }
    }
    return std::string(row_variant ? "rn_pow_libm(" : "rn_pow(") + x + ", " + val(b) + ")";
  }
  bool row_libm(const Node& n) const { return wpc && (n.region == R_ROW_FWD || n.region == R_ROW_BWD); }

  void stmt(int id, const char* indent) {
    const Node& n = P.nodes[id];
    if (n.kind == K_CONST || n.kind == K_INPUT) return;
    os << indent << "const double " << val(id) << " = ";
    switch (n.kind) {
      case K_UNARY: {
        const std::string x = val(n.a);
        switch (n.op) {
          // Row-variant transcendentals of the warp-per-chain shape use CUDA's libm (<= 1 ulp, like the JVM's own
          // Math.exp/log intrinsics): rows are summed in tree order there, so those results are not bit-comparable with
          // the oracle anyway (1e-13 agreement), and fdlibm costs twice the instructions.  Everything that stays
          // bit-exact -- invariant parts, data-free targets, the thread-per-chain kernels -- keeps fdlibm.
          case RIR_U_EXP:
            os << (row_libm(n) ? (row_functions ? "rn_row_exp(" : "exp(") : "rn_exp(") << x << ")";
            break;
          case RIR_U_LOG:
            os << (row_libm(n) ? (row_functions ? "rn_row_log(" : "log(") : "rn_log(") << x << ")";
            break;
          case RIR_U_ABS: os << "fabs(" << x << ")"; break;
          case RIR_U_NOOP: os << x; break;
          case RIR_U_SIN: os << "sin(" << x << ")"; break;
          case RIR_U_COS: os << "cos(" << x << ")"; break;
          case RIR_U_TAN: os << "tan(" << x << ")"; break;
          case RIR_U_ASIN: os << "asin(" << x << ")"; break;
          case RIR_U_ACOS: os << "acos(" << x << ")"; break;
          case RIR_U_ATAN: os << "atan(" << x << ")"; break;
          case U_NEG: os << "(-" << x << ")"; break;
          case U_RECIP: os << recip(x, row_libm(n)); break;
          case U_SQRT: os << "sqrt(" << x << ")"; break;
        }
        break;
      }
      case K_BINARY: {
        const std::string x = val(n.a), y = val(n.b);
        switch (n.op) {
          case RIR_B_ADD: os << "(" << x << " + " << y << ")"; break;
          case RIR_B_MUL: os << "(" << x << " * " << y << ")"; break;
          case RIR_B_SUB: os << "(" << x << " - " << y << ")"; break;
          case RIR_B_DIV:
            // Reverse-sweep quotients of the warp-per-chain row bodies (adj / x, the adjoint of log): their numerators are
            // exactly 0 for half the observations of a 0/1-valued column, and a zero numerator fails the range test of
            // CUDA's inline IEEE division, whose out-of-line completion then ran for 94 % of the warps: a quarter of all
            // instructions of cfg 3 (profiles/r2_ncu_cfg3_mma_v1_regions.txt).  adj * (1 / x) keeps the inline path (the
            // numerator is 1); one more rounding, in a region that agrees with the oracle to 1e-13 by construction
            // (tree sums), not bit for bit.  Everything that is compared bit for bit keeps the exact quotient.
            if (wpc && n.region == R_ROW_BWD)
              os << "(" << x << " * " << recip(y, true) << ")";
            else
              os << "(" << x << " / " << y << ")";
            break;
          case RIR_B_POW: os << pow_expr(n.a, n.b, n.region == R_ROW_BWD || n.region == R_INV_BWD, row_libm(n)); break;
          case RIR_B_COMPARE: os << "rn_compare(" << x << ", " << y << ")"; break;
        }
        break;
      }
      case K_LOOKUP: {
        // D2I ; tableswitch ; default -> throw (ir/ExprMethodGenerator.scala:50-56): flag + NaN instead of a fault
        if (wpc && tab_off.count(id)) {
          os << "rn_tab_lookup(scr + " << tab_off.at(id) << ", " << n.c << ", " << n.d << ", " << val(n.a) << ", err)";
          break;
        }
        os << "rn_lookup" << id << "(" << val(n.a);
        for (int k = 0; k < n.c; k++) os << ", " << val(P.lookup_refs[n.b + k]);
        os << ", err)";
        break;
      }
      case K_SELEQ: os << "((rn_d2i(" << val(n.a) << ") == " << n.d << ") ? " << val(n.b) << " : " << val(n.c) << ")"; break;
      case K_ACC: os << acc_ref(n.a); break;
    }
    os << ";\n";
  }

  // small lookups become a helper with a switch (keeps operands in registers)
  void lookup_helpers() {
    for (size_t id = 0; id < P.nodes.size(); id++) {
      const Node& n = P.nodes[id];
      if (n.kind != K_LOOKUP) continue;
      if (wpc && tab_off.count((int)id)) continue;
      os << "RN_DEVICE double rn_lookup" << id << "(double idx";
      for (int k = 0; k < n.c; k++) os << ", double e" << k;
      os << ", int& err) {\n  switch (rn_d2i(idx) - (" << n.d << ")) {\n";
      for (int k = 0; k < n.c; k++) os << "    case " << k << ": return e" << k << ";\n";
      os << "    default: err |= 1; return RN_NAN;\n  }\n}\n";
    }
  }

  void density_tpc() {
    os << "// ---- emitted: log-density and gradient of the frozen DAG (" << (P.symbolic ? "symbolic" : "adjoint")
       << " gradient) ----\n";
    lookup_helpers();
    os << "RN_DEVICE void rn_density(const double (&q)[RN_N], double& dens, double (&grad)[RN_N], "
          "const double* RN_RESTRICT data, int& err) {\n";
    os << "  (void)data; (void)err;\n";
    os << "  double acc[RN_NSLOTS];\n  for (int s = 0; s < RN_NSLOTS; s++) acc[s] = 0.0;\n";
    for (int id : P.inv_fwd) stmt(id, "  ");
    for (size_t t = 0; t < P.targets.size(); t++) {
      const TargetInfo& T = P.targets[t];
      os << "  // target " << t << (T.streamed() ? " (streamed)" : " (data-free)") << "\n";
      if (T.streamed()) {
        os << "  for (long long row = 0; row < " << (long long)T.n_rows << "LL; row++) {\n";
        const int pitch = opt.pitch(t);
        os << "    const double* RN_RESTRICT rp = data + " << (unsigned long long)opt.target_base[t] << "ULL + (row >> 5) * "
           << (unsigned long long)T.n_cols * pitch << "LL + (row & 31);\n";
        row_body(
            T, "    ", [&](int k) { return "RN_LDG(rp + " + std::to_string(local_col(T, k) * pitch) + ")"; },
            [&](int slot) { return "acc[" + std::to_string(slot) + "]"; }, false, 0);
        os << "  }\n";
      } else {
        for (const AccStmt& a : T.row_acc) os << "  acc[" << a.slot << "] += " << val(a.node) << ";\n";
      }
    }
    os << "  dens = acc[0];\n";
    if (P.symbolic) {
      os << "  RN_UNROLL\n  for (int i = 0; i < RN_N; i++) grad[i] = acc[1 + i];\n";
    } else {
      for (int id : P.inv_bwd) stmt(id, "  ");
      for (uint32_t i = 0; i < P.n_params; i++) os << "  grad[" << i << "] = " << val(P.grad_nodes[i]) << ";\n";
    }
    os << "}\n";
  }

  // Function flavour: forward evaluation of the m outputs of Compiler.compile(inputs, outputs).  An output is stored as
  // soon as its node is defined (500 requirements -- Generator.MaxRequirements -- must not stay live to the end).
  void function_tpc() {
    os << "// ---- emitted: the " << P.fn_outputs.size() << " outputs of the compiled function (forward only) ----\n";
    lookup_helpers();
    os << "RN_DEVICE void rn_function(const double (&q)[RN_NQ], double* RN_RESTRICT out, const long long os, int& err) {\n";
    os << "  (void)q; (void)err;\n";
    std::map<int, std::vector<int>> out_at;
    std::vector<int> tail;
    for (size_t j = 0; j < P.fn_outputs.size(); j++) {
      const Node& n = P.nodes[P.fn_outputs[j]];
      if (n.kind == K_CONST || n.kind == K_INPUT)
        tail.push_back((int)j);
      else
        out_at[P.fn_outputs[j]].push_back((int)j);
    }
    for (int id : P.inv_fwd) {
      stmt(id, "  ");
      auto it = out_at.find(id);
      if (it != out_at.end())
        for (int j : it->second) os << "  out[" << j << "LL * os] = " << val(id) << ";\n";
    }
    for (int j : tail) os << "  out[" << j << "LL * os] = " << val(P.fn_outputs[j]) << ";\n";
    os << "}\n";
  }


  // =============================================================================================================
  // Chain-batched fp64 tensor-core path (DMMA, mma.sync.m8n8k4.f64) for streamed targets whose row body is
  //     [dot products  z_d = base + sum_j q[p_j] * x_{d,j}]  ->  [elementwise code on z_d]  ->  sum over d
  // -- the Translator's left fold of a `Line` with column coefficients (compute/Translator.scala:91-125), once per
  // unrolled observation of Model.observe (core/Model.scala:98-132): logistic / Poisson / Gaussian regressions.
  // Over the 8 chains of a CTA and the 32 rows of a tile the dots are Z^T[8 x 32] = B^T[8 x d] X^T[d x 32] and their
  // adjoints G^T[8 x d] += W^T[8 x 32] X[32 x d]: warp w takes dot w (its own column block of every tile, fetched by its
  // own single-stage TMA pipeline), computes both products for ALL 8 chains with DMMA -- one staged x_ij then serves 8
  // chains instead of one (rows-across-lanes: one LDS.64 per DFMA, the shared-memory pipe was the busiest unit of round
  // 1's kernel) -- and runs the emitted elementwise code on the C fragments (lane: chain = lane/4, row slots 2*(lane%4)+{0,1}).
  // The per-warp partial sums meet in a CTA scratch and every chain's warp adds them in one fixed order (deterministic).
  // Fragment maps (PTX ISA, mma.m8n8k4 .f64): A[m = lane/4][k = lane%4], B[k = lane%4][n = lane/4], C[m = lane/4][n = 2*(lane%4)+{0,1}].
  //   forward   m = chain, k = term, n = row slot;   backward  m = chain, k = row slot (2*(lane%4)+h for k-step h), n = term.
  // Row slot n of an 8-row group is physical row n ^ ((n >> 2) & 1): with a column pitch of 36 doubles both B-operand
  // access patterns are then bank-conflict free per half-warp.
  // =============================================================================================================
  struct MmaDot {
    int z = -1, w = -1, base = -1;
    std::vector<int> cols;     // local column index of every term
    std::vector<int> leaves;   // leaves of the output sum owned by this dot
    std::vector<int> fwd, bwd; // row nodes its elementwise code needs, emission order
    std::vector<AccStmt> acc;  // accumulations other than density / dot-term adjoints: (index into plan.other_slots, node)
    int cmin = 0, cmax = 0;
  };
  struct MmaPlan {
    bool ok = false;
    std::vector<int> params;       // common term -> parameter map
    std::vector<int> param_slot;   // accumulator slot of every term's parameter
    std::vector<MmaDot> dots;
    std::vector<int> other_slots;  // accumulator slots (besides 0 and the term parameters') the elementwise code adds to
    int KS = 0, DT = 0, region_doubles = 0, redw = 0;
    bool uniform = false;  // every dot is the same code over its own column block (the unrolled observations of Model.observe):
                           // ONE copy of the per-dot code serves all warps, only the block's first column differs
  };
  std::vector<MmaPlan> plans;
  std::vector<int> mma_inv;        // invariant nodes some elementwise body reads (published per chain through shared memory)
  int mma_inv_off = 0;
  bool mma_all_ok = false;
  int mma_shared_doubles = 0;
  static constexpr int MMA_WARPS = 8;  // warps of one chain group = column-block regions / barriers per CTA
  int mma_groups() const { return opt.mma_chains >= 16 ? 2 : 1; }

  static MmaPlan why(MmaPlan& pl, int line) {
    if (getenv("RN_MMA_DEBUG")) fprintf(stderr, "[rn mma] target not eligible for the DMMA path: check %d\n", line);
    return pl;
  }
  MmaPlan plan_mma(const TargetInfo& T, size_t t) {
    MmaPlan pl;
    const int pitch = opt.pitch(t);
    if (P.symbolic || !T.streamed() || T.dots.empty() || !T.row_scatter.empty() || pitch < 36 || T.dots.size() > 64) return why(pl, 1);
    pl.params = T.dots[0].params;
    if (pl.params.size() < 4) return why(pl, 2);
    for (const DotInfo& d : T.dots)
      if (d.params != pl.params) return why(pl, 3);
    std::set<int> rowset(T.row_fwd.begin(), T.row_fwd.end());
    rowset.insert(T.row_bwd.begin(), T.row_bwd.end());
    // dot internals: the term products and the partial sums of the fold
    std::map<int, int> zdot;
    std::set<int> internal;
    for (size_t di = 0; di < T.dots.size(); di++) {
      const DotInfo& d = T.dots[di];
      zdot[d.node] = (int)di;
      int cur = d.node;
      for (size_t k = d.params.size(); k-- > 0;) {
        const Node& a = P.nodes[cur];
        if (k == 0 && d.base < 0) {
          internal.insert(cur);  // the first term itself
          break;
        }
        if (a.kind != K_BINARY || a.op != RIR_B_ADD) return why(pl, 4);
        internal.insert(a.b);
        if (cur != d.node) internal.insert(cur);
        cur = a.a;
      }
    }
    // which dots a row node depends on (through z_d); touching a dot internal any other way disqualifies
    std::map<int, uint64_t> memo;
    bool bad = false;
    std::vector<int> ops;
    std::function<uint64_t(int)> mask = [&](int id) -> uint64_t {
      auto z = zdot.find(id);
      if (z != zdot.end()) return 1ull << z->second;
      if (internal.count(id)) {
        bad = true;
        return 0;
      }
      if (!rowset.count(id)) return 0;
      auto it = memo.find(id);
      if (it != memo.end()) return it->second;
      std::vector<int> o;
      operands(id, o);
      uint64_t m = 0;
      for (int x : o) m |= mask(x);
      memo[id] = m;
      return m;
    };
    auto single = [&](uint64_t m) { return m != 0 && (m & (m - 1)) == 0; };
    auto owner = [&](uint64_t m) {
      int d = 0;
      while (m > 1) {
        m >>= 1;
        d++;
      }
      return d;
    };
    for (const DotInfo& d : T.dots)  // the fold's first operand (an intercept, the observation column of a residual) may be any
      if (d.base >= 0 && (mask(d.base) != 0 || bad)) return why(pl, 5);  // value that does not itself hang on a dot
    pl.dots.resize(T.dots.size());
    for (size_t di = 0; di < T.dots.size(); di++) {
      pl.dots[di].z = T.dots[di].node;
      pl.dots[di].base = T.dots[di].base;
      for (int c : T.dots[di].columns) pl.dots[di].cols.push_back(local_col(T, c - (int)P.n_params));  // DotInfo holds input indices
    }
    // output: a sum whose leaves depend on one dot each
    std::function<bool(int)> leaves = [&](int id) -> bool {
      const uint64_t m = mask(id);
      if (bad) return false;
      if (m == 0 || single(m)) {
        pl.dots[m ? owner(m) : 0].leaves.push_back(id);
        return true;
      }
      const Node& n = P.nodes[id];
      if (n.kind != K_BINARY || n.op != RIR_B_ADD) return false;
      return leaves(n.a) && leaves(n.b);
    };
    if (!leaves(T.outputs[0]) || bad) return why(pl, 6);
    // accumulations
    std::map<int, int> slot_of_param;
    std::map<int, int> other_index;
    for (const AccStmt& a : T.row_acc) {
      if (a.slot == 0 && a.node == T.outputs[0]) continue;
      const Node& c = P.nodes[a.node];
      bool term_adj = false;
      if (c.kind == K_BINARY && c.op == RIR_B_MUL && rowset.count(a.node)) {
        // MUL(adjoint of z_d, column of term k) -> the DMMA's job
        for (int swap = 0; swap < 2 && !term_adj; swap++) {
          const int wn = swap ? c.b : c.a, cn = swap ? c.a : c.b;
          const Node& col = P.nodes[cn];
          if (col.kind != K_INPUT || (uint32_t)col.a < P.n_params) continue;
          const int lc = local_col(T, col.a - (int)P.n_params);
          for (size_t di = 0; di < pl.dots.size() && !term_adj; di++)
            for (size_t k = 0; k < pl.dots[di].cols.size(); k++)
              if (pl.dots[di].cols[k] == lc) {
                if (pl.dots[di].w >= 0 && pl.dots[di].w != wn) return why(pl, 7);
                auto sp = slot_of_param.find(pl.params[k]);
                if (sp != slot_of_param.end() && sp->second != a.slot) return why(pl, 8);
                slot_of_param[pl.params[k]] = a.slot;
                pl.dots[di].w = wn;
                term_adj = true;
                break;
              }
        }
      }
      if (term_adj) continue;
      const uint64_t m = mask(a.node);
      if (bad || (m != 0 && !single(m))) return why(pl, 9);
      if (a.slot == 0) return why(pl, 10);  // (density contributions come through the leaves only)
      if (smem_slot[a.slot] >= 0) return why(pl, 11);
      auto oi = other_index.find(a.slot);
      if (oi == other_index.end()) {
        oi = other_index.emplace(a.slot, (int)pl.other_slots.size()).first;
        pl.other_slots.push_back(a.slot);
      }
      pl.dots[m ? owner(m) : 0].acc.push_back({oi->second, a.node});
    }
    for (size_t k = 0; k < pl.params.size(); k++) {
      auto sp = slot_of_param.find(pl.params[k]);
      if (sp == slot_of_param.end() || smem_slot[sp->second] >= 0) return why(pl, 12);
      pl.param_slot.push_back(sp->second);
    }
    // needed nodes and column ranges per dot
    for (size_t di = 0; di < pl.dots.size(); di++) {
      MmaDot& d = pl.dots[di];
      if (d.w < 0) return why(pl, 13);
      std::set<int> need;
      std::set<int> colset(d.cols.begin(), d.cols.end());
      std::function<bool(int)> visit = [&](int id) -> bool {
        if (id == d.z) {
          need.insert(id);  // (keeps its place in the emission order; its operands are the DMMA's)
          return true;
        }
        if (zdot.count(id) || internal.count(id)) return false;
        const Node& n = P.nodes[id];
        if (n.kind == K_CONST) return true;
        if (n.kind == K_INPUT) {
          if ((uint32_t)n.a >= P.n_params) colset.insert(local_col(T, n.a - (int)P.n_params));
          return true;
        }
        if (!rowset.count(id)) {  // an invariant value of the chain
          if (n.region != R_INV_FWD) return false;
          if (std::find(mma_inv.begin(), mma_inv.end(), id) == mma_inv.end()) mma_inv.push_back(id);
          return true;
        }
        if (tab_off.count(id)) return false;  // table lookups read the chain's own scratch
        if (!need.insert(id).second) return true;
        std::vector<int> o;
        operands(id, o);
        for (int x : o)
          if (!visit(x)) return false;
        return true;
      };
      for (int l : d.leaves)
        if (!visit(l)) return why(pl, 14);
      if (!visit(d.w)) return why(pl, 15);
      for (const AccStmt& a : d.acc)
        if (!visit(a.node)) return why(pl, 16);
      if (d.base >= 0 && !visit(d.base)) return why(pl, 17);
      for (int id : T.row_fwd)
        if (need.count(id)) d.fwd.push_back(id);
      for (int id : T.row_bwd)
        if (need.count(id)) d.bwd.push_back(id);
      d.cmin = *colset.begin();
      d.cmax = *colset.rbegin();
      pl.region_doubles = std::max(pl.region_doubles, (d.cmax - d.cmin + 1) * pitch);
    }
    pl.KS = ((int)pl.params.size() + 3) / 4;
    pl.DT = ((int)pl.params.size() + 7) / 8;
    pl.redw = pl.DT * 8 + 1 + (int)pl.other_slots.size();
    pl.uniform = true;
    {
      const std::vector<std::string> s0 = mma_signature(T, pl, pl.dots[0]);
      for (size_t di = 1; di < pl.dots.size() && pl.uniform; di++) {
        const std::vector<std::string> sd = mma_signature(T, pl, pl.dots[di]);
        if (sd != s0) {
          pl.uniform = false;
          if (getenv("RN_MMA_DEBUG")) {
            fprintf(stderr, "[rn mma] dot %zu differs from dot 0 (%zu vs %zu statements)\n", di, sd.size(), s0.size());
            for (size_t k = 0; k < std::min(sd.size(), s0.size()); k++)
              if (sd[k] != s0[k]) {
                fprintf(stderr, "  #%zu: %s  vs  %s\n", k, s0[k].c_str(), sd[k].c_str());
                break;
              }
          }
        }
      }
    }
    pl.ok = true;
    return pl;
  }


  // canonical form of one dot's elementwise code: node kinds / ops / constants, operands as positions in the dot's own
  // statement list, columns relative to the block's first column -- equal signatures = the same code on another block
  std::vector<std::string> mma_signature(const TargetInfo& T, const MmaPlan& pl, const MmaDot& d) const {
    std::map<int, int> pos;
    std::vector<int> order = d.fwd;
    order.insert(order.end(), d.bwd.begin(), d.bwd.end());
    for (size_t k = 0; k < order.size(); k++) pos[order[k]] = (int)k;
    auto ref = [&](int id) -> std::string {
      if (id == d.z) return "z";
      auto it = pos.find(id);
      if (it != pos.end()) return "n" + std::to_string(it->second);
      const Node& n = P.nodes[id];
      if (n.kind == K_CONST) return "k" + lit(n.value);
      if (n.kind == K_INPUT) return (uint32_t)n.a < P.n_params ? "q" + std::to_string(n.a) : "c" + std::to_string(local_col(T, n.a - (int)P.n_params) - d.cmin);
      return "i" + std::to_string(id);  // invariant node of the chain
    };
    std::vector<std::string> out;
    std::vector<int> o;
    for (int id : order) {
      if (id == d.z) {
        out.push_back("Z" + (d.base >= 0 ? ref(d.base) : std::string("-")));
        continue;
      }
      const Node& n = P.nodes[id];
      // constants of the node: op; Lookup: len, low (its entries are operands); SelEq: the compared index
      std::string sg = std::to_string(n.kind) + ":" + std::to_string(n.op) + ":" + (n.kind == K_LOOKUP ? std::to_string(n.c) : std::string("-")) + ":" +
                       ((n.kind == K_LOOKUP || n.kind == K_SELEQ) ? std::to_string(n.d) : std::string("-")) + ":" + std::to_string(n.region) +
                       (tab_off.count(id) ? "T" : "");
      operands(id, o);
      for (int x : o) sg += "," + ref(x);
      out.push_back(sg);
    }
    std::string tail = "L";
    for (int l : d.leaves) tail += "," + ref(l);
    tail += "|W" + ref(d.w) + "|A";
    for (const AccStmt& a : d.acc) tail += "," + std::to_string(a.slot) + "=" + ref(a.node);
    tail += "|C";
    for (int c : d.cols) tail += "," + std::to_string(c - d.cmin);
    tail += "|" + std::to_string(d.cmax - d.cmin);
    out.push_back(tail);
    (void)pl;
    return out;
  }

  // the elementwise code of one dot for FOUR of the lane's eight (row, chain) elements of a tile (element e = 2*nt + h: 8-row
  // group nt, row slot 2*(lane%4)+h; the call handles groups roff/8 and roff/8 + 1), statement by statement across the
  // elements: four independent dependency chains for the scheduler, like the interleaved observations of the
  // rows-across-lanes body (one element at a time left a warp with a single serial chain of exp / log / divisions; eight at
  // a time spilled at 128 registers)
  void mma_helper(const TargetInfo& T, size_t t, const MmaPlan& pl, size_t di) {
    in_mma_helper = true;
    const MmaDot& d = pl.dots[di];
    const int pitch = opt.pitch(t);
    os << "RN_DEVICE void rn_mma_e" << t << "_" << di << "(const double* zz, const RnSA rp0, const RnSA rp1, const int roff, const double* RN_RESTRICT q, "
          "const double* RN_RESTRICT xv, double& dens, double* wout, double* osum, int& err) {\n"
       << "  (void)rp0; (void)rp1; (void)roff; (void)q; (void)xv; (void)osum; (void)err;\n";
    for (size_t k = 0; k < mma_inv.size(); k++) os << "  const double v" << mma_inv[k] << " = xv[" << k << "]; (void)v" << mma_inv[k] << ";\n";
    std::set<int> declared[4];
    auto sfx = [&](int e) { return "_" + std::to_string(e); };
    auto need_col = [&](int o, int e) {
      const Node& n = P.nodes[o];
      if (n.kind != K_INPUT || (uint32_t)n.a < P.n_params) return;
      const int k = n.a - (int)P.n_params;
      if (declared[e].insert(k).second)
        os << "  const double c" << k << sfx(e) << " = rn_lds(" << (e & 1 ? "rp1" : "rp0") << ", roff + " << (e >> 1) * 8 + (local_col(T, k) - d.cmin) * pitch << ");\n";
    };
    std::vector<int> o;
    auto one = [&](int id) {
      for (int e = 0; e < 4; e++) {
        node_suffix = col_suffix = sfx(e);
        if (id == d.z) {  // the dot itself: the tensor core's sum, plus the fold's first operand
          if (d.base >= 0) {
            need_col(d.base, e);
            os << "  const double " << val(d.z) << " = " << val(d.base) << " + zz[" << e << "];\n";
          } else {
            os << "  const double " << val(d.z) << " = zz[" << e << "];\n";
          }
          continue;
        }
        operands(id, o);
        for (int x : o) need_col(x, e);
        stmt(id, "  ");
      }
    };
    bool z_done = false;
    for (int id : d.fwd) {
      one(id);
      if (id == d.z) z_done = true;
    }
    if (!z_done) one(d.z);
    for (int l : d.leaves)
      for (int e = 0; e < 4; e++) {
        node_suffix = col_suffix = sfx(e);
        need_col(l, e);
        os << "  dens += " << val(l) << ";\n";
      }
    for (int id : d.bwd) one(id);
    for (int e = 0; e < 4; e++) {
      node_suffix = col_suffix = sfx(e);
      need_col(d.w, e);
      os << "  wout[" << e << "] = " << val(d.w) << ";\n";
      for (const AccStmt& a : d.acc) {
        need_col(a.node, e);
        os << "  osum[" << a.slot << "] += " << val(a.node) << ";\n";
      }
    }
    node_suffix.clear();
    col_suffix.clear();
    os << "}\n";
    in_mma_helper = false;
  }

  void mma_block(const TargetInfo& T, size_t t, const MmaPlan& pl, unsigned long long n_full) {
    const int pitch = opt.pitch(t), NP = (int)pl.params.size(), KS = pl.KS, DT = pl.DT, NO = (int)pl.other_slots.size();
    const unsigned long long base = (unsigned long long)opt.target_base[t], td = (unsigned long long)T.n_cols * pitch;
    const int NG = mma_groups();
    os << "    if (tma.on) {  // chain-batched DMMA over the CTA's " << 8 * NG << " chains: warp w <-> dot w % 8 for chain group w / 8 (see Emitter::mma_block)\n"
       << "      const int wfull = (int)(threadIdx.x >> 5), wid = wfull & 7, cg = wfull >> 3, ln = (int)(threadIdx.x & 31), mc = ln >> 2, mk = ln & 3;\n"
       << "      (void)cg;\n";
    if (!mma_inv.empty()) {
      os << "      if (ln == 0) {\n";
      for (size_t k = 0; k < mma_inv.size(); k++) os << "        scr[" << (mma_inv_off + (int)k) << "] = " << val(mma_inv[k]) << ";\n";
      os << "      }\n";
    }
    os << "      rn_cta_bar(tma.nthreads);  // every chain's q (and invariants) are in its slice\n"
       << "      const double* qo = q + (cg * 8 + mc - wfull) * RN_WPC_SMEM_DOUBLES;\n"
       << "      const double* xo = scr + (cg * 8 + mc - wfull) * RN_WPC_SMEM_DOUBLES + " << mma_inv_off << ";\n"
       << "      (void)xo;\n"
       << "      double ar[" << KS << "];\n";
    for (int ks = 0; ks < KS; ks++) {
      // term ks*4 + mk: parameter index by lane
      os << "      ar[" << ks << "] = ";
      std::string e = "0.0";
      for (int k = 3; k >= 0; k--) {
        const int term = ks * 4 + k;
        const std::string v = term < NP ? "qo[" + std::to_string(pl.params[term]) + "]" : "0.0";
        e = k == 3 ? v : "(mk == " + std::to_string(k) + " ? " + v + " : " + e + ")";
      }
      os << e << ";\n";
    }
    os << "      double g[" << DT << "][2];\n      for (int i = 0; i < " << DT << "; i++) g[i][0] = g[i][1] = 0.0;\n"
       << "      double dsum = 0.0, osum[" << std::max(1, NO) << "];\n      for (int i = 0; i < " << std::max(1, NO) << "; i++) osum[i] = 0.0;\n"
       << "      double* const region = tma.stage + (size_t)wid * " << pl.region_doubles << ";\n"
       << "      unsigned long long* const bar = tma.full + wid;\n"
       << "      const double* RN_RESTRICT src = data + " << base << "ULL;\n";
    // the per-dot code: once for all warps when the dots are the same code over their own column blocks (then only the
    // block's first column differs -- a table indexed by the dot), else one copy per dot.  Kept SMALL on purpose: eight
    // unrolled copies (170 KB of SASS) thrashed the instruction cache and ran 3x SLOWER than rows-across-lanes
    // (profiles/r2_bench_mma_v1_icache_thrash.txt); the 8-row groups of a tile are a rolled loop for the same reason.
    const size_t ncopies = pl.uniform ? 1 : pl.dots.size();
    if (pl.uniform) {
      os << "      static const int MMA_CMIN" << t << "[" << pl.dots.size() << "] = {";
      for (size_t di = 0; di < pl.dots.size(); di++) os << (di ? ", " : "") << pl.dots[di].cmin;
      os << "};\n";
    }
    for (size_t ci = 0; ci < ncopies; ci++) {
      const MmaDot& d = pl.dots[ci];
      const unsigned bytes = (unsigned)((d.cmax - d.cmin + 1) * pitch * 8);
      // the B-operand addresses: per lane a base (term by lane, row slot by lane) plus compile-time offsets when the dot's
      // columns are an arithmetic progression (the Translator folds a Vec.dot in column order); else per-lane offset tables
      bool ap = true;
      const int step = d.cols.size() > 1 ? d.cols[1] - d.cols[0] : 1;
      for (size_t k = 1; k < d.cols.size(); k++)
        if (d.cols[k] - d.cols[k - 1] != step) ap = false;
      auto off = [&](int term) { return (d.cols[term < NP ? term : 0] - d.cmin) * pitch; };
      auto by_lane = [&](const char* lane, int n, std::function<std::string(int)> f) {  // nested select over lane index 0..n-1
        std::string e;
        for (int k = n - 1; k >= 0; k--) e = k == n - 1 ? f(k) : "(" + std::string(lane) + " == " + std::to_string(k) + " ? " + f(k) + " : " + e + ")";
        return e;
      };
      if (pl.uniform)
        os << "      for (int dot = wid; dot < " << pl.dots.size() << "; dot += " << MMA_WARPS << ") {  // this warp's dots (same code, other column block)\n"
           << "        const double* RN_RESTRICT s0 = src + (size_t)MMA_CMIN" << t << "[dot] * " << pitch << ";\n";
      else
        os << "      if (wid == " << (ci % MMA_WARPS) << ") {  // dot " << ci << ": columns " << d.cmin << ".." << d.cmax << " of the tile\n"
           << "        const double* RN_RESTRICT s0 = src + " << (unsigned long long)d.cmin * pitch << "ULL;\n";
      os << "        if (ln == 0 && cg == 0) rn_tma_load_raw(region, bar, s0, " << bytes << "u);\n"
         << "        const int pf = mc ^ ((mc >> 2) & 1), pb0 = (2 * mk) ^ ((mk >> 1) & 1), pb1 = (2 * mk + 1) ^ ((mk >> 1) & 1);\n";
      if (ap) {
        os << "        const RnSA bf = rn_sa(region + pf + (" << (d.cols[0] - d.cmin) << " + " << step << " * mk) * " << pitch << ");\n"
           << "        const RnSA bb0 = rn_sa(region + pb0 + (" << (d.cols[0] - d.cmin) << " + " << step << " * mc) * " << pitch << ");\n"
           << "        const RnSA bb1 = rn_sa(region + pb1 + (" << (d.cols[0] - d.cmin) << " + " << step << " * mc) * " << pitch << ");\n";
      } else {
        os << "        int fo[" << KS << "], bo[" << DT << "];\n";
        for (int ks = 0; ks < KS; ks++)
          os << "        fo[" << ks << "] = " << by_lane("mk", 4, [&](int k) { return std::to_string(off(ks * 4 + k)); }) << ";\n";
        for (int dt = 0; dt < DT; dt++)
          os << "        bo[" << dt << "] = " << by_lane("mc", 8, [&](int k) { return std::to_string(off(dt * 8 + k)); }) << ";\n";
        os << "        const RnSA bf = rn_sa(region + pf), bb0 = rn_sa(region + pb0), bb1 = rn_sa(region + pb1);\n";
      }
      os << "        const RnSA e0 = rn_sa(region + pb0), e1 = rn_sa(region + pb1);\n";
      // padded terms (beyond the NP of the dot) multiply an operand of exact zeros; their B address must still be a finite
      // number of the tile: the last group falls back to term 0's column
      auto fwd_addr = [&](int ks) -> std::string {
        if (!ap) return "fo[" + std::to_string(ks) + "]";
        const int first = ks * 4;
        if (first + 3 < NP) return std::to_string(4 * step * ks * pitch);
        return "(mk < " + std::to_string(NP - first) + " ? " + std::to_string(4 * step * ks * pitch) + " : " + std::to_string(off(0)) + " - (" +
               std::to_string(d.cols[0] - d.cmin) + " + " + std::to_string(step) + " * mk) * " + std::to_string(pitch) + ")";
      };
      auto bwd_addr = [&](int dt) -> std::string {
        if (!ap) return "bo[" + std::to_string(dt) + "]";
        const int first = dt * 8;
        if (first + 7 < NP) return std::to_string(8 * step * dt * pitch);
        return "(mc < " + std::to_string(NP - first) + " ? " + std::to_string(8 * step * dt * pitch) + " : " + std::to_string(off(0)) + " - (" +
               std::to_string(d.cols[0] - d.cmin) + " + " + std::to_string(step) + " * mc) * " + std::to_string(pitch) + ")";
      };
      os << "        for (unsigned tile = 0; tile < " << n_full << "u; tile++) {\n"
         << "          rn_mbar_wait_warp(bar, tma.seq & 1u);\n          tma.seq += 1;\n"
         << "          double z[8], wv[8];\n"
         << "          RN_UNROLL\n          for (int e = 0; e < 8; e++) z[e] = 0.0;\n";
      for (int ks = 0; ks < KS; ks++)  // term groups outermost: four independent accumulator chains (the tile's 8-row groups)
        for (int nt = 0; nt < 4; nt++)
          os << "          rn_dmma(z[" << 2 * nt << "], z[" << 2 * nt + 1 << "], ar[" << ks << "], rn_lds(bf, " << nt * 8 << " + " << fwd_addr(ks) << "));\n";
      os << "          rn_mma_e" << t << "_" << ci << "(z, e0, e1, 0, qo, xo, dsum, wv, osum, err);\n"
         << "          rn_mma_e" << t << "_" << ci << "(z + 4, e0, e1, 16, qo, xo, dsum, wv + 4, osum, err);\n";
      for (int nt = 0; nt < 4; nt++)
        for (int h = 0; h < 2; h++)
          for (int dt = 0; dt < DT; dt++)
            os << "          rn_dmma(g[" << dt << "][0], g[" << dt << "][1], wv[" << 2 * nt + h << "], rn_lds(" << (h ? "bb1" : "bb0") << ", " << nt * 8 << " + "
               << bwd_addr(dt) << "));\n";
      os
         << "          " << (NG > 1 ? "rn_pair_bar(2 + wid, 64);  // both warps of the pair are done with the block" : "__syncwarp();") << "\n"
         << "          if (ln == 0 && cg == 0 && tile + 1 < " << n_full << "u) rn_tma_load_raw(region, bar, s0 + (size_t)(tile + 1) * " << td << "ULL, " << bytes << "u);\n"
         << "        }\n      }\n";
    }
    // per-warp partials -> CTA scratch [warp][chain][redw]; chain wid's warp totals them in warp order
    const int NPAD = DT * 8;
    os << "      double* const red = tma.stage + (size_t)" << MMA_WARPS << " * " << pl.region_doubles << ";\n"
       << "      double* const mine = red + (size_t)(wfull * 8 + mc) * " << pl.redw << ";\n";
    for (int dt = 0; dt < DT; dt++)
      os << "      mine[" << dt * 8 << " + 2 * mk] = g[" << dt << "][0];\n      mine[" << dt * 8 << " + 2 * mk + 1] = g[" << dt << "][1];\n";
    os << "      dsum += __shfl_xor_sync(0xffffffffu, dsum, 1);\n      dsum += __shfl_xor_sync(0xffffffffu, dsum, 2);\n"
       << "      if (mk == 0) mine[" << NPAD << "] = dsum;\n";
    for (int k = 0; k < NO; k++)
      os << "      osum[" << k << "] += __shfl_xor_sync(0xffffffffu, osum[" << k << "], 1);\n      osum[" << k
         << "] += __shfl_xor_sync(0xffffffffu, osum[" << k << "], 2);\n      if (mk == 0) mine[" << NPAD + 1 + k << "] = osum[" << k << "];\n";
    os << "      rn_cta_bar(tma.nthreads);\n"
       << "      double* const tot = red + (size_t)(wfull * 8 + wid) * " << pl.redw << ";  // (read by this warp only)\n"
       << "      for (int j = ln; j < " << pl.redw << "; j += 32) {\n"
       << "        double s = 0.0;\n"
       << "        for (int w8 = 0; w8 < " << std::min<int>(MMA_WARPS, (int)pl.dots.size()) << "; w8++) s += red[(size_t)((cg * 8 + w8) * 8 + wid) * " << pl.redw << " + j];\n"
       << "        tot[j] = s;\n      }\n"
       << "      __syncwarp();\n"
       << "      if (ln == 0) {\n"
       << "        " << acc_ref(0) << " += tot[" << NPAD << "];\n";
    for (int k = 0; k < NP; k++) os << "        " << acc_ref(pl.param_slot[k]) << " += tot[" << k << "];\n";
    for (int k = 0; k < NO; k++) os << "        " << acc_ref(pl.other_slots[k]) << " += tot[" << NPAD + 1 + k << "];\n";
    os << "      }\n"
       << "      row0 += " << n_full * 32ull << "LL;\n"
       << "    }\n";
  }

  // ---- re-rolling of the invariant sections (warp-per-chain) ----------------------------------------------------------
  // The reference unrolls everything: a vector of 1000 latent group effects is 1000 copies of the same prior term, 1000 table
  // entries mu + sd * z_k, 1000 gradient expressions.  On the thread-per-chain shape that is one copy per chain.  On this shape
  // every thread of the chain's group would run the same ~20 000 straight-line statements with ~2000 values live across the row
  // loops (cfg 5: 19 KB of stack per thread, 1.4e9 local-memory accesses and 244 GB of DRAM traffic per launch, a fifth of the
  // stall samples; profiles/r2_ncu_cfg5_v1.csv).  So families of isomorphic statements are found again by anti-unification
  // from three kinds of seeds -- the entries of a Lookup table, the gradient outputs of consecutive parameters, the terms of a
  // long left fold of additions -- and emitted as ONE loop over the members with the members across the group's threads:
  //   for (k = lane; k < L; k += RN_G) { w0 = q[i0 + k]; w1 = (vU * w0); ...; scr[tab + k] = w5; }
  // Leaves are either uniform (the same scalar node for every member), parameters q[a + b k], or shared accumulators
  // scr[a + b k].  Interior values other sections need are recomputed by the family that needs them.  Sums over a family are
  // accumulated per thread and reduced across the group in a fixed order (the per-element values are bit-identical to the
  // unrolled statements; only the association of those sums changes, like the row sums of this shape).
  struct VNode {
    std::vector<int> mem;
    int leaf = 0;  // 0 interior, 1 parameter gather, 2 shared-accumulator gather
    long long base = 0, stride = 0;
  };
  struct FamOut {
    int kind = 0;  // 0 table store, 1 gradient store, 2 sum
    int vn = -1;   // vnode index, or -1 - node id when the value is uniform... (not produced: uniform seeds are refused)
    long long base = 0, stride = 0;  // table offset in scratch / first parameter index
    int sum = -1;                    // index into rr_sums
  };
  struct Family {
    int L = 0;
    std::vector<VNode> vn;
    std::map<std::vector<int>, int> memo;  // member vector -> vnode index (-2 failed)
    std::set<int> uniforms;      // scalar statements the loop reads
    std::set<int> uniform_all;   // ... plus constants and parameters used uniformly
    std::vector<FamOut> outs;
    bool bwd = false;
    bool done = false;
  };
  struct Spine {
    int end = -1;                    // node holding the complete sum
    std::vector<int> chain;          // interior fold nodes (eliminated)
    std::vector<int> scalar_terms;   // terms left to the scalar code, fold order
    std::vector<int> sums;           // rr_sums indices added after them
    bool bwd = false;
  };
  std::vector<Family> fams;
  std::vector<Spine> spines;
  int rr_n_sums = 0;
  std::set<int> rr_elim;               // scalar statements not emitted
  std::map<int, int> rr_spine_of;      // end node -> spine index
  std::set<int> rr_family_tables;      // tab_fill ids stored by a family
  std::vector<char> rr_family_grad;    // parameter i: gradient stored by a family
  std::map<int, std::string> name_override;
  int rr_max_round_sums = 0;

  static bool inv_region(const Node& n) { return n.region == R_INV_FWD || n.region == R_INV_BWD; }

  // anti-unification of L nodes; returns the vnode index, -1 - id for a uniform node, or INT_MIN on failure
  static constexpr int RR_FAIL = -2147483647;
  int rr_pack(Family& F, const std::vector<int>& V) {
    bool same = true;
    for (int id : V) same = same && id == V[0];
    if (same) {
      const Node& u = P.nodes[V[0]];
      if (u.kind != K_CONST && u.kind != K_INPUT) {
        if (!inv_region(u)) return RR_FAIL;
        F.uniforms.insert(V[0]);
      } else if (u.kind == K_INPUT && (uint32_t)u.a >= P.n_params) {
        return RR_FAIL;
      }
      F.uniform_all.insert(V[0]);
      return -1 - V[0];
    }
    auto it = F.memo.find(V);
    if (it != F.memo.end()) return it->second == -2 ? RR_FAIL : it->second;
    F.memo[V] = -2;
    const Node& n0 = P.nodes[V[0]];
    for (int id : V) {
      const Node& n = P.nodes[id];
      if (n.kind != n0.kind || n.op != n0.op) return RR_FAIL;
      if (n.kind != K_CONST && n.kind != K_INPUT && !inv_region(n)) return RR_FAIL;
    }
    VNode vn;
    vn.mem = V;
    auto affine = [&](const std::function<long long(int)>& get) {
      vn.base = get(0);
      vn.stride = V.size() > 1 ? get(1) - get(0) : 0;
      for (size_t k = 0; k < V.size(); k++)
        if (get((int)k) != vn.base + vn.stride * (long long)k) return false;
      return vn.stride != 0;
    };
    switch (n0.kind) {
      case K_CONST: {
        for (int id : V)
          if (std::memcmp(&P.nodes[id].value, &n0.value, sizeof(double)) != 0) return RR_FAIL;
        F.uniform_all.insert(V[0]);
        return -1 - V[0];
      }
      case K_INPUT: {
        for (int id : V)
          if ((uint32_t)P.nodes[id].a >= P.n_params) return RR_FAIL;
        if (!affine([&](int k) { return (long long)P.nodes[V[k]].a; })) return RR_FAIL;
        vn.leaf = 1;
        break;
      }
      case K_ACC: {
        for (int id : V)
          if (smem_slot[P.nodes[id].a] < 0) return RR_FAIL;
        if (!affine([&](int k) { return (long long)smem_slot[P.nodes[V[k]].a]; })) return RR_FAIL;
        vn.base += tab_doubles;
        vn.leaf = 2;
        break;
      }
      case K_UNARY:
      case K_BINARY: {
        std::vector<int> A(V.size()), B(V.size());
        for (size_t k = 0; k < V.size(); k++) {
          A[k] = P.nodes[V[k]].a;
          B[k] = P.nodes[V[k]].b;
        }
        if (rr_pack(F, A) == RR_FAIL) return RR_FAIL;
        if (n0.kind == K_BINARY && rr_pack(F, B) == RR_FAIL) return RR_FAIL;
        break;
      }
      default: return RR_FAIL;
    }
    F.vn.push_back(vn);
    return F.memo[V] = (int)F.vn.size() - 1;
  }

  // structural hash with holes for parameters and shared accumulators: equal hashes are necessary for rr_pack to succeed
  std::vector<uint64_t> rr_hash_memo;
  uint64_t rr_hash(int id) {
    if (rr_hash_memo[id]) return rr_hash_memo[id];
    const Node& n = P.nodes[id];
    auto mix = [](uint64_t h, uint64_t v) { return (h ^ (v + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2))) * 0xff51afd7ed558ccdull; };
    uint64_t h = mix(0x1234567ull, n.kind * 64 + n.op);
    switch (n.kind) {
      case K_CONST: {
        uint64_t b;
        std::memcpy(&b, &n.value, 8);
        h = mix(h, b);
        break;
      }
      case K_INPUT: h = mix(h, (uint32_t)n.a < P.n_params ? 1 : 1000 + n.a); break;
      case K_ACC: h = mix(h, smem_slot[n.a] >= 0 ? 2 : 2000 + n.a); break;
      case K_UNARY: h = mix(h, rr_hash(n.a)); break;
      case K_BINARY: h = mix(mix(h, rr_hash(n.a)), rr_hash(n.b)); break;
      default: h = mix(h, 7777 + (uint64_t)id); break;
    }
    if (!h) h = 1;
    return rr_hash_memo[id] = h;
  }

  void rr_plan() {
    const int MINL = 32;
    if (P.symbolic || getenv("RN_NO_REROLL")) return;
    const size_t nn = P.nodes.size();
    rr_hash_memo.assign(nn, 0);
    rr_family_grad.assign(P.n_params, 0);
    // use counts over everything that is emitted
    std::vector<int> uses(nn, 0);
    std::vector<int> ops;
    auto count_list = [&](const std::vector<int>& l) {
      for (int id : l) {
        operands(id, ops);
        for (int o : ops) uses[o]++;
      }
    };
    count_list(P.inv_fwd);
    count_list(P.inv_bwd);
    for (const TargetInfo& T : P.targets) {
      count_list(T.row_fwd);
      count_list(T.row_bwd);
      for (const AccStmt& a : T.row_acc) uses[a.node]++;
      for (const ScatterStmt& sc : T.row_scatter) uses[sc.node]++, uses[sc.index_node]++;
    }
    for (const AccStmt& a : P.inv_acc) uses[a.node]++;
    for (int g : P.grad_nodes) uses[g]++;

    auto try_family = [&](const std::vector<int>& V, FamOut out) -> bool {
      Family F;
      F.L = (int)V.size();
      const int r = rr_pack(F, V);
      if (r == RR_FAIL || r < 0) return false;
      // one representative per vnode names it during emission: they must be distinct
      std::set<int> reps;
      for (const VNode& v : F.vn)
        if (!reps.insert(v.mem[0]).second || F.uniform_all.count(v.mem[0])) return false;
      out.vn = r;
      F.outs.push_back(out);
      for (const VNode& v : F.vn)
        for (int id : v.mem) F.bwd = F.bwd || P.nodes[id].region == R_INV_BWD;
      for (int u : F.uniforms) F.bwd = F.bwd || P.nodes[u].region == R_INV_BWD;
      fams.push_back(std::move(F));
      return true;
    };

    // (A) Lookup tables
    for (int id : tab_fill) {
      const Node& n = P.nodes[id];
      if (n.c < MINL) continue;
      std::vector<int> V(P.lookup_refs.begin() + n.b, P.lookup_refs.begin() + n.b + n.c);
      FamOut o;
      o.kind = 0;
      o.base = tab_off.at(id);
      if (try_family(V, o)) rr_family_tables.insert(id);
    }
    // (C) gradient outputs of runs of consecutive parameters with the same shape
    for (uint32_t i = 0; i < P.n_params;) {
      uint32_t j = i + 1;
      const uint64_t h = rr_hash(P.grad_nodes[i]);
      while (j < P.n_params && rr_hash(P.grad_nodes[j]) == h) j++;
      if ((int)(j - i) >= MINL) {
        std::vector<int> V(P.grad_nodes.begin() + i, P.grad_nodes.begin() + j);
        FamOut o;
        o.kind = 1;
        o.base = i;
        if (try_family(V, o))
          for (uint32_t k = i; k < j; k++) rr_family_grad[k] = 1;
      }
      i = j;
    }
    // (B) long left folds of additions whose interior sums have no other reader
    std::vector<char> in_chain(nn, 0);
    auto scan_spines = [&](const std::vector<int>& list) {
      for (size_t pos = list.size(); pos-- > 0;) {
        const int end = list[pos];
        const Node& e = P.nodes[end];
        if (in_chain[end] || e.kind != K_BINARY || e.op != RIR_B_ADD) continue;
        std::vector<int> chain, terms;  // terms collected last-to-first
        int cur = end;
        for (;;) {
          const Node& c = P.nodes[cur];
          terms.push_back(c.b);
          const Node& l = P.nodes[c.a];
          if (l.kind == K_BINARY && l.op == RIR_B_ADD && uses[c.a] == 1 && inv_region(l) && !in_chain[c.a]) {
            chain.push_back(c.a);
            cur = c.a;
          } else {
            terms.push_back(c.a);
            break;
          }
        }
        if ((int)terms.size() < MINL) continue;
        std::reverse(terms.begin(), terms.end());
        Spine S;
        S.end = end;
        S.chain = chain;
        S.bwd = e.region == R_INV_BWD;
        bool any = false;
        for (size_t i = 0; i < terms.size();) {
          size_t j = i + 1;
          const uint64_t h = rr_hash(terms[i]);
          while (j < terms.size() && rr_hash(terms[j]) == h) j++;
          bool ok = false;
          if ((int)(j - i) >= MINL) {
            std::vector<int> V(terms.begin() + i, terms.begin() + j);
            FamOut o;
            o.kind = 2;
            o.sum = rr_n_sums;
            if (try_family(V, o)) {
              S.sums.push_back(rr_n_sums++);
              ok = any = true;
            }
          }
          if (!ok)
            for (size_t k = i; k < j; k++) S.scalar_terms.push_back(terms[k]);
          i = j;
        }
        if (!any) continue;
        for (int c : chain) in_chain[c] = 1;
        rr_spine_of[end] = (int)spines.size();
        spines.push_back(std::move(S));
      }
    };
    scan_spines(P.inv_fwd);
    scan_spines(P.inv_bwd);
    if (fams.empty()) return;

    // which absorbed statements can go: the members of the families and the interior fold nodes, unless something that is
    // still emitted as a scalar statement (or a row body, an accumulation, an unrolled table / gradient store) reads them
    std::set<int> absorbed;
    for (const Family& F : fams)
      for (const VNode& v : F.vn)
        if (v.leaf != 1)
          for (int id : v.mem) absorbed.insert(id);
    for (const Spine& S : spines)
      for (int c : S.chain) absorbed.insert(c);
    std::vector<char> needed(nn, 0);
    std::vector<int> work;
    auto need = [&](int id) {
      if (!needed[id]) {
        needed[id] = 1;
        work.push_back(id);
      }
    };
    auto scalar_reads = [&](int id) {  // operands the scalar form of statement `id` reads
      auto sp = rr_spine_of.find(id);
      if (sp != rr_spine_of.end()) {
        for (int t : spines[sp->second].scalar_terms) need(t);
        return;
      }
      const Node& n = P.nodes[id];
      if (n.kind == K_LOOKUP && tab_off.count(id)) {
        need(n.a);
        return;  // its table is filled separately
      }
      operands(id, ops);
      for (int o : ops) need(o);
    };
    for (const std::vector<int>* l : {&P.inv_fwd, &P.inv_bwd})
      for (int id : *l)
        if (!absorbed.count(id)) scalar_reads(id);
    for (const TargetInfo& T : P.targets) {
      for (int id : T.row_fwd) scalar_reads(id);
      for (int id : T.row_bwd) scalar_reads(id);
      for (const AccStmt& a : T.row_acc) need(a.node);
      for (const ScatterStmt& sc : T.row_scatter) need(sc.node), need(sc.index_node);
    }
    for (const AccStmt& a : P.inv_acc) need(a.node);
    for (uint32_t i = 0; i < P.n_params; i++)
      if (!rr_family_grad[i]) need(P.grad_nodes[i]);
    for (int id : tab_fill)
      if (!rr_family_tables.count(id)) {
        const Node& n = P.nodes[id];
        for (int k = 0; k < n.c; k++) need(P.lookup_refs[n.b + k]);
      }
    for (const Family& F : fams)
      for (int u : F.uniforms) need(u);
    while (!work.empty()) {
      const int id = work.back();
      work.pop_back();
      if (absorbed.count(id)) scalar_reads(id);  // an absorbed statement that has to stay: so do its operands
    }
    for (int id : absorbed)
      if (!needed[id]) rr_elim.insert(id);
    // a fold whose interior sums have to stay is not re-rolled after all (its families still are: they then only feed dead sums,
    // so drop them too)
    for (size_t si = 0; si < spines.size(); si++) {
      bool broken = false;
      for (int c : spines[si].chain) broken = broken || needed[c];
      if (broken) {
        fams.clear();
        spines.clear();
        rr_elim.clear();
        rr_spine_of.clear();
        rr_family_tables.clear();
        rr_family_grad.assign(P.n_params, 0);
        rr_n_sums = 0;
        return;
      }
    }
    rr_max_round_sums = rr_n_sums;
  }

  // one family = one loop; uniform operands keep their scalar names, vnodes are named after their first member
  void rr_emit_family(const Family& F, const char* ind) {
    os << ind << "for (int k = lane; k < " << F.L << "; k += RN_G) {\n";
    const std::string in2 = std::string(ind) + "  ";
    name_override.clear();
    for (size_t i = 0; i < F.vn.size(); i++) {
      const VNode& v = F.vn[i];
      if (v.leaf) {
        name_override[v.mem[0]] = std::string(v.leaf == 1 ? "q[" : "scr[") + std::to_string(v.base) + " + " + std::to_string(v.stride) + " * k]";
      } else {
        name_override[v.mem[0]] = "w" + std::to_string(i);
        stmt(v.mem[0], in2.c_str());
      }
    }
    for (const FamOut& o : F.outs) {
      const std::string x = val(F.vn[o.vn].mem[0]);
      if (o.kind == 0) os << in2 << "scr[" << o.base << " + k] = " << x << ";\n";
      if (o.kind == 1) os << in2 << "grad[" << o.base << " + k] = " << x << ";\n";
      if (o.kind == 2) os << in2 << "s" << o.sum << " += " << x << ";\n";
    }
    name_override.clear();
    os << ind << "}\n";
  }

  // the invariant statements of one section with the families in their place: scalar statements as soon as their operands
  // exist, then every family whose uniform operands exist, then the group-wide reduction of that round's sums; repeat
  void rr_emit_section(const std::vector<int>& list, bool bwd, std::set<int>& avail, std::set<int>& sums_ready) {
    const int K = std::max(1, opt.wpc_k);
    std::vector<int> pending;
    for (int id : list)
      if (!rr_elim.count(id)) pending.push_back(id);
    std::vector<int> ops;
    auto ready = [&](int id) {
      const Node& n = P.nodes[id];
      return n.kind == K_CONST || n.kind == K_INPUT || avail.count(id) > 0;
    };
    for (int guard = 0; guard < 64; guard++) {
      std::vector<int> blocked;
      for (int id : pending) {
        bool ok = true;
        auto sp = rr_spine_of.find(id);
        if (sp != rr_spine_of.end()) {
          const Spine& S = spines[sp->second];
          for (int t : S.scalar_terms) ok = ok && ready(t);
          for (int sidx : S.sums) ok = ok && sums_ready.count(sidx) > 0;
          if (ok) {
            os << "  const double " << val(id) << " = ";
            std::string e;
            for (int t : S.scalar_terms) e = e.empty() ? val(t) : "(" + e + " + " + val(t) + ")";
            for (int sidx : S.sums) e = e.empty() ? "s" + std::to_string(sidx) : "(" + e + " + s" + std::to_string(sidx) + ")";
            os << e << ";\n";
          }
        } else {
          operands(id, ops);
          if (P.nodes[id].kind == K_LOOKUP && tab_off.count(id)) ops.resize(1);
          for (int o : ops) ok = ok && ready(o);
          if (ok) stmt(id, "  ");
        }
        if (ok)
          avail.insert(id);
        else
          blocked.push_back(id);
      }
      pending.swap(blocked);
      std::vector<int> round_sums;
      bool any_family = false;
      for (Family& F : fams) {
        if (F.done || F.bwd != bwd) continue;
        bool ok = true;
        for (int u : F.uniforms) ok = ok && ready(u);
        if (!ok) continue;
        for (const FamOut& o : F.outs)
          if (o.kind == 2) {
            os << "  double s" << o.sum << " = 0.0;\n";
            round_sums.push_back(o.sum);
          }
        rr_emit_family(F, "  ");
        F.done = true;
        any_family = true;
      }
      if (!round_sums.empty()) {
        const int m = (int)round_sums.size();
        for (int sidx : round_sums) os << "  s" << sidx << " = rn_warp_sum(s" << sidx << ");\n";
        if (K > 1) {
          os << "  {\n    double* red = scr + " << red_off << ";\n    const int wg = lane >> 5;\n    RN_SYNC();\n    if ((lane & 31) == 0) {\n";
          for (int j = 0; j < m; j++) os << "      red[wg * " << m << " + " << j << "] = s" << round_sums[j] << ";\n";
          os << "    }\n    RN_SYNC();\n";
          for (int j = 0; j < m; j++) {
            os << "    s" << round_sums[j] << " = red[" << j << "]";
            for (int k = 1; k < K; k++) os << " + red[" << k * m + j << "]";
            os << ";\n";
          }
          os << "  }\n";
        }
        for (int sidx : round_sums) sums_ready.insert(sidx);
      }
      if (pending.empty() && !any_family) break;
      if (!any_family && round_sums.empty() && !pending.empty()) {
        // nothing moved: should not happen (the fixpoint in rr_plan keeps every operand of a scalar statement); emit the rest
        // in order so that a compile error, not a wrong value, is the symptom
        for (int id : pending) stmt(id, "  ");
        pending.clear();
        break;
      }
    }
  }

  void density_wpc() {
    wpc = true;
    // which accumulator slots live in shared memory (targets of a scatter) and which in registers
    smem_slot.assign(P.n_slots, -1);
    for (const TargetInfo& T : P.targets)
      for (const ScatterStmt& sc : T.row_scatter)
        for (int k = 0; k < sc.len; k++)
          if (smem_slot[sc.slot_base + k] < 0) smem_slot[sc.slot_base + k] = n_smem_acc++;
    std::map<std::vector<int>, int> tab_by_refs;  // Lookups over the same entries (the 8 observe splits) share a table
    for (const TargetInfo& T : P.targets)
      for (int id : T.row_fwd)
        if (is_big_table(P.nodes[id])) {
          const Node& n = P.nodes[id];
          std::vector<int> refs(P.lookup_refs.begin() + n.b, P.lookup_refs.begin() + n.b + n.c);
          auto it = tab_by_refs.find(refs);
          if (it == tab_by_refs.end()) {
            it = tab_by_refs.emplace(refs, tab_doubles).first;
            tab_fill.push_back(id);
            tab_doubles += n.c;
          }
          tab_off[id] = it->second;
        }
    os << "// ---- emitted: log-density and gradient of the frozen DAG (" << (P.symbolic ? "symbolic" : "adjoint")
       << " gradient), warp-per-chain: rows across lanes ----\n";
    const int K = std::max(1, opt.wpc_k);
    // chain-batched DMMA plans (analysis always; code only with opt.mma)
    plans.assign(P.targets.size(), MmaPlan());
    mma_all_ok = K == 1;
    bool any_full = false;
    for (size_t t = 0; t < P.targets.size(); t++) {
      const TargetInfo& T = P.targets[t];
      if (!T.streamed() || T.n_rows / 32 == 0) continue;
      any_full = true;
      plans[t] = plan_mma(T, t);
      if (!plans[t].ok) mma_all_ok = false;
      mma_shared_doubles = std::max(mma_shared_doubles, MMA_WARPS * plans[t].region_doubles + mma_groups() * MMA_WARPS * 8 * plans[t].redw);
    }
    if (!any_full) mma_all_ok = false;
    if (!mma_all_ok) mma_shared_doubles = 0;
    const bool use_mma = opt.mma && mma_all_ok;
    int n_reg_acc = 0;
    for (int sl = 0; sl < P.n_slots; sl++)
      if (smem_slot[sl] < 0) n_reg_acc++;
    row_functions = !use_mma && n_reg_acc <= 8;
    rr_plan();
    // cross-warp reduction scratch of the chain's group (K warps): [warp][register accumulators..., err]; the sums of the
    // re-rolled families go through it too, before and after the row loops
    red_off = tab_doubles + n_smem_acc;
    red_doubles = K > 1 ? K * std::max(n_reg_acc + 1, rr_max_round_sums) : 0;
    mma_inv_off = tab_doubles + n_smem_acc + red_doubles;
    os << "#define RN_WPC_SCRATCH " << (tab_doubles + n_smem_acc + red_doubles + (use_mma ? (int)mma_inv.size() : 0)) << "\n";
    os << "#define RN_MMA_BARS " << (use_mma ? MMA_WARPS : 0) << "\n";
    os << "#define RN_WPC_RED_OFF " << red_off << "\n";
    os << "RN_DEVICE double rn_tab_lookup(const double* tab, int len, int low, double idx, int& err) {\n"
          "  const int k = rn_d2i(idx) - low;\n  const bool bad = (unsigned)k >= (unsigned)len;\n  err |= (int)bad;\n"
          "  const double v = tab[bad ? 0 : k];\n  return bad ? RN_NAN : v;\n}\n";
    os << "RN_DEVICE double rn_warp_sum(double x) {\n  RN_UNROLL\n  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);\n  return x;\n}\n";
    lookup_helpers();
    if (use_mma)
      for (size_t t = 0; t < P.targets.size(); t++)
        if (plans[t].ok)
          for (size_t di = 0; di < (plans[t].uniform ? 1 : plans[t].dots.size()); di++) mma_helper(P.targets[t], t, plans[t], di);
    os << "RN_DEVICE void rn_density(const double* q, double& dens, double* grad, double* scr, "
          "const double* RN_RESTRICT data, int& err_io, RnTma& tma) {\n";
    // the error flag in a register: through the reference it lived in local memory, one LDL / LOP3 / STL chain per lookup
    os << "  (void)data; (void)scr; (void)tma;\n  const int lane = (int)(threadIdx.x % RN_G);  // thread of the chain's group\n  (void)lane;\n"
       << "  int err = 0;\n";
    if (n_smem_acc) os << "  for (int k = lane; k < " << n_smem_acc << "; k += RN_G) scr[" << tab_doubles << " + k] = 0.0;\n";
    std::set<int> rr_avail, rr_sums_ready;
    if (fams.empty())
      for (int id : P.inv_fwd) stmt(id, "  ");
    else
      rr_emit_section(P.inv_fwd, false, rr_avail, rr_sums_ready);
    for (int id : tab_fill) {
      if (rr_family_tables.count(id)) continue;
      const Node& n = P.nodes[id];
      for (int k = 0; k < n.c; k++) os << "  scr[" << (tab_off.at(id) + k) << "] = " << val(P.lookup_refs[n.b + k]) << ";\n";
    }
    os << "  RN_SYNC();\n";
    for (int sl = 0; sl < P.n_slots; sl++)
      if (smem_slot[sl] < 0) os << "  double a" << sl << " = 0.0;\n";
    for (size_t t = 0; t < P.targets.size(); t++) {
      const TargetInfo& T = P.targets[t];
      os << "  // target " << t << (T.streamed() ? " (streamed, rows across the group's threads)" : " (data-free)") << "\n";
      if (T.streamed()) {
        const int pitch = opt.pitch(t);
        const unsigned long long base = (unsigned long long)opt.target_base[t], td = (unsigned long long)T.n_cols * pitch;
        const unsigned long long rows_per_tile = 32ull * K;  // a "super-tile": K consecutive 32-row tiles, one per warp
        const unsigned long long n_full = T.n_rows / rows_per_tile;
        os << "  {\n    long long row0 = lane;\n";
        if (use_mma && n_full > 0) {
          mma_block(T, t, plans[t], n_full);
        } else if (opt.tma_stages > 0 && n_full > 0) {
          // CTA lockstep over full tiles: tile t+S-1 in flight (one bulk copy) while all warps consume tile t from smem
          os << "    if (tma.on) {\n"
             << "      const unsigned n_full = " << n_full << "u, seq0 = tma.seq;\n"
             << "      const double* RN_RESTRICT src = data + " << base << "ULL;\n"
             << "      if (threadIdx.x == 0)\n"
             << "        for (unsigned p = 0; p + 1 < RN_TMA_STAGES && p < n_full; p++) rn_tma_load(tma, seq0 + p, src + (size_t)p * "
             << td * K << "ULL, " << td * K * 8 << "u);\n"
             << "      for (unsigned tile = 0; tile < n_full; tile++) {\n"
             << "        const unsigned seq = seq0 + tile;\n"
             << "        if (threadIdx.x == 0 && tile + (RN_TMA_STAGES - 1) < n_full)\n"
             << "          rn_tma_load(tma, seq + (RN_TMA_STAGES - 1), src + (size_t)(tile + (RN_TMA_STAGES - 1)) * " << td * K << "ULL, "
             << td * K * 8 << "u);\n"
             << "        rn_mbar_wait(tma.full + (seq % RN_TMA_STAGES), (seq / RN_TMA_STAGES) & 1u);\n"
             << "        const RnSA rp = rn_sa(tma.stage + (size_t)(seq % RN_TMA_STAGES) * RN_TMA_TILE_DOUBLES + (size_t)(lane >> 5) * " << td
             << " + (lane & 31));\n";
          row_body(
              T, "        ", [&](int k) { return "rn_lds_tile(rp, " + std::to_string(local_col(T, k) * pitch) + ")"; },
              [&](int slot) { return acc_ref(slot); }, true, tab_doubles);
          os << "        rn_cta_bar(tma.nthreads);\n"
             << "      }\n"
             << "      tma.seq = seq0 + n_full;\n"
             << "      row0 += " << n_full * rows_per_tile << "LL;\n"
             << "    }\n";
        }
        os << "    for (long long row = row0; row < " << (long long)T.n_rows << "LL; row += RN_G) {\n";
        os << "      const double* RN_RESTRICT rp = data + " << base << "ULL + (row >> 5) * " << td << "LL + (row & 31);\n";
        row_body(
            T, "      ", [&](int k) { return "RN_LDG(rp + " + std::to_string(local_col(T, k) * pitch) + ")"; },
            [&](int slot) { return acc_ref(slot); }, true, tab_doubles);
        os << "    }\n  }\n";
      } else {
        os << "  if (lane == 0) {\n";  // counted once by the reduction below
        for (const AccStmt& a : T.row_acc) os << "    " << acc_ref(a.slot) << " += " << val(a.node) << ";\n";
        os << "  }\n";
      }
    }
    for (int sl = 0; sl < P.n_slots; sl++)
      if (smem_slot[sl] < 0) os << "  a" << sl << " = rn_warp_sum(a" << sl << ");\n";
    os << "  err = (int)__reduce_or_sync(0xffffffffu, (unsigned)err);\n";
    if (K > 1) {
      // the K warps of the chain exchange their partial sums through shared memory; every thread adds them in the same
      // order, so all of them hold identical totals afterwards
      const int stride = n_reg_acc + 1;
      os << "  {\n    double* red = scr + " << red_off << ";\n    const int wg = lane >> 5;\n    if ((lane & 31) == 0) {\n";
      int idx = 0;
      for (int sl = 0; sl < P.n_slots; sl++)
        if (smem_slot[sl] < 0) os << "      red[wg * " << stride << " + " << idx++ << "] = a" << sl << ";\n";
      os << "      red[wg * " << stride << " + " << idx << "] = (double)err;\n    }\n    RN_SYNC();\n";
      idx = 0;
      for (int sl = 0; sl < P.n_slots; sl++)
        if (smem_slot[sl] < 0) {
          os << "    a" << sl << " = red[" << idx << "]";
          for (int k = 1; k < K; k++) os << " + red[" << k * stride + idx << "]";
          os << ";\n";
          idx++;
        }
      os << "    for (int k = 0; k < " << K << "; k++) err |= (int)red[k * " << stride << " + " << idx << "];\n  }\n";
    }
    os << "  RN_SYNC();\n";
    os << "  dens = a0;\n";
    if (P.symbolic) {
      for (uint32_t i = 0; i < P.n_params; i++) os << "  if (lane == 0) grad[" << i << "] = " << acc_ref(1 + (int)i) << ";\n";
    } else {
      if (fams.empty())
        for (int id : P.inv_bwd) stmt(id, "  ");
      else
        rr_emit_section(P.inv_bwd, true, rr_avail, rr_sums_ready);
      for (uint32_t i = 0; i < P.n_params; i++)
        if (fams.empty() || !rr_family_grad[i]) os << "  if (lane == 0) grad[" << i << "] = " << val(P.grad_nodes[i]) << ";\n";
    }
    os << "  err_io |= err;\n  RN_SYNC();\n}\n";
  }
};

}  // namespace

// vectors of n doubles in a chain's shared-memory slice (rn_sampler_wpc.cuh: rn_w_setup): q, p, gradient, [diagonal mass],
// [3 EHMC snapshots], [2 dense-mass work vectors]
static int wpc_vectors(const EmitOptions& opt) { return 3 + (opt.mass_max >= 1 ? 1 : 0) + (opt.enable_ehmc ? 3 : 0) + (opt.mass_max == 2 ? 2 : 0); }

std::string emit_density(const Program& P, const EmitOptions& opt) {
  Emitter E(P, opt);
  if (opt.backend == 1)
    E.density_wpc();
  else
    E.density_tpc();
  return E.os.str();
}

WpcSizes wpc_sizes(const Program& P, const EmitOptions& opt) {
  WpcSizes z;
  Emitter E(P, opt);
  E.density_wpc();
  // chain vectors (q, p, gradient, mass [+ EHMC snapshot]) [+ 2 scratch vectors of the dense mass matrix code] + density scratch
  z.scratch_doubles = E.tab_doubles + E.n_smem_acc + E.red_doubles + ((opt.mma && E.mma_all_ok) ? (int)E.mma_inv.size() : 0);
  z.per_warp_doubles = wpc_vectors(opt) * (int)P.n_params + z.scratch_doubles;
  for (const TargetInfo& T : P.targets)
    if (T.streamed() && T.n_rows >= 32ull * (uint64_t)std::max(1, opt.wpc_k))
      z.tile_doubles = std::max(z.tile_doubles, (int)T.n_cols * opt.pitch((size_t)(&T - &P.targets[0])) * std::max(1, opt.wpc_k));
  z.mma_ok = E.mma_all_ok;
  z.mma_shared_doubles = E.mma_shared_doubles;
  z.row_functions = E.row_functions;
  return z;
}

std::vector<int> default_pitches(const Program& P) {
  std::vector<int> p(P.targets.size(), 32);
  for (size_t t = 0; t < P.targets.size(); t++)
    if (P.targets[t].streamed() && !P.targets[t].dots.empty() && P.targets[t].n_rows >= 64) p[t] = 36;
  return p;
}

std::string emit_optimizer_source(const Program& P, const EmitOptions& opt, int history) {
  std::ostringstream os;
  os << "// generated by rainier_b200 (CUDA source emitter, optimizer flavour) -- do not edit\n";
  os << "#define RN_N " << P.n_params << "\n";
  os << "#define RN_NSLOTS " << P.n_slots << "\n";
  os << "#define RN_BACKEND " << (opt.backend == 1 ? 1 : 0) << "\n";
  os << "#define RN_LBFGS_M " << history << "\n";
  if (opt.expect_slice_doubles > 0) os << "#define RN_OPT_EXPECT_SMEM " << opt.expect_slice_doubles << "\n";
  if (opt.fast_math) os << "#define RN_FAST_MATH 1\n";
  EmitOptions eo = opt;
  if (opt.backend == 1) {  // K warps per start, independent per-warp row loads (no CTA-shared tiles: starts diverge)
    eo.wpc_k = std::max(1, opt.wpc_k);
    eo.tma_stages = 0;
    eo.enable_ehmc = false;
    os << "#define RN_WPC_K " << eo.wpc_k << "\n#define RN_TMA_STAGES 0\n#define RN_TMA_TILE_DOUBLES 0\n";
  } else {
    eo.backend = 0;
  }
  os << kPreludeSource << "\n";
  os << emit_density(P, eo) << "\n" << kOptimizerSource << "\n";
  return os.str();
}

std::string emit_function_source(const Program& P, const EmitOptions& opt) {
  std::ostringstream os;
  os << "// generated by rainier_b200 (CUDA source emitter, function flavour) -- do not edit\n";
  os << "#define RN_N " << P.n_params << "\n";
  os << "#define RN_NQ " << std::max<uint32_t>(1, P.n_params) << "\n";
  os << "#define RN_M " << P.fn_outputs.size() << "\n";
  os << "#define RN_BACKEND 0\n";
  if (opt.fast_math) os << "#define RN_FAST_MATH 1\n";
  os << kPreludeSource << "\n";
  Emitter E(P, opt);
  E.function_tpc();
  os << E.os.str() << "\n" << kFunctionSource << "\n";
  return os.str();
}

std::string emit_source(const Program& P, const EmitOptions& opt) {
  std::ostringstream os;
  os << "// generated by rainier_b200 (CUDA source emitter) -- do not edit\n";
  os << "#define RN_N " << P.n_params << "\n";
  os << "#define RN_NSLOTS " << P.n_slots << "\n";
  os << "#define RN_BACKEND " << opt.backend << "\n";
  os << "#define RN_MASS_MAX " << opt.mass_max << "\n";
  os << "#define RN_ENABLE_EHMC " << (opt.enable_ehmc ? 1 : 0) << "\n";
  if (opt.fast_math) os << "#define RN_FAST_MATH 1\n";
  if (opt.backend == 1) {
    os << "#define RN_WPC_K " << std::max(1, opt.wpc_k) << "\n";
    os << "#define RN_TMA_STAGES " << opt.tma_stages << "\n";
    {
      const WpcSizes z = wpc_sizes(P, opt);
      os << "#define RN_TMA_TILE_DOUBLES " << ((opt.mma && z.mma_ok) ? z.mma_shared_doubles : z.tile_doubles) << "\n";
    }
  }
  os << kPreludeSource << "\n";
  if (opt.backend == 1)  // (RN_WPC_SCRATCH is defined by the emitted density; macros expand where they are used)
    os << "#define RN_WPC_SMEM_DOUBLES (" << wpc_vectors(opt) << " * RN_N + RN_WPC_SCRATCH)\n";
  os << emit_density(P, opt) << "\n";
  if (opt.backend == 1) {
    os << kSamplerWpcSource << "\n";
  } else {
    os << kSamplerSource << "\n";
  }
  return os.str();
}

}  // namespace rn
