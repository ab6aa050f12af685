// rn_emit.hpp -- CUDA source emitter: Program -> one self-contained translation unit (prelude + emitted
// rn_density() + hand-written sampler kernels).  Replaces the reference's JVM bytecode emitter
// (rainier-compute/.../ir/CompiledFunction.scala:42-120 and the *Generator classes).
#pragma once
#include <string>

#include "rn_graph.hpp"

namespace rn {

struct EmitOptions {
  int backend = 0;        // 0 = thread per chain, 1 = warp per chain (rows across lanes)
  bool fast_math = false; // strength-reduce constant powers beyond what Math.pow itself special-cases
  int mass_max = 0;       // 0 identity only, 1 + diagonal, 2 + dense
  bool enable_ehmc = false;
  int tma_stages = 0;     // warp per chain: shared-memory stages of the CTA-shared data-tile pipeline (0 = off)
  int wpc_k = 1;          // warp per chain: warps owning one chain (1, 2, 4 or 8; > 1 for chains with a large state)
  std::vector<uint64_t> target_base;  // per target: element offset of its tile-major [tile][column][pitch] block in the data buffer
  std::vector<int> target_pitch;      // per target: doubles between consecutive columns of a tile (32 rows + padding; empty = 32).
                                      // 36 where the chain-batched DMMA path may run: X^T fragments are then bank-conflict free
  bool mma = false;       // warp per chain: chain-batched fp64 tensor-core contraction of the row bodies' dot products (see
                          // Emitter::mma_block); needs full CTAs of mma_chains chains (= warps, wpc_k == 1)
  int expect_slice_doubles = 0;  // optimizer: the launcher's shared-memory doubles per start (checked against the kernel's own layout at compile time)
  int interleave = 8;     // independent dataflow components of a row body (unrolled observations) emitted round-robin at a time
  int mma_chains = 8;     // 8 or 16: chains (warps) per CTA on that path -- 16 = two groups of 8 chains whose warps pair up on
                          // a dot's column block (twice the warps per SM for the same shared memory)
  int pitch(size_t t) const { return t < target_pitch.size() && target_pitch[t] > 0 ? target_pitch[t] : 32; }
};
// pitch a model should be packed with: 36 for streamed targets whose row body holds parameter x column dot products
std::vector<int> default_pitches(const Program& P);

// the generated rn_density() only
std::string emit_density(const Program& P, const EmitOptions& opt);
// full translation unit
std::string emit_source(const Program& P, const EmitOptions& opt);
// function flavour (Program from build_function): prelude + emitted rn_function() + rn_function.cuh (rn_k_eval); only
// opt.fast_math is read
std::string emit_function_source(const Program& P, const EmitOptions& opt);
// optimizer flavour: prelude + emitted thread-per-chain rn_density() + rn_optimizer.cuh (rn_k_lbfgs, `history` = the m of
// new LBFGS(x, m, eps)); reads opt.fast_math and opt.target_base
std::string emit_optimizer_source(const Program& P, const EmitOptions& opt, int history);
// shared-memory needs of the warp-per-chain kernels: doubles per warp (chain vectors + density scratch) and doubles of
// the largest data tile (n_cols * 32 over the streamed targets; 0 when nothing is streamed)
struct WpcSizes {
  int per_warp_doubles = 0;  // per CHAIN (its wpc_k warps share the slice): the sampler's vectors + scratch_doubles
  int scratch_doubles = 0;   // the emitted density's part of it (RN_WPC_SCRATCH): tables, scatter slots, reduction scratch
  int tile_doubles = 0;
  bool mma_ok = false;       // every streamed target with full tiles can take the chain-batched DMMA path
  int mma_shared_doubles = 0;  // CTA-shared doubles of that path: 8 per-warp column-block regions + the reduction scratch
  bool row_functions = false;  // the row bodies use the branch-free rn_row_* functions instead of CUDA's libm (rule: rn_emit.cpp)
};
WpcSizes wpc_sizes(const Program& P, const EmitOptions& opt);

}  // namespace rn
