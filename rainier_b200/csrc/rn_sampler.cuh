// rn_sampler.cuh -- hand-written batched HMC/EHMC integrator, appended after the emitted rn_density().
//
// One CUDA thread owns one chain (RN_BACKEND == 0, "thread per chain") and runs whole iterations --
// momentum draw, leapfrog steps, Metropolis test, adaptation, sample write -- inside one launch; chain state
// lives in registers across the L steps of an iteration and in chain-fastest (coalesced) SoA arrays between
// iterations.  Control flow follows the reference line by line so that chain c reproduces a single-chain
// reference run seeded with ScalaRNG(seeds[c]):
//   LeapFrog      rainier-sampler/src/main/scala/com/stripe/rainier/sampler/LeapFrog.scala:3-252
//   HMCSampler    .../sampler/HMC.scala:3-24         EHMCSampler  .../sampler/EHMC.scala:3-62
//   DualAvgTuner  .../sampler/DualAvg.scala:3-90     mass tuners  .../sampler/MassMatrix.scala:120-181
//   estimators    .../sampler/MassMatrixEstimator.scala:9-112
//   Driver        .../sampler/Driver.scala:7-119     Stats/RingBuffer .../sampler/Stats.scala:3-59
// The reference re-evaluates the density in every fullPs() at the position the previous update already
// evaluated (LeapFrog.scala:168-176 vs :161-166); update() is a pure function of q, so this kernel keeps the
// gradient of the last evaluation instead (l+1 evaluations per takeSteps(l) instead of 2l+1) while still
// counting gradientEvaluations the reference's way.
//
// Compile-time switches (set by the emitter): RN_N, RN_NSLOTS, RN_MASS_MAX (0 identity only, 1 +diagonal,
// 2 +dense), RN_ENABLE_EHMC.
#ifndef RN_SAMPLER_CUH
#define RN_SAMPLER_CUH

// struct RnArgs: see rn_args.h (shared verbatim with the host runtime)

#define RN_LN2 0.6931471805599453
#define RN_AT(ptr, field, c) (ptr)[(size_t)(field) * (size_t)A.chains + (size_t)(c)]

// ---- this thread's COLD state lives in shared memory -----------------------------------------------------------
// Everything a chain touches once per iteration is kept out of registers: the Stats counters, the RNG state, the energies
// carried from startIteration to finishIteration, the diagonal mass matrix and the scratch of the normal draws sit in
// dynamic shared memory as [slot][blockDim.x] -- conflict-free, one LDS/STS per access -- so that p, q, the gradient and
// the density's temporaries fit 128 registers without spilling (round 1: 80 bytes of spill traffic in the leapfrog
// loop).  Measured on B200 (profiles/r2_sweep_iter_v2_variants.jsonl): the kernel does NOT respond to occupancy (96 or
// 80 registers per thread = 20 / 24 warps per SM are no faster than 128 = 16 warps: what the extra warps hide, the
// tighter register allocation loses in instruction-level parallelism) but it does respond to CODE SIZE and instruction
// count (stall `no_instruction` 12 % with the second pass of the normal draws unrolled, 3.68 -> 3.41 ms as a loop), which
// is why the hot loops stay loops and the fdlibm functions run as one branch-free common path (rn_prelude.cuh).
// (Host emulation: blockDim.x == 1, a thread_local array.)
#if RN_MASS_MAX >= 1
#define RN_TS_NMASS RN_N
#else
#define RN_TS_NMASS 0
#endif
#if RN_ENABLE_EHMC
#define RN_TS_NSNAP RN_N
#else
#define RN_TS_NSNAP 0
#endif
#define RN_TS_P 0                                        /* momentum, RN_N + 1 slots (+1: scratch of the polar method) */
#define RN_TS_MASS (RN_N + 1)                            /* diagonal mass matrix (variances) */
#define RN_TS_SNAP (RN_TS_MASS + RN_TS_NMASS)            /* momentum of the EHMC snapshot */
#define RN_TS_STAT (RN_TS_SNAP + RN_TS_NSNAP)            /* e_mean, e_raw, trans2, grads (i64), steps (i64) */
#define RN_TS_HOT (RN_TS_STAT + 5)                       /* rng.seed (i64), rng.nng, prevH, startH: parked across the leapfrog */
#define RN_TS_DOUBLES (RN_TS_HOT + 4)
#define RN_TS_INTS 10                                    /* iters, accepted, e_n, ring_i[3], ring_full[3], rng.have */
struct RnTs {
  double* d;
  int* i;
  unsigned bs;
};
#ifdef RN_HOST_EMULATION
static thread_local double rn_ts_mem_d[RN_TS_DOUBLES];
static thread_local int rn_ts_mem_i[RN_TS_INTS];
RN_DEVICE RnTs rn_ts_get() { return RnTs{rn_ts_mem_d, rn_ts_mem_i, 1u}; }
#define RN_STCS(ptr, v) (*(ptr) = (v))
#else
extern __shared__ double rn_ts_mem[];
RN_DEVICE RnTs rn_ts_get() {
  RnTs T;
#ifdef RN_BLOCK_DIM
  T.bs = RN_BLOCK_DIM;  // the runtime compiled this module for the block size it launches with: slot offsets become immediates
#else
  T.bs = blockDim.x;
#endif
  T.d = rn_ts_mem + threadIdx.x;
  T.i = (int*)(rn_ts_mem + (size_t)RN_TS_DOUBLES * blockDim.x) + threadIdx.x;
  return T;
}
#define RN_STCS(ptr, v) __stcs((ptr), (v))  /* streaming store: samples / rings / trace must not evict the L2-resident state */
#endif
#define RN_TSD(slot) T.d[(unsigned)(slot) * T.bs]
#define RN_TSI(slot) T.i[(unsigned)(slot) * T.bs]
#define RN_Z(i) RN_TSD(RN_TS_P + (i)) /* scratch of the normal draws */
#define RN_P(i) s.p[i] /* momentum in registers: 3.25 ms vs 3.41 ms per launch at the headline size with it in shared memory */
#define RN_MASSD(i) RN_TSD(RN_TS_MASS + (i))
#define RN_ST_E_MEAN RN_TSD(RN_TS_STAT + 0)
#define RN_ST_E_RAW RN_TSD(RN_TS_STAT + 1)
#define RN_ST_TRANS2 RN_TSD(RN_TS_STAT + 2)
#define RN_ST_GRADS RN_TSD(RN_TS_STAT + 3) /* rn_i64 bit pattern */
#define RN_ST_STEPS RN_TSD(RN_TS_STAT + 4) /* rn_i64 bit pattern */
#define RN_ST_ITERS RN_TSI(0)
#define RN_ST_ACCEPTED RN_TSI(1)
#define RN_ST_E_N RN_TSI(2)
#define RN_ST_RING_I(r) RN_TSI(3 + (r))
#define RN_ST_RING_FULL(r) RN_TSI(6 + (r))
#define RN_TS_PREV_H RN_TSD(RN_TS_HOT + 2)
#define RN_TS_START_H RN_TSD(RN_TS_HOT + 3)

// counters of the iteration in flight (registers; folded into the shared-memory Stats once per iteration)
struct RnIt {
  int grads, steps, err;
};

// the RNG is idle while the trajectory is integrated: its state waits in shared memory
RN_DEVICE RnRng rn_rng_unpark(const RnTs& T) {
  RnRng r;
  r.seed = rn_d2ll(RN_TSD(RN_TS_HOT + 0));
  r.nng = RN_TSD(RN_TS_HOT + 1);
  r.have = RN_TSI(9);
  return r;
}
RN_DEVICE void rn_rng_park(const RnTs& T, const RnRng& r) {
  RN_TSD(RN_TS_HOT + 0) = rn_ll2d(r.seed);
  RN_TSD(RN_TS_HOT + 1) = r.nng;
  RN_TSI(9) = r.have;
}

RN_DEVICE void rn_ring_add(const RnArgs& A, int c, const RnTs& T, int which, double value) {  // Stats.scala:24-30
  int i = RN_ST_RING_I(which) + 1;  // i <= stats_window: `i % size` is a compare, not a division
  if (i == A.stats_window) {
    RN_ST_RING_FULL(which) = 1;
    i = 0;
  }
  RN_ST_RING_I(which) = i;
  RN_STCS(&RN_AT(A.st_rings, which * A.stats_window + i, c), value);
}

struct RnPQ {  // pqBuf's q, p and potential + the gradient at pqBuf.q
  double q[RN_N], g[RN_N];
  double U;
  double p[RN_N];
};

// velocity_i = (M^-1 p)_i  (LeapFrog.scala:205-219)
RN_DEVICE double rn_velocity_i(const RnArgs& A, int c, const RnTs& T, const RnPQ& s, int kind, int i) {
  (void)s;
  (void)T;
  (void)A;
  (void)c;
#if RN_MASS_MAX >= 2
  if (kind == 2) {  // DenseMassMatrix.squareMultiply, MassMatrix.scala:35-51
    double y = 0.0;
    for (int j = 0; j < RN_N; j++) y += RN_P(j) * RN_AT(A.mass, i * RN_N + j, c);
    return y;
  }
#endif
#if RN_MASS_MAX >= 1
  if (kind == 1) return RN_P(i) * RN_MASSD(i);
#endif
  (void)kind;
  return RN_P(i);
}

// energy = potential + dot(velocity, p)/2  (LeapFrog.scala:134-139,221-231)
RN_DEVICE double rn_energy(const RnArgs& A, int c, const RnTs& T, const RnPQ& s, int kind, double U) {
  double k = 0.0;
#if RN_MASS_MAX >= 2
  if (kind == 2) {
    for (int i = 0; i < RN_N; i++) k += (rn_velocity_i(A, c, T, s, 2, i) * RN_P(i));
    return U + k / 2.0;
  }
#endif
  RN_UNROLL
  for (int i = 0; i < RN_N; i++) k += (rn_velocity_i(A, c, T, s, kind, i) * RN_P(i));
  return U + k / 2.0;
}

RN_DEVICE double rn_log_accept(double deltaH) {  // LeapFrog.scala:141-145
  if (deltaH != deltaH) return -RN_INF;
  return rn_jmin0(-deltaH);
}


RN_DEVICE void rn_update(const RnArgs& A, RnPQ& s, RnIt& S) {  // copyQsAndUpdateDensity + potential
  double dens;
  rn_density(s.q, dens, s.g, A.data, S.err);
  s.U = dens * -1;
  S.grads += 1;
}
RN_DEVICE void rn_full_ps(const RnTs& T, RnPQ& s, double stepSize, RnIt& S) {
  (void)T;  // LeapFrog.scala:168-176 (gradient reused)
  S.grads += 1;
  RN_UNROLL
  for (int i = 0; i < RN_N; i++) RN_P(i) += stepSize * s.g[i];
}
RN_DEVICE void rn_new_qs(const RnArgs& A, int c, const RnTs& T, int kind, RnPQ& s, double stepSize) {  // :147-154
#if RN_MASS_MAX >= 2
  if (kind == 2) {
    for (int i = 0; i < RN_N; i++) s.q[i] += (stepSize * rn_velocity_i(A, c, T, s, 2, i));
    return;
  }
#endif
  RN_UNROLL
  for (int i = 0; i < RN_N; i++) s.q[i] += (stepSize * rn_velocity_i(A, c, T, s, kind, i));
}
// initialHalfThenFullStep + (l-1) twoFullSteps + finalHalfStep, LeapFrog.scala:24-33,156-191.
// `g` must hold the gradient at s.q on entry (true for params and for every state this kernel produces).
RN_DEVICE void rn_leapfrog(const RnArgs& A, int c, const RnTs& T, int kind, RnPQ& s, int l, double stepSize, RnIt& S) {
  // (one rn_update call site: the emitted density is inlined exactly once per use of rn_leapfrog)
  rn_full_ps(T, s, stepSize / 2.0, S);
  for (int i = 0;;) {
    rn_new_qs(A, c, T, kind, s, stepSize);
    rn_update(A, s, S);
    if (++i >= l) break;
    rn_full_ps(T, s, stepSize, S);
  }
  rn_full_ps(T, s, stepSize / 2.0, S);
}
RN_DEVICE void rn_take_steps(const RnArgs& A, int c, const RnTs& T, int kind, RnPQ& s, int l, double stepSize, RnIt& S) {
  rn_ring_add(A, c, T, 0, stepSize);  // stats.stepSizes.add, LeapFrog.scala:25
  rn_leapfrog(A, c, T, kind, s, l, stepSize, S);
  S.steps += l;
}

// RN_N standard normals into RN_P(0..RN_N-1), consuming java.util.Random exactly like RN_N calls of nextGaussian
// (RNG.scala:23-25: cached second variate first, then polar pairs).  The rejection loop of the polar method diverges
// inside a warp, so it is kept as small as possible: ONE flat loop over all pairs that only draws (v1, v2) and parks
// the accepted ones in the slots their variates will occupy (a lane that is done with pair k goes on to pair k+1 while
// its neighbours retry; a warp then runs max-over-lanes of the TOTAL number of attempts instead of the sum over pairs
// of the per-pair maxima), and a second, convergent pass applies sqrt(-2 log(s)/s).  s is recomputed there from the
// parked v1, v2 by the same two products and one sum -> the same bits.
RN_DEVICE void rn_draw_normals(const RnTs& T, RnRng& rng) {
  int i0 = 0;
  if (rng.have) {
    rng.have = 0;
    RN_Z(0) = rng.nng;
    i0 = 1;
  }
  const int npairs = (RN_N - i0 + 1) / 2;  // the last pair's second variate may be left over (-> rng.nng); slot RN_N is scratch
  // two attempts per trip (see rn_polar_attempt2); the second one is consumed only if it is needed: 2.488 -> 2.467 ms per launch
  // at the headline size (profiles/r2_sweep_iter_v6_polar2_merged.jsonl)
  for (int k = 0; k < npairs;) {
    double a1, a2, b1, b2;
    rn_i64 seed4, seed8;
    rn_polar_attempt2(rng, a1, a2, b1, b2, seed4, seed8);
    const double sa = a1 * a1 + a2 * a2, sb = b1 * b1 + b2 * b2;
    const bool oka = !(sa >= 1 || sa == 0);
    const int kb = k + (oka ? 1 : 0);
    const bool needb = kb < npairs;
    const bool okb = needb && !(sb >= 1 || sb == 0);
    if (oka) {
      RN_Z(i0 + 2 * k) = a1;
      RN_Z(i0 + 2 * k + 1) = a2;
    }
    if (okb) {
      RN_Z(i0 + 2 * kb) = b1;
      RN_Z(i0 + 2 * kb + 1) = b2;
    }
    rng.seed = needb ? seed8 : seed4;
    k = kb + (okb ? 1 : 0);
  }
  // the second pass kept as a loop (the kernel is sensitive to code size: 3.41 vs 3.68 ms fully unrolled, round 2), two pairs per
  // trip: with the check-free division / square root and the one-branch log the two chains of a trip overlap (2.505 -> 2.482 ms;
  // a hand-paired form through rn_strict_log_try, sharing one fallback branch, was slower: 2.554 --
  // profiles/r2_sweep_iter_v4_nocheck_div_spec_kconst.jsonl)
#pragma unroll 2
  for (int k = 0; k < npairs; k++) {
    const int i = i0 + 2 * k;
    const double v1 = RN_Z(i), v2 = RN_Z(i + 1);
    const double s = v1 * v1 + v2 * v2;
    const double multiplier = rn_polar_multiplier(s);
    RN_Z(i) = v1 * multiplier;
    if (i + 1 < RN_N) {
      RN_Z(i + 1) = v2 * multiplier;
    } else {
      rng.nng = v2 * multiplier;
      rng.have = 1;
    }
  }
}

// momentum draw, LeapFrog.scala:233-255  (result in RN_P)
RN_DEVICE void rn_initialize_ps(const RnArgs& A, int c, const RnTs& T, RnPQ& s, int kind, RnRng& rng) {
  (void)A;
  (void)c;
  (void)kind;
  (void)s;
  rn_draw_normals(T, rng);  // buf(i) = rng.standardNormal
  RN_UNROLL
  for (int i = 0; i < RN_N; i++) s.p[i] = RN_Z(i);
#if RN_MASS_MAX >= 2
  if (kind == 2) {  // DenseMassMatrix.upperTriangularSolve, MassMatrix.scala:55-72; in place: slot i holds z_i until p_i
    int i = RN_N - 1;  // replaces it, and p_i only reads z_i and the p_j, j > i, already in place
    int m = ((i + 1) * (i + 2)) / 2 - 1;
    while (i >= 0) {
      int j = RN_N - 1;
      double dot = 0.0;
      while (j > i) {
        dot += RN_Z(j) * RN_AT(A.chol, m, c);
        j -= 1;
        m -= 1;
      }
      RN_Z(i) = (RN_Z(i) - dot) / RN_AT(A.chol, m, c);
      i -= 1;
      m -= 1;
    }
    for (int k = 0; k < RN_N; k++) s.p[k] = RN_Z(k);
    return;
  }
#endif
#if RN_MASS_MAX >= 1
  if (kind == 1) {
    RN_UNROLL
    for (int i = 0; i < RN_N; i++) RN_P(i) = RN_P(i) / sqrt(RN_MASSD(i));  // buf(i) / stdDevs(i), stdDevs = sqrt(elements)
    return;
  }
#endif
}

RN_DEVICE void rn_load_mass(const RnArgs& A, int c, const RnTs& T, int kind) {
  (void)A;
  (void)c;
  (void)T;
  (void)kind;
#if RN_MASS_MAX >= 1
  if (kind == 1) {
    RN_UNROLL
    for (int i = 0; i < RN_N; i++) RN_MASSD(i) = RN_AT(A.mass, i, c);
  }
#endif
}

RN_DEVICE void rn_load_stats(const RnArgs& A, int c, const RnTs& T) {
  RN_ST_GRADS = rn_ll2d(A.st_grads[c]);
  RN_ST_STEPS = rn_ll2d(A.st_steps[c]);
  RN_ST_ITERS = A.st_iters[c];
  RN_ST_ACCEPTED = A.st_accepted[c];
  RN_ST_E_MEAN = RN_AT(A.st_energy, 0, c);
  RN_ST_E_RAW = RN_AT(A.st_energy, 1, c);
  RN_ST_TRANS2 = RN_AT(A.st_energy, 2, c);
  RN_ST_E_N = A.st_energy_n[c];
  for (int r = 0; r < 3; r++) {
    RN_ST_RING_I(r) = RN_AT(A.st_ring_i, r, c);
    RN_ST_RING_FULL(r) = RN_AT(A.st_ring_full, r, c);
  }
}
RN_DEVICE void rn_store_stats(const RnArgs& A, int c, const RnTs& T, int err) {
  A.st_grads[c] = rn_d2ll(RN_ST_GRADS);
  A.st_steps[c] = rn_d2ll(RN_ST_STEPS);
  A.st_iters[c] = RN_ST_ITERS;
  A.st_accepted[c] = RN_ST_ACCEPTED;
  if (err) A.st_err[c] |= err;
  RN_AT(A.st_energy, 0, c) = RN_ST_E_MEAN;
  RN_AT(A.st_energy, 1, c) = RN_ST_E_RAW;
  RN_AT(A.st_energy, 2, c) = RN_ST_TRANS2;
  A.st_energy_n[c] = RN_ST_E_N;
  for (int r = 0; r < 3; r++) {
    RN_AT(A.st_ring_i, r, c) = RN_ST_RING_I(r);
    RN_AT(A.st_ring_full, r, c) = RN_ST_RING_FULL(r);
  }
}
// fold the counters of the finished leapfrog calls into the shared-memory Stats
RN_DEVICE void rn_fold(const RnTs& T, RnIt& S) {
  RN_ST_GRADS = rn_ll2d(rn_d2ll(RN_ST_GRADS) + (rn_i64)S.grads);
  RN_ST_STEPS = rn_ll2d(rn_d2ll(RN_ST_STEPS) + (rn_i64)S.steps);
  S.grads = 0;
  S.steps = 0;
}

// =============================================================================================================
// rn_k_init: LeapFrog.initialize(IdentityMassMatrix) (Driver.scala:22) + stepSizeTuner.initialize (Driver.scala:60)
// =============================================================================================================
RN_GLOBAL void rn_k_init(const RnArgs A) {
  const int c = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (c >= A.chains) return;
  const RnTs T = rn_ts_get();
  RnRng rng;
  rng.seed = A.rng_seed[c];
  rng.nng = A.rng_nng[c];
  rng.have = A.rng_have[c];
  rn_load_stats(A, c, T);
  RnIt S;
  S.grads = 0;
  S.steps = 0;
  S.err = 0;

  // LeapFrog.initialize, LeapFrog.scala:102-116
  RnPQ s;
  rn_draw_normals(T, rng);  // pqBuf(i) = rng.standardNormal, i in nVars until 2 nVars
  RN_UNROLL
  for (int i = 0; i < RN_N; i++) s.q[i] = RN_Z(i);
  rn_update(A, s, S);
  double cq[RN_N], cg[RN_N];
  const double cU = s.U;
  RN_UNROLL
  for (int i = 0; i < RN_N; i++) {
    cq[i] = s.q[i];
    cg[i] = s.g[i];
  }
  rn_initialize_ps(A, c, T, s, 0, rng);
  RN_UNROLL
  for (int i = 0; i < RN_N; i++) RN_AT(A.params, i, c) = RN_P(i);  // params.p = the drawn momentum

  // stepSizeTuner.initialize
  double stepSize;
  if (A.step_tuner == 0) {  // DualAvgTuner.findReasonableStepSize, DualAvg.scala:27-41 (IdentityMassMatrix)
    const double H0 = rn_energy(A, c, T, s, 0, cU);
    stepSize = 1.0;
    double lap;
    rn_leapfrog(A, c, T, 0, s, 1, stepSize, S);  // tryStepping, LeapFrog.scala:14-22 (s still equals params here)
    lap = rn_log_accept(rn_energy(A, c, T, s, 0, s.U) - H0);
    const double exponent = (lap > -RN_LN2) ? 1.0 : -1.0;
    const double doubleOrHalf = (exponent > 0) ? 2.0 : 0.5;
    while (stepSize != 0.0 && (exponent * lap > -exponent * RN_LN2)) {
      stepSize *= doubleOrHalf;
      RN_UNROLL
      for (int i = 0; i < RN_N; i++) {
        RN_P(i) = RN_AT(A.params, i, c);
        s.q[i] = cq[i];
        s.g[i] = cg[i];
      }
      s.U = cU;
      rn_leapfrog(A, c, T, 0, s, 1, stepSize, S);
      lap = rn_log_accept(rn_energy(A, c, T, s, 0, s.U) - H0);
    }
    // DualAvg.apply, DualAvg.scala:80-90
    RN_AT(A.da, 1, c) = rn_log(stepSize);
    RN_AT(A.da, 2, c) = 0.0;
    RN_AT(A.da, 3, c) = 0.0;
    RN_AT(A.da, 4, c) = rn_log(10 * stepSize);
    A.da_iter[c] = 0;
  } else {
    stepSize = A.static_step;
  }
  RN_AT(A.da, 0, c) = stepSize;

  RN_UNROLL
  for (int i = 0; i < RN_N; i++) {
    RN_AT(A.params, RN_N + i, c) = cq[i];
    RN_AT(A.grad, i, c) = cg[i];
  }
  RN_AT(A.params, 2 * RN_N, c) = cU;
  A.rng_seed[c] = rng.seed;
  A.rng_nng[c] = rng.nng;
  A.rng_have[c] = rng.have;
  rn_fold(T, S);
  rn_store_stats(A, c, T, S.err);
}

// =============================================================================================================
// rn_k_warmup / rn_k_iter: A.n_iter iterations of Driver.warmup's loop (PHASE 0, Driver.scala:67-88) or of
// Driver.collectSamples (PHASE 1, Driver.scala:102-117).  Two entry points of one body so that the sampling kernel
// carries neither the code nor the registers of the adaptation.
// =============================================================================================================
template <int PHASE>
RN_DEVICE void rn_iterate(const RnArgs& A) {
  const int c = A.chain_begin + (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (c >= A.chain_end) return;
  const RnTs T = rn_ts_get();
  {
    RnRng rng;
    rng.seed = A.rng_seed[c];
    rng.nng = A.rng_nng[c];
    rng.have = A.rng_have[c];
    rn_rng_park(T, rng);
  }
  rn_load_stats(A, c, T);
  RnIt S;
  S.grads = 0;
  S.steps = 0;
  S.err = 0;
  int kind = A.mass_kind;
  rn_load_mass(A, c, T, kind);

  // step size in force: warmup uses the tuner's running value; sampling uses stepSizeTuner.stepSize
  // (= rn_exp(logStepSizeBar) for DualAvg, Driver.scala:37 / DualAvg.scala:23-25).  The rest of the DualAvg state is
  // touched once per warmup iteration and stays in (L1/L2-resident) global memory.
  double stepSize = RN_AT(A.da, 0, c);
  if (PHASE == 1 && A.step_tuner == 0) stepSize = rn_exp(RN_AT(A.da, 2, c));
  int win_size = A.win_size, win_i = A.win_i, win_j = A.win_j, est_samples = A.est_samples;
#if RN_ENABLE_EHMC
  int ring_i = 0, ring_full = 0;
  if (A.sampler == 1) {
    ring_i = A.ring_i[c];
    ring_full = A.ring_full[c];
  }
#endif
  // prevH = energy(params) at startIteration (LeapFrog.scala:54) is, by construction, the energy finishIteration of the
  // previous iteration filed under energyVariance (same function of the same numbers, :62-75) -- unless the mass matrix
  // was replaced in between.  It is carried in a register and recomputed only then (and at the start of a launch).
  bool havePrevH = false;

  // The current position, its gradient and potential stay in registers from one iteration to the next -- after an
  // accepted proposal they ARE the state the next iteration starts from, so only a rejection re-reads them from `params` (which is
  // written on accept exactly as before: it is what a rejection restores, what isUTurn measures against, and the state the launch
  // leaves behind).  The drawn momentum reaches `params` only where the reference's copy survives the iteration: on rejection
  // (from the scratch of the normal draws, intact while the momentum lives in registers under the identity mass).  With the
  // compile-time CTA size: 2.446 -> 2.400 ms per launch (profiles/r2_sweep_iter_v7_keep_state_block_dim.jsonl).
  RnPQ s;
  RN_UNROLL
  for (int i = 0; i < RN_N; i++) {
    s.q[i] = RN_AT(A.params, RN_N + i, c);
    s.g[i] = RN_AT(A.grad, i, c);
  }
  s.U = RN_AT(A.params, 2 * RN_N, c);

  for (int it = 0; it < A.n_iter; it++) {
    // ---------------- lf.startIteration, LeapFrog.scala:52-59 ----------------
    const double cU = s.U;
    if (!havePrevH) {
      RN_UNROLL
      for (int i = 0; i < RN_N; i++) RN_P(i) = RN_AT(A.params, i, c);  // old momentum
      RN_TS_PREV_H = rn_energy(A, c, T, s, kind, cU);
    }
    {
      RnRng rng = rn_rng_unpark(T);
      rn_initialize_ps(A, c, T, s, kind, rng);
      rn_rng_park(T, rng);
    }
    if (kind != 0) {  // initializePs writes into params (LeapFrog.scala:55); identity mass: on rejection only, below
      RN_UNROLL
      for (int i = 0; i < RN_N; i++) RN_AT(A.params, i, c) = RN_P(i);
    }
    s.U = cU;
    RN_TS_START_H = rn_energy(A, c, T, s, kind, cU);  // finishIteration's energy(params), :62
    const double usedStep = stepSize;

    // ---------------- sampler.warmup / sampler.run ----------------
    if (A.sampler == 0) {  // HMCSampler, HMC.scala:6-23
      rn_take_steps(A, c, T, kind, s, A.n_steps, stepSize, S);
    }
#if RN_ENABLE_EHMC
    else {  // EHMCSampler, EHMC.scala:15-61
      bool count = false;
      if (PHASE == 0 && !ring_full) count = true;  // shouldCountSteps, :29-30 (|| short-circuits: no draw while the ring fills)
      else if (PHASE == 0) {
        RnRng rng = rn_rng_unpark(T);
        count = rn_uniform(rng) < A.p_count;
        rn_rng_park(T, rng);
      }
      if (count) {  // countSteps, :32-50
        RnPQ snap;
        int l = 0;
        for (;;) {
          double out = 0.0;  // lf.isUTurn(params), LeapFrog.scala:35-47
          RN_UNROLL
          for (int i = 0; i < RN_N; i++) out += (s.q[i] - RN_AT(A.params, RN_N + i, c)) * RN_P(i);
          const bool uturn = (out != out) ? true : (out < 0);
          if (uturn || !(l < A.max_steps)) break;
          l += 1;
          rn_take_steps(A, c, T, kind, s, 1, stepSize, S);
          if (l == A.min_steps) {
            snap = s;
          }
        }
        if (l < A.min_steps) {
          rn_take_steps(A, c, T, kind, s, A.min_steps - l, stepSize, S);
        } else {
          s = snap;
        }
        // steps.add(l), Stats.scala:24-30
        ring_i += 1;
        if (ring_i == A.buf_size) ring_full = 1;
        ring_i = ring_i % A.buf_size;
        RN_AT(A.ring, ring_i, c) = (double)l;
      } else {  // steps.sample().toInt, Stats.scala:40-45
        RnRng rng = rn_rng_unpark(T);
        const int idx = ring_full ? rn_rng_int(rng, A.buf_size) : rn_rng_int(rng, ring_i + 1);
        rn_rng_park(T, rng);
        const int nsteps = rn_d2i(RN_AT(A.ring, idx, c));
        rn_take_steps(A, c, T, kind, s, nsteps, stepSize, S);
      }
    }
#endif

    // ---------------- lf.finishIteration, LeapFrog.scala:61-82 ----------------
    const double endH = rn_energy(A, c, T, s, kind, s.U);
    const double startH = RN_TS_START_H;
    const double deltaH = endH - startH;
    const double a = rn_log_accept(deltaH);
    bool accept;
    {
      RnRng rng = rn_rng_unpark(T);
      accept = a > rn_log(rn_uniform(rng));
      rn_rng_park(T, rng);
    }
    double eH;
    if (accept) {
      RN_UNROLL
      for (int i = 0; i < RN_N; i++) {
        RN_AT(A.params, i, c) = RN_P(i);
        RN_AT(A.params, RN_N + i, c) = s.q[i];
        RN_AT(A.grad, i, c) = s.g[i];
      }
      RN_AT(A.params, 2 * RN_N, c) = s.U;
      eH = endH;
      RN_ST_ACCEPTED += 1;
    } else {
      RN_UNROLL
      for (int i = 0; i < RN_N; i++) s.q[i] = RN_AT(A.params, RN_N + i, c);  // s.q := current position either way
      RN_UNROLL
      for (int i = 0; i < RN_N; i++) s.g[i] = RN_AT(A.grad, i, c);
      s.U = RN_AT(A.params, 2 * RN_N, c);
      if (kind == 0) {  // the momentum drawn at startIteration stays in params (LeapFrog.scala:55)
        RN_UNROLL
        for (int i = 0; i < RN_N; i++) RN_AT(A.params, i, c) = RN_Z(i);
      }
      eH = startH;
    }
    {  // stats.energyVariance.update(eH); energyTransitions2 += pow(eH - prevH, 2)
      const int e_n = RN_ST_E_N + 1;
      RN_ST_E_N = e_n;
      double e_mean = RN_ST_E_MEAN;
      const double oldDiff = eH - e_mean;
      e_mean += (oldDiff / (double)e_n);
      RN_ST_E_MEAN = e_mean;
      const double newDiff = eH - e_mean;
      RN_ST_E_RAW += oldDiff * newDiff;
      const double d = eH - RN_TS_PREV_H;
      RN_ST_TRANS2 += d * d;
    }
    RN_TS_PREV_H = eH;
    havePrevH = true;
    RN_ST_ITERS += 1;
    rn_ring_add(A, c, T, 1, rn_exp(a));
    rn_ring_add(A, c, T, 2, (double)S.grads);  // stats.gradientEvaluations - iterationStartGrads

    if (A.trace) {
      double* tr = A.trace + (size_t)it * 4 * (size_t)A.chains;
      tr[0 * (size_t)A.chains + c] = a;
      tr[1 * (size_t)A.chains + c] = accept ? 1.0 : 0.0;
      tr[2 * (size_t)A.chains + c] = usedStep;
      tr[3 * (size_t)A.chains + c] = (double)S.steps;
    }
    rn_fold(T, S);

    if (PHASE == 0) {
      // ---------------- stepSizeTuner.update, Driver.scala:69 / DualAvg.scala:58-77 ----------------
      if (A.step_tuner == 0) {
        const double newAcceptanceProb = rn_exp(a);
        const int daIter = A.da_iter[c] + 1;
        A.da_iter[c] = daIter;
        const double avgErrorMultiplier = 1.0 / ((double)daIter + 10);
        const double stepSizeMultiplier = rn_pow((double)daIter, -0.75);
        const double avgError = ((1.0 - avgErrorMultiplier) * RN_AT(A.da, 3, c) + (avgErrorMultiplier * (A.delta - newAcceptanceProb)));
        RN_AT(A.da, 3, c) = avgError;
        const double logStepSize = (RN_AT(A.da, 4, c) - (avgError * sqrt((double)daIter) / 0.05));
        RN_AT(A.da, 1, c) = logStepSize;
        RN_AT(A.da, 2, c) = (stepSizeMultiplier * logStepSize + (1.0 - stepSizeMultiplier) * RN_AT(A.da, 2, c));
        stepSize = rn_exp(logStepSize);
      }
      // ---------------- massMatrixTuner.update(sample), Driver.scala:74-80 / MassMatrix.scala:147-164 -------
#if RN_MASS_MAX >= 1
      if (A.mass_tuner == 1 || A.mass_tuner == 2) {
        win_j += 1;
        if (A.adaptation == 1) {
          // pooled extension: per-chain Welford statistics of the window; combined over chains (and ranks) at the window
          // end (rn_k_pool_reduce / rn_k_pool_apply) -- launches are cut at window ends in this mode
          if (!(win_j < A.skip_first || (A.total_warmup - win_j) < A.skip_last)) {
            win_i += 1;
            RN_UNROLL
            for (int i = 0; i < RN_N; i++) {  // the chain's Welford mean / M2 over this window
              double mean = RN_AT(A.est_mean, i, c);
              const double od = s.q[i] - mean;
              mean += od / (double)win_i;
              RN_AT(A.est_mean, i, c) = mean;
              RN_AT(A.est_raw, i, c) += od * (s.q[i] - mean);
            }
            if (win_i == win_size) {
              win_i = 0;
              win_size = rn_d2i(win_size * A.win_expansion);
            }
          }
        } else if (!(win_j < A.skip_first || (A.total_warmup - win_j) < A.skip_last)) {
          win_i += 1;
          est_samples += 1;  // VarianceEstimator.update, MassMatrixEstimator.scala:69-83
#if RN_MASS_MAX >= 2
          double oldDiff[RN_N], newDiff[RN_N];
#endif
          RN_UNROLL
          for (int i = 0; i < RN_N; i++) {
            double mean = RN_AT(A.est_mean, i, c);
            const double od = s.q[i] - mean;
            mean += (od / (double)est_samples);
            const double nd = s.q[i] - mean;
            RN_AT(A.est_mean, i, c) = mean;
            RN_AT(A.est_raw, i, c) += od * nd;
#if RN_MASS_MAX >= 2
            oldDiff[i] = od;
            newDiff[i] = nd;
#endif
          }
#if RN_MASS_MAX >= 2
          if (A.mass_tuner == 2) {  // CovarianceEstimator.update, :28-41
            for (int j = 0; j < RN_N; j++)
              for (int k = 0; k < RN_N; k++) RN_AT(A.est_cov, j * RN_N + k, c) += newDiff[j] * oldDiff[k];
          }
#endif
          if (win_i == win_size) {
            win_i = 0;
            win_size = rn_d2i(win_size * A.win_expansion);
            havePrevH = false;  // the next startIteration measures params with the NEW matrix
            if (A.mass_tuner == 1) {  // DiagonalMassMatrix(variance()), :92-103
              kind = 1;
              RN_UNROLL
              for (int i = 0; i < RN_N; i++) {
                const double v = RN_AT(A.est_raw, i, c) / (double)est_samples;
                if (v == 0.0) S.err |= 2;  // require(!elements.contains(0.0)), MassMatrix.scala:8
                RN_MASSD(i) = v;
                RN_AT(A.mass, i, c) = v;
                RN_AT(A.est_mean, i, c) = 0.0;  // reset(): mean/raw only, NOT samples (:60-67)
                RN_AT(A.est_raw, i, c) = 0.0;
              }
            }
#if RN_MASS_MAX >= 2
            else {  // DenseMassMatrix(covariance()), :43-50 + Cholesky MassMatrix.scala:76-117
              kind = 2;
              const double z = (double)(est_samples - 1);
              for (int i = 0; i < RN_N * RN_N; i++) {
                const double v = RN_AT(A.est_cov, i, c) / z;
                if (v == 0.0) S.err |= 2;
                RN_AT(A.mass, i, c) = v;
                RN_AT(A.est_cov, i, c) = 0.0;
              }
              for (int i = 0; i < RN_N; i++) {
                RN_AT(A.est_mean, i, c) = 0.0;
                RN_AT(A.est_raw, i, c) = 0.0;
              }
              double lower[(RN_N * (RN_N + 1)) / 2];
              int l = 0;
              for (int i = 0; i < RN_N; i++)
                for (int k = 0; k <= i; k++) {
                  double sum = 0.0;
                  for (int j = 0; j < k; j++) sum += lower[(i * (i + 1)) / 2 + j] * lower[(k * (k + 1)) / 2 + j];
                  const double x = RN_AT(A.mass, i * RN_N + k, c) - sum;
                  if (i == k)
                    lower[l] = sqrt(x);
                  else {
                    const double diag = lower[((k + 1) * (k + 2)) / 2 - 1];
                    lower[l] = (1.0 / diag * x);
                  }
                  l += 1;
                }
              l = 0;
              for (int i = 0; i < RN_N; i++)
                for (int k = 0; k < (RN_N - i); k++) {
                  RN_AT(A.chol, l, c) = lower[((k + i) * (k + i + 1)) / 2 + i];
                  l += 1;
                }
            }
#endif
            // stepSize = stepSizeTuner.reset(), Driver.scala:78 / DualAvg.scala:17-21
            if (A.step_tuner == 0) {
              const double ss = rn_exp(RN_AT(A.da, 2, c));
              RN_AT(A.da, 1, c) = rn_log(ss);
              RN_AT(A.da, 2, c) = 0.0;
              RN_AT(A.da, 3, c) = 0.0;
              A.da_iter[c] = 0;
              RN_AT(A.da, 4, c) = rn_log(10 * ss);
              stepSize = ss;
            }
          }
        }
      }
#endif
    } else if (A.samples) {  // lf.variables(params, output), Driver.scala:105-107
      double* out = A.samples + (size_t)it * RN_N * (size_t)A.chains;
      RN_UNROLL
      for (int i = 0; i < RN_N; i++) RN_STCS(&out[(size_t)i * (size_t)A.chains + c], s.q[i]);
    }
  }

  if (PHASE == 0) RN_AT(A.da, 0, c) = stepSize;
#if RN_ENABLE_EHMC
  if (A.sampler == 1) {
    A.ring_i[c] = ring_i;
    A.ring_full[c] = ring_full;
  }
#endif
  {
    const RnRng rng = rn_rng_unpark(T);
    A.rng_seed[c] = rng.seed;
    A.rng_nng[c] = rng.nng;
    A.rng_have[c] = rng.have;
  }
  rn_store_stats(A, c, T, S.err);
}
RN_GLOBAL void rn_k_warmup(const RnArgs A) { rn_iterate<0>(A); }
RN_GLOBAL void rn_k_iter(const RnArgs A) { rn_iterate<1>(A); }
#define RN_K_WARMUP rn_k_warmup

// =============================================================================================================
// rn_k_density: DensityFunction.update/density/gradient for a batch of positions (Model.scala:38-50).
// q: [N][chains] ; out: [N+1][chains] = density, gradient
// =============================================================================================================
RN_GLOBAL void rn_k_density(const double* RN_RESTRICT qin, double* RN_RESTRICT out, const double* data, int* err,
                            int chains) {
  const int c = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (c >= chains) return;
  double q[RN_N], g[RN_N], dens;
  RN_UNROLL
  for (int i = 0; i < RN_N; i++) q[i] = qin[(size_t)i * chains + c];
  int e = 0;
  rn_density(q, dens, g, data, e);
  out[c] = dens;
  RN_UNROLL
  for (int i = 0; i < RN_N; i++) out[(size_t)(i + 1) * chains + c] = g[i];
#ifdef RN_HOST_EMULATION
  if (e) *err |= e;
#else
  if (e) atomicOr(err, e);
#endif
}

// =============================================================================================================
// rn_k_transpose: [rows][cols] -> [cols][rows] (sample chunks [iter][n][chain] -> [chain][iter][n] before the
// device->host copy of rn_sample).  32x32 tiles through shared memory, both sides coalesced.
// =============================================================================================================
#ifndef RN_HOST_EMULATION
RN_GLOBAL void rn_k_transpose(const double* RN_RESTRICT src, double* RN_RESTRICT dst, int rows, int cols,
                              long long src_ld, long long dst_ld, long long dst_off) {
  // dst[c * dst_ld + dst_off + r] = src[r * src_ld + c]   (a block of `cols` chains out of src_ld)
  __shared__ double tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += 8) {
    const int r = r0 + j, c = c0 + threadIdx.x;
    if (r < rows && c < cols) tile[j][threadIdx.x] = src[(size_t)r * (size_t)src_ld + c];
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += 8) {
    const int c = c0 + j, r = r0 + threadIdx.x;
    if (r < rows && c < cols) dst[(size_t)c * (size_t)dst_ld + (size_t)dst_off + r] = tile[threadIdx.x][j];
  }
}
#endif

// =============================================================================================================
// Pooled mass-matrix adaptation (RN_ADAPT_POOLED; an extension, not reference semantics): at a window end the chains'
// Welford statistics of the window (mean_c, M2_c over L draws) are combined over all chains of this GPU and, through two
// small ncclAllReduce calls, over all ranks: first the means (-> pooled mean), then M2_c + L (mean_c - mean)^2 (Chan's
// parallel variance: no s2/n - mean^2 cancellation).  Reductions run in a fixed order (no atomics): the shared diagonal
// mass matrix is reproducible run to run.  It is applied to every chain, statistics cleared, DualAvg restarted from each
// chain's averaged step size (Driver.scala:75-80).
// =============================================================================================================
#ifndef RN_HOST_EMULATION
RN_GLOBAL void rn_k_pool_reduce(const RnArgs A, double* pool, int window_len, int pass) {
  // One block per parameter; thread t adds chains t, t + 256, ... in order, then a fixed tree: the result does not depend
  // on scheduling (no atomics).  pass 0: pool[1 + i] = sum over chains of the chain's window mean, pool[0] = chains.
  // pass 1 (after the all-reduce of pass 0): pool[1 + n + i] = sum over chains of [M2_c + L (mean_c - mean)^2] -- Chan's
  // combination of the chains' Welford statistics around the POOLED mean (no s2/n - mean^2 cancellation).
  __shared__ double red[256];
  const int i = (int)blockIdx.x;
  const double gmean = pass ? pool[1 + i] / pool[0] : 0.0;
  const double* mean = A.est_mean + (size_t)i * A.chains;
  const double* m2 = A.est_raw + (size_t)i * A.chains;
  double acc = 0.0;
  for (int c = (int)threadIdx.x; c < A.chains; c += (int)blockDim.x) {
    if (pass) {
      const double d = mean[c] - gmean;
      acc += m2[c] + (double)window_len * d * d;
    } else {
      acc += mean[c];
    }
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = (int)blockDim.x / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    pool[1 + (pass ? RN_N : 0) + i] = red[0];
    if (!pass && i == 0) pool[0] = (double)A.chains;
  }
}
RN_GLOBAL void rn_k_pool_apply(const RnArgs A, const double* pool, int window_len) {
  const int c = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (c >= A.chains) return;
  const double cnt = pool[0] * (double)window_len;  // draws of the window over all chains of all ranks
  for (int i = 0; i < RN_N; i++) {
    const double var = pool[1 + RN_N + i] / cnt;
    if (!(var > 0.0)) A.st_err[c] |= 2;
    RN_AT(A.mass, i, c) = var;
    RN_AT(A.est_mean, i, c) = 0.0;
    RN_AT(A.est_raw, i, c) = 0.0;
  }
  if (A.step_tuner == 0) {  // stepSizeTuner.reset(), DualAvg.scala:17-21
    const double ss = rn_exp(RN_AT(A.da, 2, c));
    RN_AT(A.da, 0, c) = ss;
    RN_AT(A.da, 1, c) = rn_log(ss);
    RN_AT(A.da, 2, c) = 0.0;
    RN_AT(A.da, 3, c) = 0.0;
    RN_AT(A.da, 4, c) = rn_log(10 * ss);
    A.da_iter[c] = 0;
  }
}
#endif

#endif  // RN_SAMPLER_CUH
