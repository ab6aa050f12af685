"""The hand-written thread-per-chain sampler source (rn_sampler.cuh) compiled for the host and run against the oracle on
this box (no GPU): the same LeapFrog / HMC / EHMC / DualAvg / mass-matrix logic the GPU executes, one emulated thread
per chain (tests/host_emulation.py).  Bit-exact: g++ -ffp-contract=off + the prelude's fdlibm = the oracle's arithmetic.
The GPU tests (-m gpu) remain the parity tests proper; this is the CPU-side safety net for the kernel source."""
import numpy as np
import pytest

from oracle.rainier_py import configs, sbc_models
from oracle.rainier_py.binding import OracleModel
from rainier_b200 import abi, api

import host_emulation as he


def _run(model, config, seeds, dense=False):
    rir, cols = model.compile(True)
    cfg, keep = api.lower_config(config)
    cfg.backend = abi.RN_BACKEND_THREAD
    cm = api.CudaModel(rir, cols, device=-1)
    config.backend = abi.RN_BACKEND_THREAD
    got = he.sample(cm.emit_source(config), cfg, seeds, cm)
    ref = OracleModel(rir, cols).sample(cfg, seeds=seeds, trace=True, dense_mass=dense)
    assert np.array_equal(got["trace"][:, :, 1], ref["trace"][:, :, 1]), "accept decisions differ"
    assert np.array_equal(got["trace"][:, :, 3], ref["trace"][:, :, 3]), "leapfrog step counts differ"
    assert np.array_equal(got["samples"], ref["samples"]), "samples are not bit-identical"
    for k, o in enumerate(ref["stats"]):
        assert got["stats"][k, 0] == o.gradient_evaluations and got["stats"][k, 1] == o.leapfrog_steps
        assert got["stats"][k, 2] == o.accepted and got["stats"][k, 3] == o.rng.seed48 and got["stats"][k, 4] == 0
    assert np.array_equal(got["mass"], ref["mass"])
    return got


def _cfg(it, warm, sampler, step, mass, **kw):
    return api.make_config(iterations=it, warmupIterations=warm, sampler=sampler, stepSizeTuner=step, massMatrixTuner=mass, **kw)


def test_hmc_dualavg_funnel_on_host():
    _run(configs.funnel(), _cfg(30, 120, api.HMCSampler(5), api.DualAvgTuner(0.8), api.IdentityMassMatrixTuner()), np.arange(6) + 7)


def test_round2b_source_variants_on_host():
    """the round-2b forms of the sampler source (two polar attempts and two second-pass pairs per trip, speculative fdlibm common
    paths with their coefficients in the constant bank, state kept in registers across iterations) are bit-exact -- even and odd
    numbers of parameters (odd: the cached second variate alternates)"""
    _run(configs.funnel(), _cfg(12, 40, api.HMCSampler(5), api.DualAvgTuner(0.8), api.IdentityMassMatrixTuner()), np.arange(4) + 7)
    _run(configs.funnel(7), _cfg(12, 30, api.HMCSampler(4), api.DualAvgTuner(0.8), api.IdentityMassMatrixTuner()), np.arange(3) + 3)
    model = sbc_models.build("SBCGamma")[0]
    _run(model, _cfg(10, 30, api.HMCSampler(3), api.DualAvgTuner(0.8), api.IdentityMassMatrixTuner()), np.arange(3) + 2)
    _run(configs.eight_schools(), api.SamplerConfig(iterations=10, warmupIterations=60), np.arange(2) + 11)


def test_default_config_eight_schools_on_host():
    """EHMC + DualAvg + windowed diagonal mass adaptation (DefaultConfig, Sampler.scala:17-27)"""
    _run(configs.eight_schools(), api.SamplerConfig(iterations=40, warmupIterations=260), np.arange(5) + 11)


def test_dense_mass_tuner_on_host():
    cfg = _cfg(20, 200, api.EHMCSampler(32, 1, 10, 0.1), api.DualAvgTuner(0.8), api.DenseMassMatrixTuner(40, 1.5, 20, 20))
    _run(configs.eight_schools(), cfg, np.arange(3) + 5, dense=True)


def test_streamed_rows_on_host():
    """a streamed target (sequential row order of DataFunction.compute) under HMC with a static step size"""
    model = sbc_models.build("SBCLaplace")[0]
    _run(model, _cfg(15, 40, api.HMCSampler(2), api.DualAvgTuner(0.8), api.IdentityMassMatrixTuner()), np.arange(4) + 1)


# ---------------------------------------------------------------------------------------------------------------
# warp-per-chain source (rn_sampler_wpc.cuh + the emitted rows-across-lanes density) on 32 host threads per chain
# ---------------------------------------------------------------------------------------------------------------
def _run_wpc(model, config, seeds, tol, rir_gpu=None, cols_gpu=None, tma="0", k="1", chains_per_cta=1):
    import os
    rir, cols = model.compile(True)
    config.backend = abi.RN_BACKEND_WARP
    cfg, keep = api.lower_config(config)
    os.environ["RN_TMA"] = tma  # "0": per-warp loads; "2": the tile pipeline, emulated synchronously (memcpy + barriers)
    os.environ["RN_WPC_K"] = k  # warps per chain
    try:
        cm = api.CudaModel(rir_gpu if rir_gpu is not None else rir, cols_gpu if cols_gpu is not None else cols, device=-1)
        src = cm.emit_source(config)
    finally:
        del os.environ["RN_TMA"], os.environ["RN_WPC_K"]
    assert "#define RN_BACKEND 1" in src and ("#define RN_TMA_STAGES %s" % tma) in src and ("#define RN_WPC_K %s" % k) in src
    q = np.random.default_rng(0).normal(size=(2, cm.nVars)) * 0.3
    om = OracleModel(rir, cols)
    d, err = he.density(src, q, None, cm)
    ref_d = om.density_batch(q)
    assert err == 0 and np.max(np.abs(d - ref_d) / np.maximum(np.abs(ref_d), 1e-9)) < tol
    got = he.sample(src, cfg, seeds, cm, chains_per_cta=chains_per_cta)
    dense = cfg.mass_tuner == abi.RN_MASS_DENSE or (cfg.mass_tuner == abi.RN_MASS_STATIC and cfg.static_matrix == abi.RN_MATRIX_DENSE)
    ref = om.sample(cfg, seeds=seeds, trace=True, dense_mass=dense)
    assert np.array_equal(got["trace"][:, :, 1], ref["trace"][:, :, 1]), "accept decisions differ"
    assert np.array_equal(got["trace"][:, :, 3], ref["trace"][:, :, 3]), "leapfrog step counts differ"
    assert np.max(np.abs(got["samples"] - ref["samples"]) / np.maximum(np.abs(ref["samples"]), 1e-9)) < tol
    if cfg.mass_tuner == abi.RN_MASS_DENSE and got["mass_kind"] == 2:  # the adapted covariance matrix itself
        assert np.max(np.abs(got["mass"] - ref["mass"]) / np.maximum(np.abs(ref["mass"]), 1e-9)) < max(tol, 1e-300)
    for k, o in enumerate(ref["stats"]):
        assert got["stats"][k, 0] == o.gradient_evaluations and got["stats"][k, 3] == o.rng.seed48


def test_wpc_data_free_model_is_bit_exact_on_host():
    _run_wpc(configs.eight_schools(), api.SamplerConfig(iterations=12, warmupIterations=70), np.arange(2) + 3, tol=1e-300)


def test_wpc_streamed_logistic_regression_on_host():
    """rows across 32 emulated lanes, butterfly reduction, HMC with a static step size in the stable regime; the GPU
    side differentiates the primal RIR itself (adjoint mode, what the Scala CudaCompiler sends)"""
    model = configs.logreg(300, 3)
    prir, pcols = model.compile(False)
    cfg = api.make_config(iterations=6, warmupIterations=0, sampler=api.HMCSampler(3), stepSizeTuner=api.StaticStepSize(0.02),
                          massMatrixTuner=api.IdentityMassMatrixTuner())
    _run_wpc(model, cfg, np.arange(2) + 9, tol=1e-9, rir_gpu=prir, cols_gpu=pcols)
    # same run through the data-tile pipeline: full 32-row tiles from the staged buffer, ragged remainder from global
    # memory, two stages cycling across targets and density calls (300 observations -> 37 rows per split target)
    _run_wpc(model, cfg, np.arange(2) + 9, tol=1e-9, rir_gpu=prir, cols_gpu=pcols, tma="2")


def test_wpc_two_warps_per_chain_on_host():
    """K = 2: 64 emulated threads per chain, named group barrier, cross-warp reduction scratch, 64-row super-tiles"""
    _run_wpc(configs.eight_schools(), api.SamplerConfig(iterations=8, warmupIterations=60), np.arange(2) + 3, tol=1e-300, k="2")
    model = configs.logreg(600, 3)
    prir, pcols = model.compile(False)
    cfg = api.make_config(iterations=4, warmupIterations=0, sampler=api.HMCSampler(3), stepSizeTuner=api.StaticStepSize(0.02),
                          massMatrixTuner=api.IdentityMassMatrixTuner())
    _run_wpc(model, cfg, np.arange(2) + 9, tol=1e-9, rir_gpu=prir, cols_gpu=pcols, tma="2", k="2")


def _standard_normal_model():
    from oracle.rainier_py.compute import Real
    from oracle.rainier_py.core import Model
    # NormalDensityFunction of the reference's LeapFrogTest: density = x*x / -2.0, gradient = -x
    return Model.track_(list(Real.parameters(1, lambda t: (t[0] * t[0]) / -2.0)))


def test_reference_leapfrog_test_standard_normal_on_host():
    """rainier-test/.../sampler/LeapFrogTest.scala:60-69 ("standard normal, identity matrix"): ScalaRNG(123), 1000
    iterations of takeSteps(1) at stepSize 1.0; |mean| < 0.2 and |variance - 1| < 0.2 -- through the emitted + hand-written
    kernel source on the host, bit-identical to the oracle's run of the same chain."""
    cfg = _cfg(1000, 0, api.HMCSampler(1), api.StaticStepSize(1.0), api.IdentityMassMatrixTuner())
    got = _run(_standard_normal_model(), cfg, np.array([123]))
    x = got["samples"][0, :, 0]
    assert abs(x.mean()) < 0.2
    assert abs(((x - 0.0) ** 2).sum() / (len(x) - 1) - 1.0) < 0.2


def test_wpc_dense_mass_matrix_on_host():
    """DenseMassMatrixTuner on the warp-per-chain kernels (opt-in: AUTO keeps dense configurations on the thread-per-chain
    kernels): mat-vec rows across the lanes, back-substitution and Cholesky on one lane, all in the reference's summation
    order -> bit-exact on a data-free model, adapted covariance matrix included (MassMatrix.scala:35-117,
    MassMatrixEstimator.scala:9-50); streamed rows within 1e-9 with equal accept decisions.  (Static dense matrices: GPU
    test only -- the host emulation shim has no static-matrix upload.)"""
    # short trajectories: every emulated barrier is a pthread barrier over 32 host threads
    cfg = api.make_config(iterations=4, warmupIterations=65, sampler=api.EHMCSampler(16, 1, 10, 0.1), stepSizeTuner=api.DualAvgTuner(0.8),
                          massMatrixTuner=api.DenseMassMatrixTuner(20, 1.5, 10, 10))  # windows end at iterations 30 and 60
    _run_wpc(configs.eight_schools(), cfg, np.arange(1) + 3, tol=1e-300)
    model = configs.logreg(300, 3)
    prir, pcols = model.compile(False)
    cfg = api.make_config(iterations=4, warmupIterations=40, sampler=api.HMCSampler(3), stepSizeTuner=api.DualAvgTuner(0.8),
                          massMatrixTuner=api.DenseMassMatrixTuner(15, 1.5, 5, 5))
    _run_wpc(model, cfg, np.arange(1) + 9, tol=1e-9, rir_gpu=prir, cols_gpu=pcols, tma="2")


def test_wpc_dense_mass_matrix_beyond_the_thread_shape_limit():
    """70 parameters: more than the thread-per-chain kernels keep in thread-local Cholesky scratch (n <= 64) -- the
    warp-per-chain shape holds matrix, factor and estimator in the chain's global state; still bit-exact on a data-free model"""
    model = configs.funnel(70)
    cfg = api.make_config(iterations=2, warmupIterations=34, sampler=api.HMCSampler(2), stepSizeTuner=api.DualAvgTuner(0.8),
                          massMatrixTuner=api.DenseMassMatrixTuner(12, 1.5, 4, 4))
    _run_wpc(model, cfg, np.arange(1) + 3, tol=1e-300)
    cfg.backend = abi.RN_BACKEND_THREAD
    with pytest.raises(api.RainierCudaError) as e:
        api.CudaModel(*model.compile(True), device=-1).sample(cfg, seeds=[1])
    assert e.value.code == abi.RN_E_UNSUPPORTED


def test_static_mass_matrices_on_host_both_shapes():
    """StaticMassMatrix(DiagonalMassMatrix / DenseMassMatrix) (Sampler.scala:47-50, MassMatrix.scala:3-32): velocity,
    momentum draw through the packed Cholesky factor, energy -- on the thread-per-chain source and on the warp-per-chain
    source, bit-exact on a data-free model (the reference's LeapFrogTest uses a static DiagonalMassMatrix, :70-78)."""
    n = 10
    diag = api.DiagonalMassMatrix(np.linspace(0.5, 2.0, n))
    A = np.random.default_rng(3).normal(size=(n, n)) * 0.2 + np.eye(n) * 1.5
    dense = api.DenseMassMatrix((A @ A.T).reshape(-1))
    for mass in (diag, dense):
        cfg = _cfg(6, 25, api.HMCSampler(3), api.DualAvgTuner(0.8), api.StaticMassMatrix(mass))
        got = _run(configs.funnel(), cfg, np.arange(3) + 1, dense=mass is dense)  # thread per chain; compared with the oracle inside _run
        assert got["mass_kind"] == (1 if mass is diag else 2)
        cfgw = api.make_config(iterations=4, warmupIterations=20, sampler=api.EHMCSampler(8, 1, 6, 0.2), stepSizeTuner=api.DualAvgTuner(0.8),
                               massMatrixTuner=api.StaticMassMatrix(mass))
        _run_wpc(configs.funnel(), cfgw, np.arange(1) + 5, tol=1e-300)


def test_wpc_several_chains_per_cta_share_the_data_tiles_on_host():
    """The lockstep protocol of the CTA-shared data tiles (rn_sampler_wpc.cuh / emitted tile loop): 3 chains per emulated CTA
    (96 host threads; the second CTA of the launch has one chain and two idle slots), thread 0 of the CTA issues every
    "bulk copy", all chain-owning warps consume the same staged tile between the tile barrier pair; 2 stages; then the same
    with 2 warps per chain.  HMC (every chain evaluates the density equally often), streamed logistic regression."""
    model = configs.logreg(300, 3)
    prir, pcols = model.compile(False)
    cfg = api.make_config(iterations=4, warmupIterations=12, sampler=api.HMCSampler(3), stepSizeTuner=api.DualAvgTuner(0.8),
                          massMatrixTuner=api.IdentityMassMatrixTuner())
    _run_wpc(model, cfg, np.arange(4) + 9, tol=1e-9, rir_gpu=prir, cols_gpu=pcols, tma="2", chains_per_cta=3)
    model = configs.logreg(600, 3)
    prir, pcols = model.compile(False)
    cfg = api.make_config(iterations=3, warmupIterations=0, sampler=api.HMCSampler(2), stepSizeTuner=api.StaticStepSize(0.02),
                          massMatrixTuner=api.IdentityMassMatrixTuner())
    _run_wpc(model, cfg, np.arange(3) + 9, tol=1e-9, rir_gpu=prir, cols_gpu=pcols, tma="2", k="2", chains_per_cta=2)


def test_wpc_rerolled_invariant_sections_on_host():
    """A vector of 48 latent group effects (cfg 5's shape, small): the warp-per-chain density re-rolls the 48 table entries,
    prior terms and gradient outputs into loops across the group's threads (rn_emit.cpp: rr_plan).  Same values as the
    unrolled statements (RN_NO_REROLL) to rounding of the re-associated sums, same accept decisions as the oracle."""
    import os
    model = configs.poisson_glm(48, 768)
    prir, pcols = model.compile(False)
    cfg = api.make_config(iterations=4, warmupIterations=0, sampler=api.HMCSampler(3), stepSizeTuner=api.StaticStepSize(0.004),
                          massMatrixTuner=api.IdentityMassMatrixTuner())
    cfg.backend = abi.RN_BACKEND_WARP
    cm = api.CudaModel(prir, pcols, device=-1)
    src = cm.emit_source(cfg)
    dens = src[src.index("// ---- emitted"):src.index("// rn_sampler_wpc.cuh --")]
    assert "for (int k = lane; k < 48; k += RN_G) {" in dens and "grad[2 + k] = " in dens and "scr[0 + k] = " in dens
    assert dens.count("\n") < 700, "the invariant sections are loops, not 48 copies"
    os.environ["RN_NO_REROLL"] = "1"
    try:
        src0 = api.CudaModel(prir, pcols, device=-1).emit_source(cfg)
    finally:
        del os.environ["RN_NO_REROLL"]
    assert "grad[2 + k] = " not in src0[src0.index("// ---- emitted"):src0.index("// rn_sampler_wpc.cuh --")]
    q = np.random.default_rng(4).normal(size=(3, cm.nVars)) * 0.3
    d1, e1 = he.density(src, q, None, cm)
    d0, e0 = he.density(src0, q, None, cm)
    assert e0 == 0 and e1 == 0
    assert np.max(np.abs(d1 - d0) / np.maximum(np.abs(d0), 1e-9)) < 1e-12
    _run_wpc(model, cfg, np.arange(2) + 9, tol=1e-9, rir_gpu=prir, cols_gpu=pcols, tma="2")
    _run_wpc(model, cfg, np.arange(2) + 9, tol=1e-9, rir_gpu=prir, cols_gpu=pcols, tma="2", k="2", chains_per_cta=2)


def test_wpc_row_bodies_with_cuda_libm_on_host(monkeypatch):
    """row bodies that keep more than 8 accumulators in registers use CUDA's exp / log instead of the branch-free row functions
    (rn_emit.cpp: row_functions): the rows-across-lanes logistic regression with 8 covariates (9 accumulators) and no DMMA path -- same accept
    decisions as the oracle, densities to the tolerance of this shape"""
    monkeypatch.setenv("RN_MMA", "0")
    model = configs.logreg(600, 8)  # 75 rows of 8 observations: data tiles with two warps per chain as well
    prir, pcols = model.compile(False)
    cfg = api.make_config(iterations=5, warmupIterations=0, sampler=api.HMCSampler(3), stepSizeTuner=api.StaticStepSize(0.02),
                          massMatrixTuner=api.IdentityMassMatrixTuner())
    cfg.backend = abi.RN_BACKEND_WARP
    src = api.CudaModel(prir, pcols, device=-1).emit_source(cfg)
    dens = src[src.index("// ---- emitted"):src.index("// rn_sampler_wpc.cuh --")]
    assert " exp(" in dens and " log(" in dens and "rn_row_" not in dens
    _run_wpc(model, cfg, np.arange(2) + 9, tol=1e-9, rir_gpu=prir, cols_gpu=pcols, tma="2")
    _run_wpc(model, cfg, np.arange(2) + 9, tol=1e-9, rir_gpu=prir, cols_gpu=pcols, tma="2", k="2", chains_per_cta=2)
