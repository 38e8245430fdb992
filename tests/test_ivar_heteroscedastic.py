"""Greedy IVAR under a heteroscedastic noise function nu(x) (space.noiseFunc): the cost of design + [c] takes the per-point
nugget nu(design + [c]), the reference's branch of costFunctionGP_IVAR.evaluate (experimentalDesign.py:110-114).  The
device engine keeps its candidate running variance noise-inclusive, var_D(c) + nu(c), and runs the unchanged kernels
with scalar noise 0.

The oracles are tests/hetero_oracle.py.
CPU: the vectorised oracle with a nu vector against the reference's loop with the callable; both oracles with a constant
nu against the float-noise oracles; the candidate-sharding protocol (gloo) with nu(p) travelling in the pivot record;
rejected noise functions.
GPU: every loop mode against the reference's loop; each pick's cost against costFunctionGP_IVAR.evaluate; a constant
noise function against the scalar run; pinv's zero-variance rule where nu = 0; the stateless scoring call; a mid-size run
against the vectorised oracle."""
import functools
import os
import socket

import numpy as np
import pytest

from oracle import gpexp_oracle as orc
from tests.cases import product_kernel, spec
from tests.hetero_oracle import fast_greedy_ivar_nu, ref_greedy_ivar_nu

DMMA, I8 = 1, 2
HDR = 3 + 16


# ---- noise functions: pointwise and deterministic; cond(K_DD + diag nu) stays <~ 1e6 on the designs below -------------
def nu_golden(p):
    """The function test_gpu_parity pins against the unmodified reference (gp/hetero/ivar_cost)."""
    return 1e-4 + 1e-3 * p[:, 0] ** 2


def nu_span(p):
    """1e-6 at x0 = -1 to 1e-3 at x0 = 1: three orders of magnitude."""
    return 1e-6 * 1e3 ** np.clip((p[:, 0] + 1.0) / 2.0, 0.0, 1.0)


def nu_half_zero(p):
    """Exactly 0 for x0 < 0."""
    return np.where(p[:, 0] < 0.0, 0.0, 1e-4 + 1e-3 * p[:, 0] ** 2)


def nu_mehler(p):
    """At least 1e-2, the noise level of cfg-4's Mehler kernel."""
    return 1e-2 * (1.0 + 10.0 * p[:, 0] ** 2)


def nu_mehler_span(p):
    """1e-2 at x0 <= -2 to 10 at x0 >= 2."""
    return 1e-2 * 1e3 ** np.clip((p[:, 0] + 2.0) / 4.0, 0.0, 1.0)


def _sample(name, rng, *shapes):
    d = spec(name).dim
    if name.startswith("mehler"):
        return [rng.standard_normal((n, d)) for n in shapes]
    return [rng.uniform(-1, 1, (n, d)) for n in shapes]


def _rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b)) / np.abs(np.asarray(b))))


CPU_CASES = [("se_ard_2d_wide", nu_golden), ("se_ard_2d_wide", nu_span), ("se_ard_2d_wide", nu_half_zero),
             ("matern_5d", nu_golden), ("matern_5d", nu_span), ("matern_5d", nu_half_zero),
             ("mehler_3d", nu_mehler), ("mehler_3d", nu_mehler_span)]


# ------------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,nu", CPU_CASES, ids=[f"{n}-{f.__name__}" for n, f in CPU_CASES])
def test_fast_oracle_with_noise_vector_equals_reference_loop(name, nu):
    rng = np.random.default_rng(31)
    cand, mc = _sample(name, rng, 60, 400)
    cand[41] = cand[7]   # a duplicated candidate: once one copy is picked the other is scored against a repeated node
    ks = spec(name)
    ref_idx, ref_costs = ref_greedy_ivar_nu(ks, cand, mc, 8, nu)
    idx, costs = fast_greedy_ivar_nu(ks, cand, mc, 8, nu(cand))
    assert idx == ref_idx
    for s in range(8):
        assert _rel(costs[s], ref_costs[s]) <= 1e-9, s


def test_constant_noise_oracles_are_the_float_oracles():
    """With nu = s2 everywhere, both heteroscedastic oracles reproduce the float-noise oracles bit for bit."""
    rng = np.random.default_rng(32)
    cand, mc = _sample("matern_5d", rng, 40, 300)
    ks, s2 = spec("matern_5d"), 1e-4
    a_idx, a_costs = orc.ref_greedy_ivar(ks, cand, mc, 6, s2)
    b_idx, b_costs = ref_greedy_ivar_nu(ks, cand, mc, 6, lambda p: np.full(p.shape[0], s2))
    assert a_idx == b_idx and all(np.array_equal(a, b) for a, b in zip(a_costs, b_costs))
    f_idx, f_costs = orc.fast_greedy_ivar(ks, cand, mc, 6, s2)
    g_idx, g_costs = fast_greedy_ivar_nu(ks, cand, mc, 6, np.full(cand.shape[0], s2))
    assert f_idx == g_idx == a_idx and all(np.array_equal(a, b) for a, b in zip(f_costs, g_costs))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, cand, mc, nu, n_points, q):
    """One rank of the sharded greedy IVAR with the engine's conventions: varC = var_D + nu on the local block, scalar
    noise 0, and the owner's rec[2] = varC[p] = var_D(p) + nu(p) as the divisor of every rank's append."""
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from gpexp_b200.engine import Shard
    shard = Shard()
    kern = orc.KernelSpec.se([0.3, 0.45], 1.7, 2)
    lo, hi = Shard.split(len(cand), world, rank)
    local = cand[lo:hi]
    reclen = HDR + n_points
    var_c, var_m = kern.prior(local) + nu[lo:hi], kern.prior(mc).copy()
    Wc, Wm = np.zeros((n_points, hi - lo)), np.zeros((n_points, len(mc)))
    picks, pivots = [], []
    for n in range(n_points):
        cost = orc.fast_ivar_scores(kern, local, mc, Wm[:n], var_m, Wc[:n], var_c, 0.0)
        j = int(np.argmin(cost))
        rec = np.zeros(reclen)
        rec[0], rec[1], rec[2] = cost[j], lo + j, var_c[j]
        rec[3:5] = local[j]
        rec[HDR:HDR + n] = Wc[:n, j]
        out = torch.zeros(world * reclen, dtype=torch.float64)
        shard.all_gather(out, torch.from_numpy(rec))
        recs = out.numpy().reshape(world, reclen)
        # gpx_select_pivot: lowest score, ties to the lowest global index
        win = recs[min(range(world), key=lambda r: (recs[r][0], recs[r][1]))]
        lnn, x, col = np.sqrt(win[2]), win[3:5][None, :], win[HDR:HDR + n]
        rc = (kern.gram(x, local)[0] - col @ Wc[:n]) / lnn
        rm = (kern.gram(x, mc)[0] - col @ Wm[:n]) / lnn
        Wc[n], Wm[n] = rc, rm
        var_c -= rc * rc
        var_m -= rm * rm
        picks.append(int(win[1]))
        pivots.append(float(win[2]))
    q.put((rank, picks, pivots))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_protocol_carries_the_pick_noise():
    import torch.multiprocessing as mp
    rng = np.random.default_rng(33)
    cand, mc = rng.uniform(-1, 1, (101, 2)), rng.uniform(-1, 1, (300, 2))
    n_points, world = 9, 2
    nu = nu_span(cand)
    ks = orc.KernelSpec.se([0.3, 0.45], 1.7, 2)
    ref, _ = fast_greedy_ivar_nu(ks, cand, mc, n_points, nu)
    assert ref == ref_greedy_ivar_nu(ks, cand, mc, n_points, nu_span)[0]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, cand, mc, nu, n_points, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, picks, pivots in results:
        assert picks == ref, (rank, picks, ref)
        # the divisor each rank used is var_D(p) + nu(p) of the pick
        for s, p in enumerate(picks):
            var = ks.prior(cand[p:p + 1])[0] if s == 0 else \
                orc.fast_posterior_variance(ks, cand[picks[:s]], cand[p:p + 1], nu[picks[:s]])[0]
            assert abs(pivots[s] - (var + nu[p])) <= 1e-12 * ks.signal, (rank, s)


@pytest.mark.parametrize("bad,what", [(lambda p: np.full(p.shape[0] + 1, 1e-4), "values for"),
                                      (lambda p: np.where(p[:, 0] > 0.5, np.nan, 1e-4), "not finite"),
                                      (lambda p: np.where(p[:, 0] > 0.5, -1e-8, 1e-4), "negative")],
                         ids=["length", "nan", "negative"])
def test_bad_noise_function_is_rejected(bad, what):
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space
    rng = np.random.default_rng(34)
    cand, mc = rng.uniform(-1, 1, (50, 2)), rng.uniform(-1, 1, (80, 2))
    cf = ed.costFunctionGP_IVAR(gpmod.GP(product_kernel("se_ard_2d_wide"), 1e-6), 1, Space(2, None, None, noise=bad),
                                mcPoints=mc)
    with pytest.raises(ValueError, match=what):
        ed.performGreedyIVARExperimentalDesign(cf, cand, 4)
    with pytest.raises(ValueError, match=what):
        ed.beginGreedyIVARExperimentalDesign(cf, cand, 4)
    with pytest.raises(ValueError, match=what):
        ed.scoreCandidatesIVAR(cf, cand[:3], cand)


def test_vector_gp_noise_without_noise_function_is_still_refused():
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space
    rng = np.random.default_rng(35)
    cand, mc = rng.uniform(-1, 1, (50, 2)), rng.uniform(-1, 1, (80, 2))
    cf = ed.costFunctionGP_IVAR(gpmod.GP(product_kernel("se_ard_2d_wide"), np.full(50, 1e-6)), 1, Space(2, None, None),
                                mcPoints=mc)
    with pytest.raises(NotImplementedError, match="scalar noise"):
        ed.performGreedyIVARExperimentalDesign(cf, cand, 4)


# ------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import _lib, engine
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space
    from gpexp_b200.device import Device
    ed.VERBOSE = False

    class NS:
        pass
    ns = NS()
    ns.ed, ns.lib, ns.check, ns.engine, ns.gp, ns.Space = ed, _lib.lib, _lib.check, engine, gpmod, Space
    ns.dev = Device.get(0)
    yield ns
    ns.check(ns.lib.gpx_set_ivar_core(ns.dev.h, I8), "gpx_set_ivar_core")


GPU_CASES = [("se_ard_2d_wide", nu_golden), ("matern_5d", nu_span), ("mehler_3d", nu_mehler)]
N_GPU = 12


@functools.lru_cache(maxsize=None)
def _reference_run(name):
    """C = 200 candidates, M = 2 000 integration points, 12 steps of the reference's loop (about 10 s each)."""
    nu = dict(GPU_CASES)[name]
    cand, mc = _sample(name, np.random.default_rng(36), 200, 2000)
    idx, costs = ref_greedy_ivar_nu(spec(name), cand, mc, N_GPU, nu)
    return cand, mc, idx, costs


LOOP_MODES = ["trace_i8", "trace_dmma", "trace_resident", "loop_i8", "loop_dmma", "resident", "one_kernel"]


@pytest.mark.gpu
@pytest.mark.parametrize("name,nu", GPU_CASES, ids=[n for n, _ in GPU_CASES])
def test_every_loop_mode_matches_reference(env, name, nu):
    ed = env.ed
    cand, mc, ref_idx, ref_costs = _reference_run(name)
    k = product_kernel(name)
    space = env.Space(spec(name).dim, None, None, noise=nu)
    # gp.noise is not used once the space carries a noise function (experimentalDesign.py:110-114)
    cf = ed.costFunctionGP_IVAR(env.gp.GP(k, 0.5), 1, space, mcPoints=mc)
    want = np.array([c[i] for c, i in zip(ref_costs, ref_idx)])
    launches = {}
    for mode in LOOP_MODES:
        env.check(env.lib.gpx_set_ivar_core(env.dev.h, DMMA if mode.endswith("dmma") else I8), "gpx_set_ivar_core")
        try:
            resident = mode in ("trace_resident", "resident", "one_kernel")
            eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, N_GPU, resident=resident)
            if mode.startswith("trace"):
                eng.score_trace = []
            if resident:
                eng.ONE_KERNEL_PAIRS = cand.shape[0] * mc.shape[0] if mode == "one_kernel" else 0
            l0 = env.dev.launches
            idx = eng.run(N_GPU)
            launches[mode] = env.dev.launches - l0
        finally:
            env.check(env.lib.gpx_set_ivar_core(env.dev.h, I8), "gpx_set_ivar_core")
        assert [int(i) for i in idx] == ref_idx, (name, mode)
        assert _rel(eng.pick_scores[:N_GPU].cpu().numpy(), want) <= 1e-9, (name, mode)
        if eng.score_trace is not None:
            for s, c in enumerate(eng.score_trace):
                assert _rel(c, ref_costs[s]) <= 1e-9, (name, mode, s)
    assert launches["one_kernel"] < launches["resident"], launches   # the cooperative kernel ran the loop
    # the public driver: each pick's cost is the golden-pinned cost function of the design up to that pick
    idx = ed.performGreedyIVARExperimentalDesign(cf, cand, N_GPU, returnIndices=True)
    assert [int(i) for i in idx] == ref_idx
    design = cand[ref_idx]
    nu_d = nu(design)
    ks = spec(name)
    for i in range(N_GPU):
        one = ed.costFunctionGP_IVAR(env.gp.GP(k, 0.5), i + 1, space, mcPoints=mc).evaluate(design[: i + 1])
        assert abs(cf.lastScores[i] - one) <= 1e-9 * abs(one), (name, i)
        # the pivot of step i is var_D(p) + nu(p) of the pick
        var = ks.prior(design[:1])[0] if i == 0 else \
            orc.fast_posterior_variance(ks, design[:i], design[i:i + 1], nu_d[:i])[0]
        assert abs(cf.lastPivots[i] - (var + nu_d[i])) <= 1e-9 * (var + nu_d[i]), (name, i)
    assert cf.illConditionedFrom is None


@pytest.mark.gpu
def test_constant_noise_function_equals_scalar_noise(env):
    ed = env.ed
    rng = np.random.default_rng(37)
    cand, mc = rng.uniform(-1, 1, (1500, 2)), rng.uniform(-1, 1, (2000, 2))
    k, s2, N = product_kernel("se_ard_2d_wide"), 1e-4, 20
    cf_s = ed.costFunctionGP_IVAR(env.gp.GP(k, s2), 1, env.Space(2, None, None), mcPoints=mc)
    cf_h = ed.costFunctionGP_IVAR(env.gp.GP(k, s2), 1, env.Space(2, None, None, noise=lambda p: np.full(p.shape[0], s2)),
                                  mcPoints=mc)
    for resident in (False, True):
        a = ed.performGreedyIVARExperimentalDesign(cf_s, cand, N, returnIndices=True, resident=resident)
        b = ed.performGreedyIVARExperimentalDesign(cf_h, cand, N, returnIndices=True, resident=resident)
        assert np.array_equal(a, b), resident
        # var_D + s2 is rounded once at set-up instead of at every scoring: the last bits may differ
        assert _rel(cf_h.lastScores, cf_s.lastScores) <= 1e-13, resident
    traces = []
    for cf in (cf_s, cf_h):
        eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, N, resident=False)
        eng.score_trace = []
        eng.run(N)
        traces.append(eng.score_trace)
    for s, (x, y) in enumerate(zip(*traces)):
        assert _rel(y, x) <= 1e-13, s


@pytest.mark.gpu
def test_varying_noise_changes_the_design(env):
    """Against the scalar run at the same mean noise, the design moves: nu is not ignored."""
    ed = env.ed
    rng = np.random.default_rng(38)
    cand, mc = rng.uniform(-1, 1, (1000, 2)), rng.uniform(-1, 1, (1500, 2))
    k, ks, N = product_kernel("se_ard_2d_wide"), spec("se_ard_2d_wide"), 16

    def nu(p):
        return 0.1 * (1.0 + p[:, 0]) ** 2   # 0 at x0 = -1, 0.4 at x0 = 1

    mean = float(np.mean(nu(cand)))
    cf_h = ed.costFunctionGP_IVAR(env.gp.GP(k, mean), 1, env.Space(2, None, None, noise=nu), mcPoints=mc)
    cf_s = ed.costFunctionGP_IVAR(env.gp.GP(k, mean), 1, env.Space(2, None, None), mcPoints=mc)
    h = [int(i) for i in ed.performGreedyIVARExperimentalDesign(cf_h, cand, N, returnIndices=True)]
    s = [int(i) for i in ed.performGreedyIVARExperimentalDesign(cf_s, cand, N, returnIndices=True)]
    assert h == fast_greedy_ivar_nu(ks, cand, mc, N, nu(cand))[0]
    assert s == orc.fast_greedy_ivar(ks, cand, mc, N, mean)[0]
    assert h != s


@pytest.mark.gpu
def test_zero_noise_half_domain_follows_the_pinv_rule(env):
    """Re-scoring a picked candidate: where nu = 0 the Gram of design + [p] is singular and pinv drops the repeated node
    (reduction 0, the cost of the design itself); where nu > 0 the repeated measurement still reduces the variance."""
    ed = env.ed
    rng = np.random.default_rng(39)
    cand, mc = rng.uniform(-1, 1, (60, 2)), rng.uniform(-1, 1, (400, 2))
    ks, k, N = spec("se_ard_2d_wide"), product_kernel("se_ard_2d_wide"), 10
    ref_idx, ref_costs = ref_greedy_ivar_nu(ks, cand, mc, N, nu_half_zero)
    cf = ed.costFunctionGP_IVAR(env.gp.GP(k, 1e-6), 1, env.Space(2, None, None, noise=nu_half_zero), mcPoints=mc)
    eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, N, resident=False)
    eng.score_trace = []
    assert [int(i) for i in eng.run(N)] == ref_idx
    nu = nu_half_zero(cand)
    seen_zero = seen_pos = False
    for s in range(1, N):
        got = eng.score_trace[s]
        assert _rel(got, ref_costs[s]) <= 1e-9, s
        design = cand[ref_idx[:s]]
        base = orc.ref_ivar_cost(ks, design, mc, nu_half_zero(design))
        for p in ref_idx[:s]:
            if nu[p] == 0.0:
                seen_zero = True
                assert abs(got[p] - base) <= 1e-9 * base and abs(ref_costs[s][p] - base) <= 1e-9 * base, (s, p)
            else:
                seen_pos = True
                assert got[p] < base * (1 - 1e-9), (s, p)
    assert seen_zero and seen_pos


@pytest.mark.gpu
def test_score_candidates_with_noise_function(env):
    ed = env.ed
    rng = np.random.default_rng(40)
    name, nu = "matern_5d", nu_span
    ks, k = spec(name), product_kernel(name)
    cand, mc, design = _sample(name, rng, 3000, 2000, 30)
    cf = ed.costFunctionGP_IVAR(env.gp.GP(k, 0.5), 1, env.Space(5, None, None, noise=nu), mcPoints=mc)
    costs, best = ed.scoreCandidatesIVAR(cf, design, cand)
    # arg-min of the vectorised restatement over all candidates
    from scipy.linalg import solve_triangular
    low = np.linalg.cholesky(ks.gram(design, design) + np.diag(nu(design)))
    w_m, w_c = solve_triangular(low, ks.gram(design, mc), lower=True), solve_triangular(low, ks.gram(design, cand), lower=True)
    var_m, var_c = ks.prior(mc) - np.sum(w_m ** 2, axis=0), ks.prior(cand) - np.sum(w_c ** 2, axis=0)
    fast = orc.fast_ivar_scores(ks, cand, mc, w_m, var_m, w_c, var_c, nu(cand))
    assert best == int(np.argmin(fast))
    assert _rel(costs, fast) <= 1e-9
    sample = np.concatenate([[best], rng.permutation(cand.shape[0])[:49]])
    for c in sample:
        pts = np.vstack([design, cand[c:c + 1]])
        ref = orc.ref_ivar_cost(ks, pts, mc, nu(pts))
        assert abs(costs[c] - ref) <= 1e-9 * ref, c


@pytest.mark.gpu
def test_mid_size_matches_fast_oracle(env):
    """20 000 candidates, 64 steps, cfg-2's kernel.  The numpy oracle re-evaluates K(M, C) at every step (10-30 ns per
    pair and step on one core), so the integration points are kept to 1 500."""
    ed = env.ed
    rng = np.random.default_rng(41)
    C, M, N = 20_000, 1500, 64
    cand, mc = rng.uniform(-1, 1, (C, 2)), rng.uniform(-1, 1, (M, 2))
    ks, k = spec("se_ard_2d"), product_kernel("se_ard_2d")
    ref, costs = fast_greedy_ivar_nu(ks, cand, mc, N, nu_golden(cand))
    want = np.array([c[i] for c, i in zip(costs, ref)])
    cf = ed.costFunctionGP_IVAR(env.gp.GP(k, 1e-6), 1, env.Space(2, None, None, noise=nu_golden), mcPoints=mc)
    for resident in (False, True):
        idx = ed.performGreedyIVARExperimentalDesign(cf, cand, N, returnIndices=True, resident=resident)
        assert [int(i) for i in idx] == ref, resident
        assert _rel(cf.lastScores, want) <= 1e-9, resident
