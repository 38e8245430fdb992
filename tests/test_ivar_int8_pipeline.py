"""The INT8 IVAR core's accumulator hand-off: each CTA walks 10-25 M tiles through the one set of TMEM accumulators,
which the epilogue hands back to the MMA issuer before it finishes each tile.  Seeded designs at n = 1 .. 257 cover
1-5 K chunks per tile and the operand ring wrapping across tile boundaries; the last M tile and the last candidate
tile are partial."""
import numpy as np
import pytest

DMMA, I8 = 1, 2
C, M = 300, 39_950  # 5 candidate tiles of 64; 313 M tiles of 128 (the last with 14 rows): 11 tiles per CTA on 148 SMs
NS = (1, 31, 32, 33, 64, 65, 160, 255, 256, 257)


@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; the product path has no CPU fallback")
    import gpexp_b200.experimentalDesign as ed
    from gpexp_b200 import _lib, kernels
    from gpexp_b200 import gp as gpmod
    from gpexp_b200.approximation import Space
    from gpexp_b200.device import Device
    from gpexp_b200.engine import DesignFactor
    ed.VERBOSE = False
    dev = Device.get(0)
    yield ed, _lib, kernels, gpmod, Space, dev, DesignFactor
    _lib.check(_lib.lib.gpx_set_ivar_core(dev.h, I8), "gpx_set_ivar_core")
    dev.force_diff_form = False


def _scores(env, eng, core):
    ed, _lib, _, _, _, dev, _ = env
    _lib.check(_lib.lib.gpx_set_ivar_core(dev.h, core), "gpx_set_ivar_core")
    try:
        l0 = dev.launches
        eng.score()
        launches = dev.launches - l0
    finally:
        _lib.check(_lib.lib.gpx_set_ivar_core(dev.h, I8), "gpx_set_ivar_core")
    return eng.scores[: eng.cand.n].cpu().numpy().copy(), launches


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["se", "matern", "mehler"])
@pytest.mark.parametrize("diff", [False, True])
def test_i8_many_tiles_per_cta(env, family, diff):
    ed, _, K, gpmod, Space, dev, DesignFactor = env
    rng = np.random.default_rng(11)
    if family == "se":
        cand, mc = rng.uniform(-1, 1, (C, 2)), rng.uniform(-1, 1, (M, 2))
        k, noise = K.KernelSquaredExponential([0.06, 0.09], 1.0, 2), 1e-6
    elif family == "matern":
        cand, mc = rng.uniform(-1, 1, (C, 3)), rng.uniform(-1, 1, (M, 3))
        k, noise = K.KernelIsoMatern(0.4, 1.0, 3), 1e-4
    else:
        cand, mc = rng.standard_normal((C, 3)), rng.standard_normal((M, 3))
        k, noise = K.KernelMehlerND([0.9, 0.8, 0.7], 3), 1e-2
    dev.force_diff_form = diff
    try:
        cf = ed.costFunctionGP_IVAR(gpmod.GP(k, noise), 1, Space(cand.shape[1], None, None), mcPoints=mc)
        eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, max(NS) + 1, resident=False)
        for n in NS:
            eng.load_design(DesignFactor(dev, dev.points(cand[rng.permutation(C)[:n]]), noise))
            b0 = _scores(env, eng, I8)[0]  # the first call after a load also prepares the prologue operands
            a, la = _scores(env, eng, DMMA)
            b, lb = _scores(env, eng, I8)
            assert lb == la + 2, (n, la, lb)  # the INT8 call ran its two slicing launches: the INT8 core scored it
            assert np.all(np.isfinite(b)), n
            assert np.array_equal(b, b0), n
            assert np.max(np.abs(a - b) / np.abs(a)) <= 1e-11, (family, diff, n)
    finally:
        dev.force_diff_form = False
