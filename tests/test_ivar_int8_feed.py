"""How the INT8 IVAR core feeds its tensor cores: 32-byte K chunks through a 4-stage operand ring and 10 stacked-slice
MMAs per K step (one A slice against up to four adjacent B slices, writing several diagonals at once).

The design sizes put K on both sides of the 32-byte chunk edges, and with 39 950 integration points each CTA walks
many M tiles (the last one partial), so the ring wraps across tile boundaries at every chunk count.  The candidate
counts give one partial tile (C = 40), a second tile holding one candidate (65) and an odd tile count (170).  The
design points are drawn apart from the candidates, so n can exceed C."""
import numpy as np
import pytest

DMMA, I8 = 1, 2
M = 39_950
NS = (1, 31, 32, 33, 63, 64, 65, 96, 97, 160, 255, 257, 1023)


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
@pytest.mark.parametrize("C", [40, 65, 170])
@pytest.mark.parametrize("family", ["se", "matern", "mehler"])
@pytest.mark.parametrize("diff", [False, True])
def test_i8_feed(env, C, family, diff):
    ed, _, K, gpmod, Space, dev, DesignFactor = env
    rng = np.random.default_rng(C)
    if family == "se":
        d, k, noise = 2, K.KernelSquaredExponential([0.06, 0.09], 1.0, 2), 1e-6
    elif family == "matern":
        d, k, noise = 3, K.KernelIsoMatern(0.4, 1.0, 3), 1e-4
    else:
        d, k, noise = 3, K.KernelMehlerND([0.9, 0.8, 0.7], 3), 1e-2
    draw = rng.standard_normal if family == "mehler" else (lambda shape: rng.uniform(-1, 1, shape))
    cand, mc = draw((C, d)), draw((M, d))
    dev.force_diff_form = diff
    try:
        cf = ed.costFunctionGP_IVAR(gpmod.GP(k, noise), 1, Space(d, None, None), mcPoints=mc)
        eng = ed.beginGreedyIVARExperimentalDesign(cf, cand, max(NS) + 1, resident=False)
        for n in NS:
            eng.load_design(DesignFactor(dev, dev.points(draw((n, d))), noise))
            b0 = _scores(env, eng, I8)[0]  # the first call after a load also prepares the prologue operands
            a, la = _scores(env, eng, DMMA)
            b, lb = _scores(env, eng, I8)
            assert lb == la + 2, (n, la, lb)  # the INT8 call ran its two slicing launches: the INT8 core scored it
            assert np.all(np.isfinite(b)), n
            assert np.array_equal(b, b0), n
            assert np.max(np.abs(a - b) / np.abs(a)) <= 1e-11, (C, family, diff, n)
    finally:
        dev.force_diff_form = False
