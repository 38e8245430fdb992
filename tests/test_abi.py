"""CPU-side checks of the drop-in boundary: the shared library loads without a GPU, exports every
symbol include/gpexp_b200.h declares, the ctypes table matches the header, and the product path
fails loudly (no CPU fallback) when there is no device."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    text = open(os.path.join(ROOT, "include", "gpexp_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    decls = re.findall(r"\b(?:int|int64_t|const char\*)\s+(gpx_\w+)\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    return {name: [a.strip() for a in args.split(",") if a.strip() and a.strip() != "void"] for name, args in decls}


def test_library_exports_every_declared_symbol():
    from gpexp_b200 import _lib
    funcs = header_functions()
    assert len(funcs) >= 30
    for name in funcs:
        assert hasattr(_lib.lib, name), f"{name} declared in the header but not exported"
    assert _lib.lib.gpx_version() == _lib.GPX_VERSION == 200


def test_ctypes_table_matches_header():
    from gpexp_b200 import _lib
    funcs = header_functions()
    assert set(funcs) == set(_lib.SIGNATURES), set(funcs) ^ set(_lib.SIGNATURES)
    for name, args in funcs.items():
        assert len(args) == len(_lib.SIGNATURES[name]), (name, args)


def test_constants_match_header():
    from gpexp_b200 import _lib
    text = open(os.path.join(ROOT, "include", "gpexp_b200.h")).read()
    defs = dict(re.findall(r"#define\s+(GPX_\w+)\s+(\(?-?\d+\)?)", text))
    val = lambda k: int(defs[k].strip("()"))  # noqa: E731
    assert val("GPX_MAX_DIM") == _lib.GPX_MAX_DIM and val("GPX_KROWS") == _lib.GPX_KROWS
    assert (val("GPX_SE"), val("GPX_MATERN32"), val("GPX_MEHLER")) == (_lib.SE, _lib.MATERN32, _lib.MEHLER)
    assert (val("GPX_SIDE_A"), val("GPX_SIDE_B")) == (_lib.SIDE_A, _lib.SIDE_B)
    assert (val("GPX_ROW_KERNEL"), val("GPX_ROW_MATRIX")) == (_lib.ROW_KERNEL, _lib.ROW_MATRIX)
    assert _lib.GPX_PIVOT_HDR == 3 + _lib.GPX_MAX_DIM


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("this check is for the CPU-only container")
    from gpexp_b200 import kernels
    from gpexp_b200._lib import GpxError
    k = kernels.KernelSquaredExponential([0.1], 1.0, 2)
    with pytest.raises(GpxError):
        k.evaluate(np.zeros((3, 2)), np.zeros((3, 2)))
    import ctypes as C
    from gpexp_b200 import _lib
    h = C.c_void_p()
    rc = _lib.lib.gpx_create(0, C.byref(h))
    assert rc != 0 and h.value is None
    assert "no CPU fallback" in _lib.last_error() or "CUDA" in _lib.last_error()


def test_product_never_imports_oracle():
    bad = []
    for dirpath, _, files in os.walk(os.path.join(ROOT, "gpexp_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M) or "/root/reference" in src:
                    bad.append(f)
    assert not bad, bad


def test_api_surface_matches_reference_names():
    """Class / function names, constructor signatures and hyperParam keys of the reference."""
    import inspect
    from gpexp_b200 import experimentalDesign as ed, gp, kernels, gp_kernel_utilities as gku
    from gpexp_b200.approximation import Space
    k = kernels.KernelSquaredExponential([0.3], 2.0, 3)
    assert k.hyperParam == {'cl0': 0.3, 'cl1': 0.3, 'cl2': 0.3, 'signalSize': 2.0} and k.dimension == 3
    assert kernels.KernelIsoMatern(0.7, 1.5, 4).hyperParam == {'rho': 0.7, 'signalSize': 1.5}
    m = kernels.KernelMehlerND([0.1, 0.2], 2)
    assert m.hyperParam == {0: 0.1, 1: 0.2} and len(m.oneDKern) == 2
    m.updateHyperParameters({0: 0.3, 1: 0.4})
    assert m.oneDKern[1].hyperParam == {'t': 0.4} and m._gpx_spec()[2] == [0.3, 0.4]
    with pytest.raises(AssertionError):
        kernels.KernelMehler1D(0.5, 2)
    with pytest.raises(AssertionError):
        k.updateHyperParameters({'bogus': 1.0})
    assert list(inspect.signature(ed.performGreedyVarExperimentalDesign).parameters)[:6] == \
        ['kernel', 'mcPoints', 'nPoints', 'dimension', 'weights', 'indKeepStart']
    # reference signature + one trailing keyword extension (shard) for the column-sharded engine
    assert list(inspect.signature(ed.performGreedyMIExperimentalDesign).parameters)[:3] == ['costFuncMI', 'nPoints', 'start']
    assert list(inspect.signature(gku.calculateCovarianceMatrix).parameters) == ['kernel', 'points', 'nugget']
    assert list(inspect.signature(gp.GP.evaluateVariance).parameters) == ['self', 'newpt', 'parallel']
    assert list(inspect.signature(gp.GP.addNodesAndComputeCovariance).parameters) == ['self', 'nodes', 'noiseIn']
    assert list(inspect.signature(ed.costFunctionGP_MI.__init__).parameters) == \
        ['self', 'gaussianProcess', 'nInputs', 'space', 'nmc', 'mcpoints', 'square']
    s = Space(2, None, None)
    assert s.dimension == 2 and s.noiseFunc is None
    g = gp.GP(k, 1e-6)
    assert g.noise == 1e-6 and g.kernel is not k and g.pts is None and g.covarianceMatrix is None
    import gpexp_b200
    gpexp_b200.install_as_gpExp(False)  # standalone registration: the package's own modules answer to `gpExp`
    import gpExp.experimentalDesign as red
    assert red.costFunctionGP_IVAR is ed.costFunctionGP_IVAR
    for name in [m for m in list(__import__("sys").modules) if m == "gpExp" or m.startswith("gpExp.")]:
        del __import__("sys").modules[name]


def test_patch_reference_rebinds_only_hot_methods():
    """install_as_gpExp(path) with the reference importable keeps the reference's classes, constructors and optimiser loops
    and rebinds only the device methods (VERDICT r1: do not re-type reference host code)."""
    path = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(path, "gpExp")):
        pytest.skip("no reference package available (set GPEXP_REFERENCE and run __graft_entry__.build() to stage it)")
    import sys
    import gpexp_b200
    from gpexp_b200 import experimentalDesign as ed, gp, gp_kernel_utilities as gku, kernels
    ref = gpexp_b200.install_as_gpExp(path)
    try:
        import gpExp.experimentalDesign as red
        import gpExp.gp as rgp
        import gpExp.gp_kernel_utilities as rku
        import gpExp.kernels as rk
        assert ref.__gpexp_b200_patched__ and os.path.realpath(ref.__file__).startswith(os.path.realpath(path))
        for cls, methods in kernels.DEVICE_METHODS.items():
            for name, fn in methods.items():
                assert getattr(getattr(rk, cls), name) is fn
        assert rk.KernelSquaredExponential.__init__.__module__ == "gpExp.kernels"
        assert rk.KernelMehlerND.updateHyperParameters.__module__ == "gpExp.kernels"
        for name, fn in gp.DEVICE_METHODS.items():
            assert getattr(rgp.GP, name) is fn
        assert rgp.GP.__init__.__module__ == "gpExp.gp" and rgp.GP.findOptParamsLogLike.__module__ == "gpExp.gp"
        assert isinstance(rgp.GP.__dict__["covarianceMatrix"], property)
        assert rku.calculateCovarianceMatrix is gku.calculateCovarianceMatrix is rgp.calculateCovarianceMatrix
        assert red.costFunctionGP_IVAR.evaluate is ed.costFunctionGP_IVAR.evaluate
        assert red.costFunctionGP_IVAR.__init__.__module__ == "gpExp.experimentalDesign"
        assert red.performGreedyMIExperimentalDesign is ed.performGreedyMIExperimentalDesign
        for name in ("ExperimentalDesignDerivative", "ExperimentalDesignNoDerivative", "ExperimentalDesignGreedyWithDerivatives"):
            assert getattr(red, name).begin.__module__ == "gpExp.experimentalDesign"
        # constructing reference objects works without a device; the hot call then fails loudly (no CPU fallback)
        k = rk.KernelSquaredExponential([0.3], 2.0, 3)
        assert k.hyperParam['cl2'] == 0.3 and k._gpx_spec()[0] == 0
        g = rgp.GP(k, 1e-6)
        assert g.covarianceMatrix is None and g._pending is None
    finally:
        for name in [m for m in list(sys.modules) if m == "gpExp" or m.startswith("gpExp.")]:
            del sys.modules[name]


def test_host_logic_splits_and_scales():
    from gpexp_b200.engine import Shard, prior_scale
    from gpexp_b200 import _lib
    for n, w in [(10, 3), (7, 8), (1_000_000, 8), (5, 1)]:
        blocks = [Shard.split(n, w, r) for r in range(w)]
        assert blocks[0][0] == 0 and blocks[-1][1] == n
        assert all(blocks[i][1] == blocks[i + 1][0] for i in range(w - 1))
        sizes = [b - a for a, b in blocks]
        assert max(sizes) - min(sizes) <= 1
    # block-cyclic ownership of the MI factor columns: global g on rank (g // B) % world at ((g // B) // world) * B + g % B
    from gpexp_b200.engine import ShardedMIEngine
    for V, B, world in [(1000, 256, 3), (2048, 256, 8), (100, 256, 2), (5000, 512, 4)]:
        seen = np.zeros(V, dtype=int)
        for rank in range(world):
            cols = ShardedMIEngine.cyclic_columns(V, B, world, rank)
            seen[cols] += 1
            assert np.all(np.diff(cols) > 0)
            for loc in (0, len(cols) // 2, len(cols) - 1):
                if len(cols):
                    assert ShardedMIEngine.cyclic_local(int(cols[loc]), V, B, world, rank) == loc
            other = (rank + 1) % world
            if world > 1 and len(cols):
                assert ShardedMIEngine.cyclic_local(int(cols[0]), V, B, world, other) == -1
        assert np.all(seen == 1)
    assert prior_scale(_lib.SE, [0.1, 0.2, 3.0]) == 3.0
    assert prior_scale(_lib.MATERN32, [0.5, 2.0]) == 2.0
    assert abs(prior_scale(_lib.MEHLER, [0.6, 0.8]) - (1 / 0.8) * (1 / 0.6)) < 1e-15
