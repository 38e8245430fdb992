"""gpexp_b200 -- B200-native (sm_100a CUDA) implementation of the greedy experimental-design hot path of goroda/GPEXP behind
the reference's own Python API:

    gpexp_b200.kernels              <->  gpExp/kernels.py
    gpexp_b200.gp                   <->  gpExp/gp.py
    gpexp_b200.gp_kernel_utilities  <->  gpExp/gp_kernel_utilities.py
    gpexp_b200.experimentalDesign   <->  gpExp/experimentalDesign.py   (cost functions + greedy drivers)
    gpexp_b200.approximation        <->  gpExp/approximation.py        (Space)

`install_as_gpExp()` makes `import gpExp.*` run on the GPU path: when the reference package is importable it PATCHES it
(the reference keeps its constructors, optimiser loops, samplers; only the hot methods are rebound to the device
implementations); otherwise it registers this package's standalone modules under the name `gpExp`.
There is no CPU fallback.
"""
import importlib
import sys

__version__ = "0.2.0"


def patch_reference(ref):
    """Rebind the hot-path methods of an imported reference package `ref` (module `gpExp`) to the device implementations.

    Rebound (everything else stays the reference's own code):
      gpExp.kernels            Kernel.evaluate / evaluateF of every family, KernelSquaredExponential.derivative
      gpExp.gp_kernel_utilities calculateCovarianceMatrix, calculateCovarianceMatrixFITC, covTimesV,
                               calculateKernelBasisFunctionsMC
      gpExp.gp.GP              train, evaluate, addNodesAndComputeCovariance, evaluateVariance,
                               evaluateVarianceDerivative, computeLogLike, loglikeParams, covarianceMatrix / precisionMatrix
      gpExp.experimentalDesign costFunctionGP_IVAR.evaluate / derivative, costFunctionGP_MI.evaluate,
                               performGreedyVar / MI ExperimentalDesign (+ the new greedy-IVAR drivers: begin / perform /
                               refineGreedyIVARExperimentalDesign, scoreCandidatesIVAR; the exchange refinements
                               refineGreedyMI / Var ExperimentalDesign)
    Returns `ref`."""
    from . import experimentalDesign as ed, gp, gp_kernel_utilities as gku, kernels
    rk = importlib.import_module(ref.__name__ + ".kernels")
    rku = importlib.import_module(ref.__name__ + ".gp_kernel_utilities")
    rgp = importlib.import_module(ref.__name__ + ".gp")
    red = importlib.import_module(ref.__name__ + ".experimentalDesign")
    for cls_name, methods in kernels.DEVICE_METHODS.items():
        cls = getattr(rk, cls_name)
        for name, fn in methods.items():
            setattr(cls, name, fn)
    for name in ("calculateCovarianceMatrix", "calculateCovarianceMatrixFITC", "covTimesV", "calculateKernelBasisFunctionsMC"):
        setattr(rku, name, getattr(gku, name))
    # names the reference modules imported by value (gp.py:44, experimentalDesign.py imports)
    for mod in (rgp, red):
        if hasattr(mod, "calculateCovarianceMatrix"):
            mod.calculateCovarianceMatrix = gku.calculateCovarianceMatrix
    for name, obj in {**gp.DEVICE_ATTRS, **gp.DEVICE_METHODS}.items():
        setattr(rgp.GP, name, obj)
    for cls_name, methods in ed.DEVICE_METHODS.items():
        cls = getattr(red, cls_name)
        for name, fn in methods.items():
            setattr(cls, name, fn)
    for name, fn in ed.DEVICE_FUNCTIONS.items():
        setattr(red, name, fn)
    ref.__gpexp_b200_patched__ = True
    return ref


def install_as_gpExp(reference=None):
    """Make `import gpExp...` use the device path.

    reference : None  -> try `import gpExp` (the user's installed reference) and patch it; if it cannot be imported,
                         register this package's standalone modules as `gpExp`;
                a path -> directory that contains the reference's `gpExp/` package (put first on sys.path, then patched);
                False  -> standalone registration without looking for the reference."""
    if reference is not False:
        if isinstance(reference, str) and reference not in sys.path:
            sys.path.insert(0, reference)
        existing = sys.modules.get("gpExp")
        if existing is not None and getattr(existing, "__gpexp_b200_standalone__", False):
            for name in [m for m in sys.modules if m == "gpExp" or m.startswith("gpExp.")]:
                del sys.modules[name]
        try:
            ref = importlib.import_module("gpExp")
            return patch_reference(ref)
        except ImportError:
            if reference is not None:
                raise
    from . import approximation, experimentalDesign, gp, gp_kernel_utilities, kernels
    pkg = sys.modules[__name__]
    pkg.__gpexp_b200_standalone__ = True
    sys.modules["gpExp"] = pkg
    for name, mod in [("kernels", kernels), ("gp", gp), ("gp_kernel_utilities", gp_kernel_utilities),
                      ("experimentalDesign", experimentalDesign), ("approximation", approximation)]:
        sys.modules["gpExp." + name] = mod
    return pkg
