"""lsqfit_b200 -- B200-native batched Levenberg-Marquardt engine behind lsqfit's ``fitter=`` seam.

Scope: ONE hot path of gplepage/lsqfit, rebuilt as hand-written sm_100a CUDA behind a C ABI
(include/b200lm.h):   whiten -> residual + Jacobian -> trust-region LM -> fit.p propagation,
batched over thousands to millions of independent fits.  See DESIGN.md / INTEGRATION.md.

There is no CPU fallback: importing this package without the built extension raises, and
creating a plan without a CUDA device raises.
"""
from . import _cabi                                    # noqa: F401  (fails loudly if the .so is missing)
from ._cabi import B200LMError
from .functors import Functor, FAMILY, NIST_FORM
from .user_functor import cuda_functor, UserFunctor
from .engine import Plan, BatchResult, STOPPING_CRITERION, normalize_tol
from .whiten import PDF, cov_blocks
from .fitter import b200_lm, ChivSpec, DeviceChiv
from .fit import nonlinear_fit, gammaQ, BatchFits, FitView, wavg, WAvg
from .dense import DenseFit
from .bootstrap import bootstrap_means, normals
from .multifit import MultiFitter, FunctorModel, SharedExpModel, ChainedFit

__version__ = "0.1.0"


def available():
    """[(family id, np, nx, name)] of the compiled device functors."""
    return _cabi.functor_table()


def register(lsqfit_module=None):
    """Install the engine into a real ``lsqfit`` (needs lsqfit + gvar importable).

    * adds ``'b200_lm'`` to ``lsqfit.nonlinear_fit.FITTERS`` (reference
      src/lsqfit/__init__.py:110-128, 453);
    * wraps ``lsqfit._build_chiv_chivw`` (bound at :2074, called at :571) so that the
      ``chiv`` object handed to the fitter carries a ``b200`` ChivSpec when ``fcn`` is a
      ``lsqfit_b200.Functor``.
    ``bootstrapped_fit_iter``, ``simulated_fit_iter`` and ``MultiFitter`` then run unchanged
    with ``fitter='b200_lm'``.  See INTEGRATION.md for the binding details.
    """
    if lsqfit_module is None:
        import lsqfit as lsqfit_module           # raises ImportError when absent
    from ._lsqfit_hook import install
    return install(lsqfit_module)
