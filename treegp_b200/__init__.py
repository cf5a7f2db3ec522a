"""treegp_b200 -- B200-native (sm_100a) implementation of treegp's Gaussian-process hot path.

Public names mirror /root/reference/treegp/__init__.py:23-36: ``GPInterpolation``, ``two_pcf`` and
``log_likelihood`` (the classes, as in the reference), the three treegp kernels and ``eval_kernel``.
All O(N^2)/O(N^3) arithmetic runs in hand-written CUDA behind the C ABI of include/treegp_b200.h;
there is no CPU fallback.
"""
from . import kernels as _k, log_likelihood as _ll, two_pcf as _tp, gp_interp as _gi, meanify as _mf, utils as _ut

AnisotropicRBF, AnisotropicVonKarman, VonKarman, eval_kernel = (
    _k.AnisotropicRBF, _k.AnisotropicVonKarman, _k.VonKarman, _k.eval_kernel)
GPInterpolation = _gi.GPInterpolation
from .gp_batch import GPInterpolationBatch  # noqa: E402  (extension: many small problems per device call)
# as in the reference, these two names are the classes (they shadow the sub-modules of the same name)
log_likelihood, two_pcf = _ll.log_likelihood, _tp.two_pcf
meanify = _mf.meanify
comp_eb, comp_eb_treecorr = _ut.comp_eb, _ut.comp_eb_treecorr
from .grf import sample_grf  # noqa: E402  (extension: device-side synthetic fields)

__version__ = "0.1.0"

__all__ = [
    "__version__",
    "GPInterpolation",
    "GPInterpolationBatch",
    "two_pcf",
    "log_likelihood",
    "AnisotropicRBF",
    "VonKarman",
    "AnisotropicVonKarman",
    "eval_kernel",
    "meanify",
    "comp_eb",
    "comp_eb_treecorr",
]
