"""Import the UNMODIFIED reference (facebookresearch/vggsfm) with stub third-party modules -- TEST INFRASTRUCTURE ONLY.

Used by the golden generators under tools/ to produce the fixtures in tests/golden/ from a checkout of the reference
named by the VGGSFM_REFERENCE environment variable.  The test suite, smoke() and bench.py never call this module: they
compare against the stored fixtures.
Recipe: SURVEY.md Appendix C.
"""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("VGGSFM_REFERENCE", "")


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "vggsfm"))


class _Stub(types.ModuleType):
    def __getattr__(self, k):
        if k.startswith("__"):
            raise AttributeError(k)
        m = _Stub(self.__name__ + "." + k)
        setattr(self, k, m)
        return m

    def __call__(self, *a, **kw):
        raise RuntimeError("stub called: " + self.__name__)


_STUBS = ["hydra", "hydra.utils", "pycolmap", "pyceres", "kornia", "kornia.core", "kornia.core.check",
          "kornia.geometry", "kornia.geometry.conversions", "kornia.geometry.linalg", "kornia.geometry.solvers",
          "kornia.geometry.epipolar", "kornia.geometry.epipolar.fundamental", "kornia.geometry.homography",
          "kornia.geometry.calibration", "kornia.geometry.calibration.pnp", "kornia.geometry.subpix",
          "kornia.utils", "kornia.utils._compat", "kornia.utils.grid"]


def install():
    """Put the reference on sys.path with stubs for the absent third-party packages."""
    if not available():
        raise RuntimeError("set VGGSFM_REFERENCE to a checkout of facebookresearch/vggsfm")
    import torch
    for name in _STUBS:
        sys.modules.setdefault(name, _Stub(name))
    sys.modules["kornia.core"].Tensor = torch.Tensor
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


def contiguous_tracks(tn):
    """torch>=2.2 workaround for vggsfm/utils/triangulation.py:817-819 (caller side, no reference edit)."""
    return tn.transpose(0, 1).contiguous().transpose(0, 1)
