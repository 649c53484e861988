"""tblup_b200: B200-native (sm_100a) GBLUP fitness evaluation behind the evaluator interface of
ianwhale/tblup (tblup/evaluator.py).  Python here is host-side plumbing over the C-ABI library
``libtblup_b200.so``; the arithmetic runs in hand-written CUDA kernels (tblup_b200/csrc)."""
from .engine import GblupEngine, MODE_AUTO, MODE_GBLUP, MODE_SNPBLUP  # noqa: F401
from .model import PanelModel  # noqa: F401
from .reml import H2Estimate  # noqa: F401

__all__ = ["GblupEngine", "MODE_AUTO", "MODE_GBLUP", "MODE_SNPBLUP", "PanelModel", "H2Estimate"]
