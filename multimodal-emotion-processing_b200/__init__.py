"""mmemo_b200 — B200-native (sm_100a) hot path of youngzhou97qz/Multimodal-emotion-processing.

Import as ``mmemo_b200`` (see ``mmemo_b200/__init__.py``).  Sub-modules mirror the reference
scripts: ``realformer`` (others/realformer.py), ``cmu_mosei`` (cmu-mosei/run.py), ``ren_mme``
(Ren-MME/run.py), ``rencecps`` (rencecps/run.py), ``robot_demo`` (robot_demo.py).  The CUDA
library is loaded lazily by ``mmemo_b200._lib`` on the first kernel call and raises if it is
missing: there is no CPU fallback.
"""
__version__ = "0.1.0"

from .blocks import get_precision, precision, set_precision  # noqa: E402,F401
from . import batching, cmu_mosei, ensemble, optim, realformer, ren_mme, rencecps, robot_demo, synth, trainer  # noqa: E402,F401
from . import folds  # noqa: E402,F401
from .encoder import ResidualEncoder  # noqa: E402,F401
