"""``from probaforms_b200.models import RealNVP`` mirrors ``from probaforms.models import RealNVP``
(reference probaforms/models/__init__.py:1); ``ConditionalNormal`` and ``CVAE`` likewise mirror ``probaforms.models.ConditionalNormal`` and ``probaforms.models.CVAE``."""
from .interfaces import GenModel
from .nflow import InvertibleLayer, NormalizingFlow
from .realnvp import RealNVP, RealNVPLayer, gen_network
from .cnormal import ConditionalNormal
from .cvae import CVAE

__all__ = ["RealNVP", "ConditionalNormal", "CVAE", "RealNVPLayer", "NormalizingFlow", "InvertibleLayer", "GenModel", "gen_network"]
