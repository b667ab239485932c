"""``from probaforms_b200.models import RealNVP`` mirrors ``from probaforms.models import RealNVP``
(reference probaforms/models/__init__.py:1); ``ConditionalNormal`` likewise mirrors ``probaforms.models.ConditionalNormal``."""
from .interfaces import GenModel
from .nflow import InvertibleLayer, NormalizingFlow
from .realnvp import RealNVP, RealNVPLayer, gen_network
from .cnormal import ConditionalNormal

__all__ = ["RealNVP", "ConditionalNormal", "RealNVPLayer", "NormalizingFlow", "InvertibleLayer", "GenModel", "gen_network"]
