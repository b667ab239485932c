"""``from probaforms_b200.models import RealNVP`` mirrors ``from probaforms.models import RealNVP``
(reference probaforms/models/__init__.py:1); ``ConditionalNormal``, ``CVAE`` and ``ConditionalWGAN`` likewise mirror ``probaforms.models.ConditionalNormal``,
``probaforms.models.CVAE`` and ``probaforms.models.ConditionalWGAN``."""
from .interfaces import GenModel
from .nflow import InvertibleLayer, NormalizingFlow
from .realnvp import RealNVP, RealNVPLayer, gen_network
from .cnormal import ConditionalNormal
from .cvae import CVAE
from .wgan import ConditionalWGAN, Generator, Discriminator

__all__ = ["RealNVP", "ConditionalNormal", "CVAE", "ConditionalWGAN", "Generator", "Discriminator", "RealNVPLayer", "NormalizingFlow", "InvertibleLayer", "GenModel", "gen_network"]
