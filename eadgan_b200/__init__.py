"""eadgan_b200 -- B200-native (sm_100a) implementation of EAD-GAN's adversarial training
step behind the reference's own torch.nn / torch.optim surface.  See DESIGN.md."""
from . import functional, nn, optim  # noqa: F401
from .frozen import freeze  # noqa: F401
from .patch import patch, unpatch  # noqa: F401

__version__ = "0.1.0"
