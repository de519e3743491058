"""cnn_with_pde_b200 -- sm_100a implementation of the PDE block of MariMamgo/CNN-with-PDE.

One sub-module per reference script, exporting a class with the reference's name,
constructor signature, parameter names and state_dict layout; ``forward`` runs hand-written
CUDA kernels through the C ABI of ``libpde_b200.so`` (``include/pde_b200.h``)::

    from cnn_with_pde_b200.mnist_test import DiffusionLayer            # mnist_test.py:11
    from cnn_with_pde_b200.fashion_mnist import DiffusionLayer         # fashion_mnist.py:18
    from cnn_with_pde_b200.SVHN import DiffusionLayer                  # SVHN.py:12
    from cnn_with_pde_b200.cifar10 import EnhancedDiffusionLayer       # cifar10.py:24
    from cnn_with_pde_b200.cifar_2version import LearnableDiffusionLayer  # cifar_2version.py:20
    from cnn_with_pde_b200.emotion_recognition import PDELayer         # emotion_recognition.py:56
    from cnn_with_pde_b200.tiny_imagenet import ImprovedDiffusionLayer # tiny_imagenet.py:14

There is no CPU path: inputs must be CUDA float tensors and the library must be built
(``python cnn-with-pde_b200/build.py`` or ``__graft_entry__.build()``).
"""
from . import _cabi  # noqa: F401
from .functional import AdiConfig, EmoConfig, TinyConfig, adi_layer, emotion_layer, tiny_layer  # noqa: F401
from . import ops  # noqa: F401,E402  (registers the pde_b200:: custom ops that traced calls go through)
from . import mnist_test, fashion_mnist, SVHN, cifar10, cifar_2version, emotion_recognition, tiny_imagenet  # noqa: F401,E402

__all__ = ["mnist_test", "fashion_mnist", "SVHN", "cifar10", "cifar_2version", "emotion_recognition",
           "tiny_imagenet", "adi_layer", "emotion_layer", "tiny_layer", "AdiConfig", "EmoConfig", "TinyConfig"]
