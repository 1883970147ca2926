"""B200-native (sm_100a) nanoGPT training / sampling step for char-level ABC music models.

Drop-in for the reference's nanoGPT/model.py call surface (GPT, GPTConfig, configure_optimizers, generate),
backed by hand-written CUDA kernels in libabcgpt.so (C ABI: include/abcgpt.h).  Importing the package does not
need a GPU; constructing tensors on / calling the model on anything but a CUDA device raises.
"""
from .model import GPT, GPTConfig  # noqa: F401
from .optim import FusedAdamW  # noqa: F401
from .ddp import DDP, TunesFormerDDP  # noqa: F401
from .data import DeviceTokenStream  # noqa: F401
from .tunesformer import Patchilizer, TunesFormerShaped, pack_tunes  # noqa: F401


def clip_grad_norm_(model, max_norm):
    """Fused replacement for torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm) (train.py:352)."""
    return model.clip_grad_norm_(max_norm)
