"""unetb200 -- host-side Python layer of the B200-native UNet hot path.

``_lib``        ctypes binding of libunetb200.so (C ABI: include/unetb200.h)
``ops``         tensor-level wrappers (pointer / shape / stream marshalling only)
``functional``  torch.autograd.Function per UNet part
``backward_pass`` what a backward pass owns outside autograd (deferred reductions, side stream, hand-offs)
``losses``      dice / boundary / fused CE+dice
``ddp``         data-parallel gradient all-reduce (NCCL) overlapped with backward
``graph``       whole-step CUDA graph
``optim``       fused clip_grad_norm_ + RMSprop
``eval_tail``   evaluate.py / predict.py tails on the device (argmax + class dice, resize + argmax)
``data``        uint8 input pipeline on the device (BasicDataset.preprocess + rotation augmentation)
"""
from . import _lib  # noqa: F401

__all__ = ["_lib", "ops", "functional", "backward_pass", "losses", "ddp", "graph", "optim", "eval_tail", "data"]
