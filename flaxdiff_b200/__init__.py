"""flaxdiff_b200 - a B200-native (sm_100a) diffusion training / sampling engine with the
flaxdiff.schedulers / predictors / samplers / trainer / models.simple_unet.Unet API surface.

Host code is Python (PyTorch tensors as the container); all image- and activation-sized
arithmetic runs in the hand-written CUDA kernels of libfdx.so (include/fdx.h).  There is no
CPU or eager fallback: ops raise if the library is missing or tensors are not on a GPU.
"""
__version__ = "0.1.0"
