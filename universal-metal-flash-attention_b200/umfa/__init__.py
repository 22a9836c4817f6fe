"""umfa -- numpy/ctypes adapter over libMFAFFI.so (B200 build); mirrors the reference's python-ffi package."""
from ._ffi import MFAError
from ._version import __version__
from .core import (MFABuffer, MFAContext, attention, flash_attention_backward, flash_attention_forward, flash_attention_kvcache,
                   flash_attention_varlen_backward, flash_attention_varlen_forward, quantize, quantized_attention,
                   runtime_quantized_attention, runtime_quantized_backward)
from .utils import create_context, get_version, is_device_available, is_metal_available, print_system_info

__all__ = ["MFAContext", "MFABuffer", "flash_attention_forward", "flash_attention_backward",
           "flash_attention_varlen_forward", "flash_attention_varlen_backward", "flash_attention_kvcache", "attention",
           "quantized_attention", "runtime_quantized_attention", "runtime_quantized_backward", "quantize", "MFAError",
           "create_context", "is_metal_available", "is_device_available", "get_version", "print_system_info",
           "__version__"]
