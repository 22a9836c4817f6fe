"""CUDA twin of the reference's PyTorch adapter package `pytorch_custom_op_ffi`
(examples/pytorch-custom-op-ffi/python/pytorch_custom_op_ffi/__init__.py): same public names, B200 underneath.

    from pytorch_custom_op_ffi import register_metal_sdpa_backend, use_metal_sdpa
    with use_metal_sdpa():
        out = torch.nn.functional.scaled_dot_product_attention(q, k, v, is_causal=True)   # CUDA tensors
"""
from .backend import (MetalSDPAContext, is_metal_sdpa_available, metal_sdpa_version, register_metal_sdpa_backend,
                      unregister_metal_sdpa_backend, use_metal_sdpa)
from .ext import metal_flash_attention_varlen, metal_flash_attention_with_kvcache

__version__ = "0.1.0"
__all__ = ["register_metal_sdpa_backend", "unregister_metal_sdpa_backend", "use_metal_sdpa", "is_metal_sdpa_available",
           "metal_sdpa_version", "MetalSDPAContext", "metal_flash_attention_varlen",
           "metal_flash_attention_with_kvcache"]
