"""Drop-in replacement for the reference's `apla` package (src/apla/__init__.py): same module names, class
names and helper signatures, backed by the sm_100a kernels of libapla_b200.so."""
from .appla_attn import APLA_Attention
from .appla_attn_mem_eff import APLA_MemEffAttention
from .apla_vit import build_apla, replace_attn_with_apla
from .apla_block import FusedAplaBlock, attention_probabilities, fuse_apla_blocks
from .patch_embed import FusedPatchEmbed, cache_pos_encoding, fuse_patch_embed

__all__ = ["APLA_Attention", "APLA_MemEffAttention", "build_apla", "replace_attn_with_apla", "FusedAplaBlock",
           "fuse_apla_blocks", "attention_probabilities", "FusedPatchEmbed", "fuse_patch_embed", "cache_pos_encoding"]
