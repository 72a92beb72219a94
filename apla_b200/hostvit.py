"""Host ViT used by tests, smoke() and bench.py: a plain-PyTorch stand-in for the reference's timm/DINO-style
`VisionTransformer` (src/utils/transformers/vit.py:310-437, factories :511-596) and `Classifier`
(src/defaults/models.py:24-92).  The reference tree is not available on the GPU box, so the model the `apla`
package is dropped into has to live here.  It is NOT part of the accelerated path: the APLA modules and the
fused step engine replace its block arithmetic.

Contract kept with the reference so that checkpoints and golden vectors interchange:
  * same module / parameter names (`patch_embed.proj`, `cls_token`, `pos_embed`, `blocks.N.{norm1,attn,ls1,norm2,mlp,
    ls2}`, `norm`, `fc`) and the attributes `replace_attn_with_apla` reads from `block.attn`
    (`dim, num_heads, scale, qkv, proj, attn_drop.p, proj_drop.p`; src/apla/apla_vit.py:15-56);
  * same random-number consumption order on the global CPU generator (PatchEmbed conv, per block qkv/proj/fc1/fc2
    default Linear inits, trunc-normal pos_embed and cls_token, then a trunc-normal re-draw of every Linear in
    module order) -- verified bit-exactly against digests recorded from the reference in tests/golden/.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F


@dataclass
class VitArch:
    embed_dim: int
    depth: int
    num_heads: int
    mlp_ratio: float = 4.0
    qkv_bias: bool = True


ARCHS = {
    "vit_tiny": VitArch(192, 12, 3),
    "vit_small": VitArch(384, 12, 6),
    "vit_base": VitArch(768, 12, 12),
    "vit_large": VitArch(1024, 24, 16),
}


def _trunc_normal_(t: torch.Tensor, std: float) -> torch.Tensor:
    # inverse-CDF sampling of N(0, std) truncated to [-2, 2] (absolute bounds, as the reference uses)
    lo = 0.5 * (1.0 + math.erf(-2.0 / std / math.sqrt(2.0)))
    hi = 0.5 * (1.0 + math.erf(2.0 / std / math.sqrt(2.0)))
    with torch.no_grad():
        t.uniform_(2 * lo - 1, 2 * hi - 1).erfinv_().mul_(std * math.sqrt(2.0)).add_(0.0).clamp_(min=-2.0, max=2.0)
    return t


class SoftmaxAttention(nn.Module):
    """Stock multi-head attention with a fused qkv Linear; returns (out, attn) like the reference's."""

    def __init__(self, dim: int, num_heads: int, qkv_bias: bool, attn_drop: float = 0.0, proj_drop: float = 0.0):
        super().__init__()
        self.dim, self.num_heads = dim, num_heads
        self.scale = (dim // num_heads) ** -0.5
        self.qkv = nn.Linear(dim, 3 * dim, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)

    def forward(self, x):
        B, N, C = x.shape
        q, k, v = self.qkv(x).view(B, N, 3, self.num_heads, C // self.num_heads).permute(2, 0, 3, 1, 4)
        attn = self.attn_drop(torch.softmax((q @ k.transpose(-2, -1)) * self.scale, dim=-1))
        out = (attn @ v).transpose(1, 2).reshape(B, N, C)
        return self.proj_drop(self.proj(out)), attn


class FeedForward(nn.Module):
    def __init__(self, dim: int, hidden: int):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.act = nn.GELU()
        self.fc2 = nn.Linear(hidden, dim)

    def forward(self, x):
        return self.fc2(self.act(self.fc1(x)))


class ChannelScale(nn.Module):
    """LayerScale: per-channel learnable gain named `gamma`."""

    def __init__(self, dim: int, init: float):
        super().__init__()
        self.gamma = nn.Parameter(init * torch.ones(dim))

    def forward(self, x):
        return x * self.gamma


def drop_path(x, drop_prob: float = 0.0, training: bool = False):
    """Stochastic depth (vit.py drop_path): in training, every sample of the batch is kept with probability
    keep = 1 - drop_prob -- one draw per sample and call -- and the kept ones are scaled by 1 / keep."""
    if drop_prob == 0.0 or not training:
        return x
    keep = 1.0 - drop_prob
    mask = (keep + torch.rand((x.shape[0],) + (1,) * (x.ndim - 1), dtype=x.dtype, device=x.device)).floor_()
    return x.div(keep) * mask


class DropPath(nn.Module):
    def __init__(self, drop_prob: Optional[float] = None):
        super().__init__()
        self.drop_prob = drop_prob

    def forward(self, x):
        return drop_path(x, self.drop_prob, self.training)


class EncoderBlock(nn.Module):
    def __init__(self, dim: int, num_heads: int, mlp_ratio: float, qkv_bias: bool, eps: float,
                 layerscale: Optional[float], drop_path_rate: float = 0.0):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=eps)
        self.attn = SoftmaxAttention(dim, num_heads, qkv_bias)
        # one module for both branches, as the reference's Block: each call draws its own masks
        self.drop_path = DropPath(drop_path_rate) if drop_path_rate > 0.0 else nn.Identity()
        self.norm2 = nn.LayerNorm(dim, eps=eps)
        self.mlp = FeedForward(dim, int(dim * mlp_ratio))
        self.ls1 = ChannelScale(dim, layerscale) if layerscale is not None else nn.Identity()
        self.ls2 = ChannelScale(dim, layerscale) if layerscale is not None else nn.Identity()

    def forward(self, x):
        y = self.attn(self.norm1(x))
        y = y[0] if isinstance(y, tuple) else y
        x = x + self.drop_path(self.ls1(y))
        return x + self.drop_path(self.ls2(self.mlp(self.norm2(x))))


class PatchProjection(nn.Module):
    def __init__(self, img_size: int, patch: int, dim: int):
        super().__init__()
        self.img_size, self.patch_size = img_size, patch
        self.num_patches = (img_size // patch) ** 2
        self.proj = nn.Conv2d(3, dim, kernel_size=patch, stride=patch)

    def forward(self, x):
        return self.proj(x).flatten(2).transpose(1, 2)


class HostViT(nn.Module):
    def __init__(self, arch: VitArch, img_size: int = 518, patch_size: int = 14, layerscale: Optional[float] = 1.0,
                 eps: float = 1e-6, drop_path_rate: float = 0.0):
        super().__init__()
        D = arch.embed_dim
        self.arch = arch
        self.num_features = self.embed_dim = D
        self.patch_embed = PatchProjection(img_size, patch_size, D)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, D))
        self.pos_embed = nn.Parameter(torch.zeros(1, self.patch_embed.num_patches + 1, D))
        # stochastic depth rising linearly over depth (vit.py: dpr = linspace(0, drop_path_rate, depth)); no RNG drawn
        dpr = [float(p) for p in torch.linspace(0, drop_path_rate, arch.depth)]
        self.blocks = nn.ModuleList(
            [EncoderBlock(D, arch.num_heads, arch.mlp_ratio, arch.qkv_bias, eps, layerscale, dpr[i])
             for i in range(arch.depth)])
        self.norm = nn.LayerNorm(D, eps=eps)
        self.fc = nn.Identity()
        _trunc_normal_(self.pos_embed, 0.02)
        _trunc_normal_(self.cls_token, 0.02)
        for m in self.modules():        # same traversal order as nn.Module.apply for Linear leaves
            if isinstance(m, nn.Linear):
                _trunc_normal_(m.weight, 0.02)
                if m.bias is not None:
                    nn.init.zeros_(m.bias)
            elif isinstance(m, nn.LayerNorm):
                nn.init.ones_(m.weight)
                nn.init.zeros_(m.bias)

    def pos_for(self, npatch: int) -> torch.Tensor:
        """Position table for an `npatch`-patch grid: bicubic resize of the stored table when the grid differs."""
        table = self.pos_embed
        n0 = table.shape[1] - 1
        if npatch == n0:
            return table
        D = table.shape[-1]
        s = int(math.sqrt(n0))
        grid = table[:, 1:].reshape(1, s, s, D).permute(0, 3, 1, 2)
        grid = F.interpolate(grid, scale_factor=math.sqrt(npatch / n0), mode="bicubic", align_corners=False,
                             recompute_scale_factor=False)
        return torch.cat((table[:, :1], grid.permute(0, 2, 3, 1).reshape(1, -1, D)), dim=1)

    def tokens(self, images):
        x = self.patch_embed(images)
        x = torch.cat((self.cls_token.expand(x.shape[0], -1, -1), x), dim=1)
        return x + self.pos_for(x.shape[1] - 1)

    def forward_features(self, images):
        x = self.tokens(images)
        for blk in self.blocks:
            x = blk(x)
        return self.norm(x)[:, 0]

    def forward(self, images):
        return self.fc(self.forward_features(images))


class HostClassifier(nn.Module):
    """backbone (+APLA) + linear head, the structure `Classifier` builds (src/defaults/models.py:39-65)."""

    def __init__(self, backbone: HostViT, n_classes: int):
        super().__init__()
        self.backbone = backbone
        self.backbone.fc = nn.Identity()
        self.fc = nn.Linear(backbone.num_features, n_classes)

    def forward(self, images):
        return self.fc(self.backbone(images))


def build_classifier(arch: str, *, img_size: int, patch_size: int, n_classes: int, apla_config, is_multi_gpu=False,
                     attn_class: str = "apla_attn", layerscale: Optional[float] = 1.0, seed: Optional[int] = 0,
                     drop_path_rate: float = 0.0):
    """Construct backbone -> build_apla -> head in the reference's order (models.py:39-65) on the CPU generator.
    `drop_path_rate` is the reference's --dpr; it changes no weight."""
    from .apla.apla_vit import build_apla
    if seed is not None:
        torch.manual_seed(seed)
    a = ARCHS[arch] if isinstance(arch, str) else arch
    vit = HostViT(a, img_size=img_size, patch_size=patch_size, layerscale=layerscale, drop_path_rate=drop_path_rate)
    vit = build_apla(apla_config, vit, attn_class, is_multi_gpu=is_multi_gpu)
    return HostClassifier(vit, n_classes)
