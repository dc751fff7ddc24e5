"""Drop-in replacement for the reference `networks/swinv2_global.py` (NERSC/swin_v2_weather).

Same public surface -- `swinv2net(params)`, `swin_from_yaml(fname)`, `SwinTransformerV2Cr(...)` with the
reference constructor signature (swinv2_global.py:683-711), `forward(x) -> (B, out_chans, H, W)`,
`forward_features`, `forward_head`, `set_grad_checkpointing` -- and the same `state_dict()` key tree,
shapes, dtypes and construction order (so the same torch seed yields the same initial weights and
existing `weights.tar` / `ckpt.tar` checkpoints load).  The sub-modules below are parameter containers
with the reference's names; the arithmetic is done by hand-written sm_100a kernels through
`swin_v2_weather_b200.functional` -- there is no PyTorch/CPU fallback for the forward pass.

Differences from the reference, all deliberate:
  * the shifted-window mask is generated inside the attention kernel; `block.attn_mask` is materialised
    on demand (bit-identical to the reference's non-persistent buffer) instead of being stored;
  * torch.roll / window_partition / window_reverse never run: they are folded into kernel addressing;
  * `compute_mode`: "bf16" (default; bf16 storage + tcgen05 GEMMs, fp32 residual stream/statistics) or
    "fp32" (validation mode).  Ambient torch autocast is ignored by the kernels;
  * when no gradient will be taken -- grad mode off (torch.no_grad / torch.inference_mode), or nothing a call reads
    requires grad -- PatchEmbed, the blocks and the head run forward-only: same kernels and bits, but nothing is kept
    for a backward (no fc1 pre-activation, no row statistics).  Like deterministic mode this follows torch's state;
    there is no option.
"""
from __future__ import annotations

import math
from types import SimpleNamespace
from typing import Any, List, Optional, Tuple, Type, Union

import torch
import torch.nn as nn
from torch.utils.checkpoint import checkpoint

from .. import functional as Fn
from .. import ops

_SHADOW_ATTR = "_swinb200_shadow"


def to_2tuple(x):
    if isinstance(x, (tuple, list)):
        return tuple(x)
    return (x, x)


def bchw_to_bhwc(x: torch.Tensor) -> torch.Tensor:
    return x.permute(0, 2, 3, 1)


def bhwc_to_bchw(x: torch.Tensor) -> torch.Tensor:
    return x.permute(0, 3, 1, 2)


def _carry_shadow(dst: torch.Tensor, shadow: Optional[torch.Tensor]) -> torch.Tensor:
    """Attach the activation-type copy of `dst` (written by the producing kernel) so the next block's
    first GEMM can read it instead of re-casting the fp32 stream."""
    if shadow is not None and shadow.numel() > 0:
        setattr(dst, _SHADOW_ATTR, shadow)
    return dst


def _forward_only(*tensors: Optional[torch.Tensor]) -> bool:
    """True when no gradient can be taken through a call reading `tensors` (inputs and parameters): grad mode is off, or
    none of them requires grad.  checkpoint(use_reentrant=False) runs (and re-runs) its forward with grad enabled, so
    checkpointed training keeps the training path."""
    if not torch.is_grad_enabled():
        return True
    return not any(t is not None and t.requires_grad for t in tensors)


def _shadow_of(x_bhwc: torch.Tensor, mode: ops.ComputeMode) -> torch.Tensor:
    B, H, W, C = x_bhwc.shape
    sh = getattr(x_bhwc, _SHADOW_ATTR, None)
    if sh is not None and sh.shape == (B * H * W, C) and sh.dtype == mode.act_dtype and sh.device == x_bhwc.device:
        return sh
    return ops.to_act(x_bhwc.detach().contiguous().view(B * H * W, C), mode)


def swin_from_yaml(fname, checkpoint_stages=False):
    """reference: swinv2_global.py:47-54 (PyYAML resolves the anchors/merge keys of config/swin.yaml)."""
    import yaml
    with open(fname) as f:
        hparams = yaml.safe_load(f)
    params = SimpleNamespace()
    for k, v in hparams.items():
        setattr(params, k, v)
    return swinv2net(params, checkpoint_stages=checkpoint_stages)


def swinv2net(params, checkpoint_stages=False):
    """reference: swinv2_global.py:57-74 -- same 13 hyper-parameters."""
    act_ckpt = checkpoint_stages or params.activation_ckpt
    return SwinTransformerV2Cr(
        img_size=params.img_size,
        patch_size=params.patch_size,
        depths=(params.depth,),
        num_heads=(params.num_heads,),
        in_chans=params.n_in_channels,
        out_chans=params.n_out_channels,
        embed_dim=params.embed_dim,
        img_window_ratio=params.window_ratio,
        drop_path_rate=params.drop_path_rate,
        full_pos_embed=params.full_pos_embed,
        rel_pos=params.rel_pos,
        mlp_ratio=params.mlp_ratio,
        checkpoint_stages=act_ckpt,
        residual=params.residual,
        compute_mode=getattr(params, "compute_mode", "bf16"),
    )


class DropPath(nn.Module):
    """Per-sample stochastic depth (timm.layers.DropPath semantics; reference call sites :378,388).
    Returns the (B,) multiplier -- the mask is drawn with the same torch op and shape (B,1,1[,1]) the
    reference uses, so a shared RNG state yields the same draws -- or None when inactive."""

    def __init__(self, drop_prob: float = 0.0, scale_by_keep: bool = True):
        super().__init__()
        self.drop_prob = drop_prob
        self.scale_by_keep = scale_by_keep

    def sample_scale(self, like: torch.Tensor, ndim: int) -> Optional[torch.Tensor]:
        if self.drop_prob == 0.0 or not self.training:
            return None
        keep = 1.0 - self.drop_prob
        mask = like.new_empty((like.shape[0],) + (1,) * (ndim - 1), dtype=torch.float32).bernoulli_(keep)
        if keep > 0.0 and self.scale_by_keep:
            mask.div_(keep)
        return mask.reshape(-1).contiguous()

    def extra_repr(self):
        return f"drop_prob={round(self.drop_prob, 3):0.3f}"


class Mlp(nn.Module):
    """Parameter container with timm.layers.Mlp's sub-module names (fc1/act/drop1/norm/fc2/drop2).
    The block MLP is executed by the fused GEMM kernels; only the tiny CPB meta-MLP calls forward()."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, norm_layer=None,
                 bias=True, drop=0.0):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        bias = to_2tuple(bias)
        drop = to_2tuple(drop)
        self.fc1 = nn.Linear(in_features, hidden_features, bias=bias[0])
        self.act = act_layer()
        self.drop1 = nn.Dropout(drop[0])
        self.norm = norm_layer(hidden_features) if norm_layer is not None else nn.Identity()
        self.fc2 = nn.Linear(hidden_features, out_features, bias=bias[1])
        self.drop2 = nn.Dropout(drop[1])

    def forward(self, x):
        return self.drop2(self.fc2(self.norm(self.drop1(self.act(self.fc1(x))))))


class WindowMultiHeadAttentionNoPos(nn.Module):
    """reference: swinv2_global.py:122-201.  Holds qkv / proj / logit_scale; computed by the fused kernels."""

    def __init__(self, dim: int, num_heads: int, window_size: Tuple[int, int], drop_attn: float = 0.0,
                 drop_proj: float = 0.0, sequential_attn: bool = False) -> None:
        super().__init__()
        assert dim % num_heads == 0, \
            "The number of input features (in_features) are not divisible by the number of heads (num_heads)."
        if drop_attn != 0.0 or drop_proj != 0.0:
            raise NotImplementedError("attention / projection dropout > 0 is not used by any reference config")
        self.in_features = dim
        self.window_size = window_size
        self.num_heads = num_heads
        self.sequential_attn = sequential_attn
        self.qkv = nn.Linear(in_features=dim, out_features=dim * 3, bias=True)
        self.attn_drop = nn.Dropout(drop_attn)
        self.proj = nn.Linear(in_features=dim, out_features=dim, bias=True)
        self.proj_drop = nn.Dropout(drop_proj)
        self.logit_scale = nn.Parameter(torch.log(10 * torch.ones(num_heads)))

    def update_input_size(self, new_window_size, **kwargs: Any) -> None:
        self.window_size = new_window_size

    def logit_scale_factor(self) -> torch.Tensor:
        """exp(min(logit_scale, ln 100)) -- reference :186 / :305 (autograd handles the clamp gate)."""
        return torch.clamp(self.logit_scale, max=math.log(1.0 / 0.01)).exp()

    def position_bias(self) -> Optional[torch.Tensor]:
        return None


class WindowMultiHeadAttention(WindowMultiHeadAttentionNoPos):
    """reference: swinv2_global.py:204-321 (continuous position bias variant, `rel_pos=True`).

    The (heads, L, L) bias table is produced by the *same torch ops* as the reference
    (`meta_mlp(relative_coordinates_log)`, :274-287) so it matches bit-exactly and keeps the hidden
    dropout(0.125) semantics; the attention kernels consume the table and return its gradient."""

    def __init__(self, dim: int, num_heads: int, window_size: Tuple[int, int], drop_attn: float = 0.0,
                 drop_proj: float = 0.0, meta_hidden_dim: int = 384, sequential_attn: bool = False) -> None:
        # NOTE construction order (qkv, proj, meta_mlp, logit_scale) matters for seed-identical init (:235-248)
        nn.Module.__init__(self)
        assert dim % num_heads == 0, \
            "The number of input features (in_features) are not divisible by the number of heads (num_heads)."
        if drop_attn != 0.0 or drop_proj != 0.0:
            raise NotImplementedError("attention / projection dropout > 0 is not used by any reference config")
        self.in_features = dim
        self.window_size = window_size
        self.num_heads = num_heads
        self.sequential_attn = sequential_attn
        self.qkv = nn.Linear(in_features=dim, out_features=dim * 3, bias=True)
        self.attn_drop = nn.Dropout(drop_attn)
        self.proj = nn.Linear(in_features=dim, out_features=dim, bias=True)
        self.proj_drop = nn.Dropout(drop_proj)
        self.meta_mlp = Mlp(2, hidden_features=meta_hidden_dim, out_features=num_heads, act_layer=nn.ReLU, drop=(0.125, 0.))
        self.logit_scale = nn.Parameter(torch.log(10 * torch.ones(num_heads)))
        self._make_pair_wise_relative_positions()

    def _make_pair_wise_relative_positions(self) -> None:
        device = self.logit_scale.device
        coordinates = torch.stack(torch.meshgrid([
            torch.arange(self.window_size[0], device=device),
            torch.arange(self.window_size[1], device=device)], indexing="ij"), dim=0).flatten(1)
        relative_coordinates = coordinates[:, :, None] - coordinates[:, None, :]
        relative_coordinates = relative_coordinates.permute(1, 2, 0).reshape(-1, 2).float()
        relative_coordinates_log = torch.sign(relative_coordinates) * torch.log(1.0 + relative_coordinates.abs())
        self.register_buffer("relative_coordinates_log", relative_coordinates_log, persistent=False)

    def update_input_size(self, new_window_size, **kwargs: Any) -> None:
        self.window_size = new_window_size
        self._make_pair_wise_relative_positions()

    def _relative_positional_encodings(self) -> torch.Tensor:
        window_area = self.window_size[0] * self.window_size[1]
        relative_position_bias = self.meta_mlp(self.relative_coordinates_log)
        relative_position_bias = relative_position_bias.transpose(1, 0).reshape(self.num_heads, window_area, window_area)
        return relative_position_bias.unsqueeze(0)

    def position_bias(self) -> Optional[torch.Tensor]:
        with torch.autocast(device_type=self.logit_scale.device.type, enabled=False):
            return self._relative_positional_encodings()[0].float()


class SwinTransformerV2CrBlock(nn.Module):
    """reference: swinv2_global.py:324-497."""

    def __init__(self, dim: int, num_heads: int, feat_size: Tuple[int, int], window_size: Tuple[int, int],
                 shift_size: Tuple[int, int] = (0, 0), mlp_ratio: float = 4.0, init_values: Optional[float] = 0,
                 proj_drop: float = 0.0, drop_attn: float = 0.0, drop_path: float = 0.0, extra_norm: bool = False,
                 sequential_attn: bool = False, norm_layer: Type[nn.Module] = nn.LayerNorm, rel_pos: bool = True,
                 compute_mode: str = "bf16") -> None:
        super().__init__()
        if norm_layer is not nn.LayerNorm:
            raise NotImplementedError("only nn.LayerNorm is supported (the reference never passes anything else)")
        if proj_drop != 0.0:
            raise NotImplementedError("proj_drop > 0 is not used by any reference config")
        self.dim = dim
        self.feat_size = feat_size
        self.target_shift_size = to_2tuple(shift_size)
        self.window_size, self.shift_size = self._calc_window_shift(to_2tuple(window_size))
        self.window_area = self.window_size[0] * self.window_size[1]
        self.init_values = init_values
        self.compute_mode = compute_mode
        window_attn_block = WindowMultiHeadAttention if rel_pos else WindowMultiHeadAttentionNoPos
        self.attn = window_attn_block(dim=dim, num_heads=num_heads, window_size=self.window_size, drop_attn=drop_attn,
                                      drop_proj=proj_drop, sequential_attn=sequential_attn)
        self.norm1 = norm_layer(dim)
        self.drop_path1 = DropPath(drop_prob=drop_path) if drop_path > 0.0 else nn.Identity()
        self.mlp = Mlp(in_features=dim, hidden_features=int(dim * mlp_ratio), drop=proj_drop, out_features=dim)
        self.norm2 = norm_layer(dim)
        self.drop_path2 = DropPath(drop_prob=drop_path) if drop_path > 0.0 else nn.Identity()
        self.norm3 = nn.Identity()
        self.init_weights()

    def _calc_window_shift(self, target_window_size):
        window_size = [f if f <= w else w for f, w in zip(self.feat_size, target_window_size)]
        shift_size = [0 if f <= w else s for f, w, s in zip(self.feat_size, window_size, self.target_shift_size)]
        return tuple(window_size), tuple(shift_size)

    @property
    def attn_mask(self) -> Optional[torch.Tensor]:
        """The reference's (nW, L, L) {0,-100} buffer (swinv2_global.py:403-424), materialised on demand by the
        same device predicate the attention kernels use.  None for un-shifted blocks."""
        if not any(self.shift_size):
            return None
        H, W = self.feat_size
        return ops.shift_mask(H, W, self.window_size[0], self.window_size[1], self.shift_size[0], self.shift_size[1],
                              self.norm1.weight.device)

    def init_weights(self):
        if self.init_values is not None:
            nn.init.constant_(self.norm1.weight, self.init_values)
            nn.init.constant_(self.norm2.weight, self.init_values)

    def update_input_size(self, new_window_size: Tuple[int, int], new_feat_size: Tuple[int, int]) -> None:
        self.feat_size = new_feat_size
        self.window_size, self.shift_size = self._calc_window_shift(to_2tuple(new_window_size))
        self.window_area = self.window_size[0] * self.window_size[1]
        self.attn.update_input_size(new_window_size=self.window_size)

    def _drop_scale(self, dp: nn.Module, x: torch.Tensor, ndim: int) -> Optional[torch.Tensor]:
        return dp.sample_scale(x, ndim) if isinstance(dp, DropPath) else None

    def forward(self, x: torch.Tensor, scale: Optional[torch.Tensor] = None) -> torch.Tensor:
        """x: (B, H, W, C) fp32 -> same (reference :480-497).  `scale`: optional pre-computed exp(min(logit_scale, ln 100))
        of this block (the stage computes it for all its blocks with three launches instead of two per block)."""
        mode = ops.MODES[self.compute_mode]
        B, H, W, C = x.shape
        if (H, W) != tuple(self.feat_size):
            raise AssertionError(f"token grid ({H},{W}) doesn't match the block's feat_size {self.feat_size}")
        x = x.float()
        xb = _shadow_of(x, mode)
        a = self.attn
        # RNG draws happen in the reference's order: CPB hidden dropout (inside attention), then DropPath of
        # branch 1 (mask shaped for a 4-d tensor), then DropPath of branch 2 (3-d tensor)
        bias = a.position_bias()
        dp1 = self._drop_scale(self.drop_path1, x, 4)
        dp2 = self._drop_scale(self.drop_path2, x, 3)
        geom = (a.num_heads, self.window_size[0], self.window_size[1], self.shift_size[0], self.shift_size[1])
        scale = (a.logit_scale_factor() if scale is None else scale).float()
        weights = (a.qkv.weight, a.qkv.bias, a.proj.weight, a.proj.bias, self.norm1.weight, self.norm1.bias, self.mlp.fc1.weight,
                   self.mlp.fc1.bias, self.mlp.fc2.weight, self.mlp.fc2.bias, self.norm2.weight, self.norm2.bias)
        if _forward_only(x, scale, bias, *weights):
            out, shadow = Fn.block_forward_only(x, xb, scale, bias, *weights, dp1, dp2, geom, mode)
        else:
            out, shadow = Fn.SwinBlockFn.apply(x, xb, scale, bias, *weights, dp1, dp2, geom, mode)
        return _carry_shadow(out, shadow)


class PatchEmbed(nn.Module):
    """reference: swinv2_global.py:526-546 (parameter container; computed inside SwinTransformerV2Cr.forward_features)."""

    def __init__(self, img_size=224, patch_size=16, in_chans=3, embed_dim=768, norm_layer=None):
        super().__init__()
        img_size = to_2tuple(img_size)
        patch_size = to_2tuple(patch_size)
        self.img_size = img_size
        self.patch_size = patch_size
        self.grid_size = (img_size[0] // patch_size[0], img_size[1] // patch_size[1])
        self.num_patches = self.grid_size[0] * self.grid_size[1]
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)
        self.norm = norm_layer(embed_dim) if norm_layer else nn.Identity()


class SwinTransformerV2CrStage(nn.Module):
    """reference: swinv2_global.py:549-655 (single resolution; the reference always passes downscale=False)."""

    def __init__(self, embed_dim: int, depth: int, downscale: bool, num_heads: int, feat_size: Tuple[int, int],
                 window_size: Tuple[int, int], mlp_ratio: float = 4.0, init_values: Optional[float] = 0.0,
                 proj_drop: float = 0.0, drop_attn: float = 0.0, drop_path: Union[List[float], float] = 0.0,
                 norm_layer: Type[nn.Module] = nn.LayerNorm, extra_norm_period: int = 0, extra_norm_stage: bool = False,
                 sequential_attn: bool = False, rel_pos: bool = True, grad_checkpointing: bool = False,
                 compute_mode: str = "bf16") -> None:
        super().__init__()
        if downscale:
            raise NotImplementedError("PatchMerging stages are never instantiated by the reference (downscale=False, :745)")
        self.downscale = downscale
        self.feat_size = feat_size
        self.grad_checkpointing = grad_checkpointing
        self.downsample = nn.Identity()
        self.blocks = nn.Sequential(*[
            SwinTransformerV2CrBlock(
                dim=embed_dim, num_heads=num_heads, feat_size=self.feat_size, window_size=window_size,
                shift_size=tuple([0 if ((index % 2) == 0) else w // 2 for w in window_size]), mlp_ratio=mlp_ratio,
                init_values=init_values, proj_drop=proj_drop, drop_attn=drop_attn,
                drop_path=drop_path[index] if isinstance(drop_path, list) else drop_path, sequential_attn=sequential_attn,
                norm_layer=norm_layer, rel_pos=rel_pos, compute_mode=compute_mode)
            for index in range(depth)])

    def update_input_size(self, new_window_size, new_feat_size: Tuple[int, int]) -> None:
        self.feat_size = new_feat_size
        for block in self.blocks:
            block.update_input_size(new_window_size=new_window_size, new_feat_size=self.feat_size)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x: (B, C, H, W) view -> (B, C, H, W) view; the token stream stays (B, H, W, C) in memory (:639-655)."""
        shadow = getattr(x, _SHADOW_ATTR, None)
        x = _carry_shadow(bchw_to_bhwc(x), shadow)
        if not x.is_contiguous():
            x = x.contiguous()
        # exp(min(logit_scale, ln 100)) (reference :186 / :305) of every block at once: same torch ops on the stacked
        # parameters (bit-identical values, gradients flow back through the stack), 3 launches instead of 2 per block
        scales = torch.clamp(torch.stack([b.attn.logit_scale for b in self.blocks]), max=math.log(1.0 / 0.01)).exp().unbind(0)
        for i, block in enumerate(self.blocks):
            if self.grad_checkpointing and not torch.jit.is_scripting():
                shadow = getattr(x, _SHADOW_ATTR, None)
                y = checkpoint(block, x, scales[i], use_reentrant=False)
                x = y
            else:
                x = block(x, scales[i])
        shadow = getattr(x, _SHADOW_ATTR, None)
        return _carry_shadow(bhwc_to_bchw(x), shadow)


class SwinTransformerV2Cr(nn.Module):
    """reference: swinv2_global.py:657-865 -- same constructor signature plus `compute_mode`."""

    def __init__(self, img_size: Tuple[int, int] = (224, 224), patch_size: int = 4, window_size: Optional[int] = None,
                 img_window_ratio: int = 32, in_chans: int = 3, out_chans: int = 3, embed_dim: int = 96,
                 depths: Tuple[int, ...] = (2, 2, 6, 2), num_heads: Tuple[int, ...] = (3, 6, 12, 24), mlp_ratio: float = 4.0,
                 init_values: Optional[float] = 0., drop_rate: float = 0.0, proj_drop_rate: float = 0.0,
                 attn_drop_rate: float = 0.0, drop_path_rate: float = 0.0, norm_layer: Type[nn.Module] = nn.LayerNorm,
                 extra_norm_period: int = 0, extra_norm_stage: bool = False, sequential_attn: bool = False,
                 global_pool: str = 'avg', weight_init='skip', full_pos_embed: bool = False, rel_pos: bool = True,
                 checkpoint_stages: bool = False, residual: bool = False, compute_mode: str = "bf16", **kwargs: Any) -> None:
        super().__init__()
        if compute_mode not in ops.MODES:
            raise ValueError(f"compute_mode must be one of {sorted(ops.MODES)}")
        if len(depths) != 1 or len(num_heads) != 1:
            raise NotImplementedError("the weather model is single-stage (swinv2net passes depths=(depth,), :62-63)")
        if weight_init != 'skip':
            raise NotImplementedError("weight_init != 'skip' is broken in the reference (named_apply undefined, :775)")
        img_size = to_2tuple(img_size)
        window_size = tuple([s // img_window_ratio for s in img_size]) if window_size is None else to_2tuple(window_size)
        if patch_size != 4:
            raise NotImplementedError("the kernels are specialised for patch_size 4 (every reference config)")
        # kernel limits, checked here rather than at the first forward: the LayerNorm forward holds a row in registers
        # (C <= 2048) and the attention kernels are instantiated for head_dim <= 256.  The largest shipped config,
        # swin_73var_geo_depth24_e2048_mlp2_chweight_invar (embed_dim 2048, 8 heads of 256), sits on both limits.
        if embed_dim > 2048 or embed_dim % 8 != 0:
            raise NotImplementedError(f"embed_dim {embed_dim}: the B200 kernels support multiples of 8 up to 2048")
        if embed_dim % num_heads[0] != 0 or (embed_dim // num_heads[0]) % 8 != 0 or embed_dim // num_heads[0] > 256:
            raise NotImplementedError(f"head_dim {embed_dim / num_heads[0]:g}: the attention kernels support multiples of 8 up to 256")
        self.patch_size = patch_size
        self.img_size = img_size
        self.window_size = window_size
        self.num_features = int(embed_dim)
        self.out_chans = out_chans
        self.feature_info = []
        self.full_pos_embed = full_pos_embed
        self.checkpoint_stages = checkpoint_stages
        self.residual = residual
        self.depth = len(depths)
        self.compute_mode = compute_mode

        self.patch_embed = PatchEmbed(img_size=img_size, patch_size=patch_size, in_chans=in_chans, embed_dim=embed_dim,
                                      norm_layer=norm_layer)
        patch_grid_size = self.patch_embed.grid_size
        dpr = [x.tolist() for x in torch.linspace(0, drop_path_rate, sum(depths), device="cpu").split(depths)]
        stages = []
        for stage_idx, (depth, heads) in enumerate(zip(depths, num_heads)):
            stages += [SwinTransformerV2CrStage(
                embed_dim=embed_dim, depth=depth, downscale=False, feat_size=patch_grid_size, num_heads=heads,
                window_size=window_size, mlp_ratio=mlp_ratio, init_values=init_values, proj_drop=proj_drop_rate,
                drop_attn=attn_drop_rate, drop_path=dpr[stage_idx], extra_norm_period=extra_norm_period,
                extra_norm_stage=extra_norm_stage or (stage_idx + 1) == len(depths), sequential_attn=sequential_attn,
                norm_layer=norm_layer, rel_pos=rel_pos, grad_checkpointing=self.checkpoint_stages,
                compute_mode=compute_mode)]
            self.feature_info += [dict(num_chs=embed_dim, reduction=4, module=f'stages.{stage_idx}')]
        self.stages = nn.Sequential(*stages)
        self.head = nn.Linear(embed_dim, self.out_chans * self.patch_size * self.patch_size, bias=False)
        if self.full_pos_embed:
            self.pos_embed = nn.Parameter(torch.randn(1, embed_dim, patch_grid_size[0], patch_grid_size[1]) * .02)

    # -- compute mode plumbing -------------------------------------------------------------------------
    def set_compute_mode(self, name: str) -> "SwinTransformerV2Cr":
        if name not in ops.MODES:
            raise ValueError(f"compute_mode must be one of {sorted(ops.MODES)}")
        self.compute_mode = name
        for m in self.modules():
            if isinstance(m, SwinTransformerV2CrBlock):
                m.compute_mode = name
        return self

    # -- forward ------------------------------------------------------------------------------------------
    def _input_stats(self, input_stats, n_chans: int, device):
        """(mean, std) given for the leading channels of the input -> full-length fp32 device vectors (mean 0 / std 1 for the
        channels that pass through unchanged: zenith angle, land mask, orography)."""
        if input_stats is None:
            return None, None
        mean, std = (torch.as_tensor(t, dtype=torch.float32).reshape(-1).to(device) for t in input_stats)
        if mean.numel() != std.numel() or mean.numel() > n_chans:
            raise ValueError(f"input_stats: {mean.numel()} means / {std.numel()} stds for an input of {n_chans} channels")
        pad = n_chans - mean.numel()
        if pad:
            mean = torch.cat([mean, mean.new_zeros(pad)])
            std = torch.cat([std, std.new_ones(pad)])
        return mean.contiguous(), std.contiguous()

    def forward_features(self, x, input_stats=None) -> torch.Tensor:
        """x: (B, Cin, H, W), or a tuple / list of channel groups [(B, C0, H, W), (B or 1, C1, H, W), ...] standing for their
        concatenation along dim 1 (what PreProcessor / MultiStepWrapper would otherwise build with torch.cat).
        `input_stats` = (mean, std) per channel of a RAW field: the z-score the reference's loaders apply before the model
        (utils/data_loader_era5_dali.py:77-90) then happens inside the PatchEmbed im2col."""
        mode = ops.MODES[self.compute_mode]
        parts = [t.float() for t in x] if isinstance(x, (tuple, list)) else [x.float()]
        B, _, H, W = parts[0].shape
        assert H == self.img_size[0], f"Input image height ({H}) doesn't match model ({self.img_size[0]})."
        assert W == self.img_size[1], f"Input image width ({W}) doesn't match model ({self.img_size[1]})."
        pe = self.patch_embed
        mean, std = self._input_stats(input_stats, sum(t.shape[1] for t in parts), parts[0].device)
        pos = self.pos_embed if self.full_pos_embed else None
        if _forward_only(*parts, pe.proj.weight, pe.proj.bias, pe.norm.weight, pe.norm.bias, pos, mean, std):
            tok, shadow = Fn.patch_embed_forward_only(parts[0], pe.proj.weight, pe.proj.bias, pe.norm.weight, pe.norm.bias, pos,
                                                      self.patch_size, mode, mean, std, *parts[1:])
        else:
            tok, shadow = Fn.PatchEmbedFn.apply(parts[0], pe.proj.weight, pe.proj.bias, pe.norm.weight, pe.norm.bias, pos,
                                                self.patch_size, mode, mean, std, *parts[1:])
        x = _carry_shadow(bhwc_to_bchw(tok), shadow)
        return self.stages(x)

    def forward_head(self, x: torch.Tensor, skip: Optional[torch.Tensor] = None, skip_stats=(None, None)) -> torch.Tensor:
        mode = ops.MODES[self.compute_mode]
        shadow = getattr(x, _SHADOW_ATTR, None)
        t = bchw_to_bhwc(x)
        if not t.is_contiguous():
            t = t.contiguous()
        t = _carry_shadow(t.float(), shadow)
        if _forward_only(t, self.head.weight, skip):
            return Fn.head_forward_only(t, _shadow_of(t, mode), self.head.weight, skip, self.out_chans, self.patch_size, mode,
                                        *skip_stats)
        return Fn.HeadFn.apply(t, _shadow_of(t, mode), self.head.weight, skip, self.out_chans, self.patch_size, mode, *skip_stats)

    def forward(self, x, input_stats=None) -> torch.Tensor:
        if isinstance(x, (tuple, list)):
            x = [t.float() for t in x]
            if self.residual and x[0].shape[1] < self.out_chans:      # the skip needs the first out_chans channels in one tensor
                x = torch.cat([t.expand(x[0].shape[0], -1, -1, -1) for t in x], dim=1)
        else:
            x = x.float()
        first = x[0] if isinstance(x, list) else x
        skip = first if self.residual else None   # the reference adds zeros_like(x) otherwise (:795-802); adding 0 is skipped
        feats = self.forward_features(x, input_stats)
        skip_stats = (None, None)
        if skip is not None and input_stats is not None:
            n_in = sum(t.shape[1] for t in x) if isinstance(x, list) else x.shape[1]
            skip_stats = tuple(t[:skip.shape[1]].contiguous() for t in self._input_stats(input_stats, n_in, skip.device))
        return self.forward_head(feats, skip, skip_stats)

    # -- reference API odds and ends ----------------------------------------------------------------------------
    def update_input_size(self, new_img_size=None, new_window_size=None, img_window_ratio: int = 32) -> None:
        raise NotImplementedError("update_input_size is broken in the reference (:829-832 passes an unknown keyword)")

    @torch.jit.ignore
    def group_matcher(self, coarse=False):
        return dict(stem=r'^patch_embed', blocks=r'^stages\.(\d+)' if coarse else [
            (r'^stages\.(\d+).downsample', (0,)), (r'^stages\.(\d+)\.\w+\.(\d+)', None)])

    @torch.jit.ignore
    def set_grad_checkpointing(self, enable=True):
        for s in self.stages:
            s.grad_checkpointing = enable
