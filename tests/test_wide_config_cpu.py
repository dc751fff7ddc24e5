"""CPU: the largest shipped configuration, swin_73var_geo_depth24_e2048_mlp2_chweight_invar (embed_dim 2048, 8 heads of 256,
depth 24, mlp_ratio 2), is accepted by the constructor, has the reference's parameter tree, and its attention dispatches to
the tensor-core kernels; one step beyond its widths is still refused."""
from types import SimpleNamespace

import pytest
import torch

from swin_v2_weather_b200 import ops
from swin_v2_weather_b200._lib import BACKEND_SIMT, BACKEND_TCGEN05
from swin_v2_weather_b200.networks.swinv2_global import SwinTransformerV2Cr, swinv2net

WIDE = dict(img_size=(720, 1440), patch_size=4, depths=(24,), num_heads=(8,), in_chans=73, out_chans=73, embed_dim=2048,
            img_window_ratio=80, mlp_ratio=2, full_pos_embed=True, rel_pos=False, drop_path_rate=0.1)


def test_wide_config_parameter_count():
    """318 keys and 943,347,904 elements at 73 input channels (meta device: no memory)."""
    with torch.device("meta"):
        m = SwinTransformerV2Cr(**WIDE)
    sd = m.state_dict()
    assert len(sd) == 318
    assert sum(v.numel() for v in sd.values()) == 943_347_904
    assert m.window_size == (9, 18)
    blocks = m.stages[0].blocks
    assert [b.shift_size for b in blocks] == [(0, 0), (4, 9)] * 12
    assert blocks[0].mlp.fc1.weight.shape == (4096, 2048)
    assert blocks[0].attn.qkv.weight.shape == (3 * 2048, 2048)


def test_swinv2net_builds_the_wide_config():
    params = SimpleNamespace(img_size=[720, 1440], patch_size=4, depth=24, num_heads=8, n_in_channels=73, n_out_channels=73,
                             embed_dim=2048, window_ratio=80, drop_path_rate=0.1, full_pos_embed=True, rel_pos=False,
                             mlp_ratio=2, activation_ckpt=False, residual=False)
    with torch.device("meta"):
        m = swinv2net(params)
    assert m.num_features == 2048 and len(m.stages[0].blocks) == 24
    assert m.stages[0].blocks[0].attn.num_heads == 8


@pytest.mark.parametrize("embed_dim,heads", [(2056, 8), (2112, 8)])
def test_beyond_the_kernel_widths_is_refused(embed_dim, heads):
    """embed_dim 2056 (> 2048) and head_dim 264 (> 256) raise at construction, before any kernel could be reached."""
    cfg = dict(WIDE, embed_dim=embed_dim, num_heads=(heads,), depths=(1,))
    with torch.device("meta"), pytest.raises(NotImplementedError):
        SwinTransformerV2Cr(**cfg)


def test_head_dim_264_is_refused_within_the_embed_dim_limit():
    cfg = dict(WIDE, embed_dim=1056, num_heads=(4,), depths=(1,))     # head_dim 264, embed_dim <= 2048
    with torch.device("meta"), pytest.raises(NotImplementedError, match="head_dim 264"):
        SwinTransformerV2Cr(**cfg)


def test_wide_attention_dispatches_to_tensor_cores():
    assert ops.attn_backend_for(ops.MODE_BF16, 2048, 8, 9, 18) == BACKEND_TCGEN05
    assert 256 in ops.TCGEN05_HEAD_DIMS
    assert ops.attn_backend_for(ops.MODE_FP32, 2048, 8, 9, 18) == BACKEND_SIMT          # fp32 validation mode
    assert ops.attn_backend_for(ops.MODE_BF16_SIMT, 2048, 8, 9, 18) == BACKEND_SIMT
