"""Per-phase cycle breakdown of the tcgen05 attention backward at the full 180x360 geometry, and the launch times of the
forward and the backward (bring-up aid).  Only the backward kernel writes phase counters."""
import sys
import torch
sys.path.insert(0, ".")
from swin_v2_weather_b200 import _lib, ops
from swin_v2_weather_b200._lib import BACKEND_TCGEN05

B, H, W, C, heads = 1, 180, 360, 768, 8
T = B * H * W
torch.manual_seed(0)
qkv = torch.randn(T, 3 * C, device="cuda").bfloat16()
inv = ops.qk_normalize_(qkv, C, heads)
scale = torch.full((heads,), 10.0, device="cuda")
buf = torch.zeros(4096 * 16, dtype=torch.int64, device="cuda")
for shift in ((0, 0), (4, 9)):
    def fwd():
        return ops.window_attn_fwd(qkv, scale, None, B, H, W, C, heads, 9, 18, shift[0], shift[1], ops.MODE_BF16, backend=BACKEND_TCGEN05)

    o, lse = fwd()
    d_o = torch.randn_like(o)

    def bwd():
        ops.window_attn_bwd(qkv, inv, scale, None, o, d_o, lse, B, H, W, C, heads, 9, 18, shift[0], shift[1], ops.MODE_BF16, backend=BACKEND_TCGEN05)

    _lib.call("swinb200_debug_attn_phase_buffer", buf.data_ptr())
    buf.zero_()
    bwd()
    torch.cuda.synchronize()
    _lib.call("swinb200_debug_attn_phase_buffer", 0)
    # persistent kernel: per-CTA accumulated cycles per phase over all its items
    st = buf.view(4096, 16)[:148, :16].double()
    items = 3200 / 148
    print("bwd", shift, "mean cycles per phase per item:", [int(v / items) for v in st.mean(0).tolist()], "total/item", int(st.sum(1).mean() / items))
    for name, run in (("fwd", fwd), ("bwd", bwd)):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(5):
            run()
        ev[1].record()
        torch.cuda.synchronize()
        print("   ", name, "time per launch: %.1f us" % (ev[0].elapsed_time(ev[1]) * 1000 / 5))
