import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ultrazoom_b200 import unet as N, ops
dev = torch.device("cuda", 0)
def timed(fn, iters=10):
    for _ in range(3): fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    for _ in range(iters): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters
torch.manual_seed(9)
C = 96
x = torch.randn(1, 540, 960, C, device=dev)
blk = N.SR2XBlock(C, 2, 48).to(dev)
print("sr2x", timed(lambda: blk.forward(x)))
ib = blk.refiner.convnet
print("inverted_bottleneck", timed(lambda: ib.forward(x)))
x16 = x.to(torch.float16)
print("cast", timed(lambda: x.to(torch.float16)))
print("conv_silu", timed(lambda: N._conv_silu(x16, ib.conv1.weight)))
hid = N._conv_silu(x16, ib.conv1.weight)
print("conv_add(+zeros)", timed(lambda: N._conv_add(hid, ib.conv2.weight)))
print("zeros", timed(lambda: torch.zeros((1, 540, 960, C), dtype=torch.float32, device=dev)))
z = ib.forward(x)
print("mix", timed(lambda: blk.refiner.skip.forward(x, z)))
y = blk.refiner.forward(x)
print("subpixel", timed(lambda: blk.upscale.forward(y)))
print("subpixel conv only", timed(lambda: N.conv3x3_plain(y, blk.upscale.conv.weight)))
