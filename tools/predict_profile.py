"""GPU diagnostic: where one prediction batch spends its time (crop / forward / accumulate per colour class / finalize),
CUDA events around eager launches.  usage: predict_profile.py [side=4096] [batch=64]"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from unet_b200 import _lib, ops
from unet_b200.network import UNetB200
from unet_b200.predict_engine import TiledPredictor
side = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
B = int(sys.argv[2]) if len(sys.argv) > 2 else 64
net = UNetB200("xresnet34", 4, 2, (256, 256), B, training=False)
net.init_parameters(seed=0)
pred = TiledPredictor(net)
g = torch.Generator(device="cuda").manual_seed(1)
raster = torch.randint(0, 256, (4, side, side), dtype=torch.uint8, device="cuda", generator=g)
pred.predict_raster(raster, 0.125)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record(); pred.predict_raster(raster, 0.125); b.record(); torch.cuda.synchronize()
n = pred.last_stitch_profile
print(f"predict_raster: {a.elapsed_time(b):.2f} ms for {n['tiles_run']} tiles in {n['batches']} batches = {a.elapsed_time(b) / n['batches']:.3f} ms/batch")
# components, eager
lib, s = net.lib, ops.stream_ptr()
y0 = torch.arange(B, dtype=torch.int32, device="cuda") * 3
x0 = torch.arange(B, dtype=torch.int32, device="cuda") * 5
def timed(name, fn, reps=10):
    fn(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): fn()
    b.record(); torch.cuda.synchronize()
    print(f"{name:28s} {a.elapsed_time(b) / reps:.3f} ms")
timed("crop_tiles", lambda: _lib.check(lib.b2u_crop_tiles(raster.data_ptr(), 1, 255.0, 1.0, 4, side, side, y0.data_ptr(), x0.data_ptr(), B, 256, net.x_in.t.data_ptr(), net.x_in.ld, s)))
timed("forward (eager)", lambda: net.forward(s))
acc = torch.zeros((2, side, side), device="cuda"); cnt = torch.zeros((side, side), dtype=torch.uint8, device="cuda")
sel = torch.arange(B, dtype=torch.int32, device="cuda"); nsel = torch.tensor([B // 4], dtype=torch.int32, device="cuda")
yy = (torch.arange(B, dtype=torch.int32, device="cuda") // 8) * 256; xx = (torch.arange(B, dtype=torch.int32, device="cuda") % 8) * 256
timed("stitch_accumulate x4 classes", lambda: [_lib.check(lib.b2u_stitch_accumulate(net.logits.data_ptr(), net.logits.shape[-1], 2, B, 256, 256, yy.data_ptr(), xx.data_ptr(), sel.data_ptr(), nsel.data_ptr(), B, 0, acc.data_ptr(), cnt.data_ptr(), side, side, 0, 0, s)) for _ in range(4)])
mask = torch.empty((side, side), dtype=torch.uint8, device="cuda")
timed("stitch_finalize", lambda: _lib.check(lib.b2u_stitch_finalize(acc.data_ptr(), cnt.data_ptr(), 2, side, side, 0, mask.data_ptr(), s)))
timed("zero acc+cnt", lambda: (acc.zero_(), cnt.zero_()))
