"""Development tool: decode kodim14 many times, report mismatches and debug status."""
import os, sys
import numpy as np, torch
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
import coolchic_b200
from coolchic_b200.bitstream.header import VideoHeader, FrameHeader, CoolChicHeader
from coolchic_b200._desc import desc_from_header
from coolchic_b200 import _native
data = open(os.path.join(ROOT, "tests/golden/kodim14.cool"), "rb").read()
v = VideoHeader(); rest = v.read_header(data); f = FrameHeader(); rest = f.read_header(rest); c = CoolChicHeader(); rest = c.read_header(rest)
d = desc_from_header(c)
nnb = rest[:c.get_value("nn_n_bytes")]; lb = rest[c.get_value("nn_n_bytes"):][:c.get_value("n_bytes_latent")]
ctx = _native.get_context(0)
nn = _native.decode_nn(d, nnb)
g = np.load(os.path.join(ROOT, "tests/golden/kodim14_latents.npz"))["latents"]
n = int(sys.argv[1]) if len(sys.argv) > 1 else 20
bad = 0; times = []
for it in range(n):
    lat = None
    try:
        lat = ctx.decode_latents(d, nn, lb); torch.cuda.synchronize()
        ok = np.array_equal(lat.cpu().numpy(), g)
    except Exception as e:
        ok = False; print("EXC", str(e)[:60])
    st = ctx.last_status(); times.append(ctx.last_timing()["entropy_ms"])
    if not ok:
        bad += 1
        print("run", it, "MISMATCH status", st)
print("runs", n, "bad", bad, "entropy ms min/med/max %.2f %.2f %.2f" % (min(times), sorted(times)[len(times)//2], max(times)), "last status", st)
