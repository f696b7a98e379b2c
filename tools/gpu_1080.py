"""Development tool: 1080p synthetic stream: timings + entropy-kernel status / profile counters."""
import os, sys, time
import numpy as np, torch
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
import coolchic_b200
from coolchic_b200 import _native, synth
from coolchic_b200._desc import desc_from_header
ctx = _native.get_context(0)
ss = synth.SeedStream(ctx)
hyp = (4, 6) if "hyper" in sys.argv else None
zeros = "zeros" in sys.argv
lat_in = None
if zeros:  # all-zero latents: (almost) every symbol is the mode -> time per symbol = the coder's hot path
    tmp_h = synth.make_coolchic_header(ss.header, (1080, 1920), (0, 6), hyp)
    lat_in = torch.zeros(desc_from_header(tmp_h).n_symbols(), dtype=torch.int8, device="cuda")
cc, h, lat = synth.make_coolchic(ctx, ss, (1080, 1920), (0, 6), hyp, seed=0, latents=lat_in)
h2 = type(h)(); rest = h2.read_header(cc); d = desc_from_header(h2)
nnb = rest[:h2.get_value("nn_n_bytes")]; lb = rest[h2.get_value("nn_n_bytes"):][:h2.get_value("n_bytes_latent")]
nn = _native.decode_nn(d, nnb)
print("symbols", d.n_symbols(), "payload", len(lb), "bpp %.3f" % (len(lb) * 8 / (1080 * 1920)))
for it in range(3):
    out = ctx.decode_latents(d, nn, lb); torch.cuda.synchronize()
    st = ctx.last_status()
    print(ctx.last_timing(), st[:4])
    if any(st[4:]):
        print("  prof kcyc: coder wait %d total %d | producers wait %d arm %d win %d total %d | far %d redo-groups %d singles %d fast %d chunks %d | helper total %d" % tuple(st[4:16]))
print("round trip ok:", torch.equal(out, lat))
l = lat.cpu().numpy().astype(int); off = 0
for g in range(d.n_grids - 1, -1, -1):
    n = d.grid_h[g] * d.grid_w[g]; a = l[off:off + n]; off += n
    print("grid", g, (d.grid_h[g], d.grid_w[g]), "zeros %.2f mean|x| %.2f max %d" % ((a == 0).mean(), np.abs(a).mean(), np.abs(a).max()))
