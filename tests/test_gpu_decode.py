"""Parity tests proper: the CUDA path, called through the C-ABI, against the oracle and the
golden fixtures.  Integer work (NN ints, latents, payload bytes) must be bit-exact; the
float path is bit-exact against the oracle (same canonical fp32 order) and within the
north-star tolerance 1e-5 of the PyTorch reference."""
import os
import subprocess
import sys

import numpy as np
import pytest
from conftest import GOLDEN, ROOT

pytestmark = pytest.mark.gpu
TOL_FLOAT = 1e-5


def _decode_ref(oracle, desc, nn, payload):
    lat, _ = oracle.decode_latents(desc, nn, payload)
    return lat


# ------------------------------------------------------------------------------------------
def test_kodim14_through_c_abi(ctx, oracle, kodim14):
    import torch

    d = kodim14["desc"]
    out, lat = ctx.decode_coolchic(d, kodim14["nn_bytes"], kodim14["lat_bytes"], want_latents=True)
    torch.cuda.synchronize()
    assert ctx.last_status()[:3] == [0, 7739, 0]  # no error, 7738 words + 1 over-read, no slow path
    assert np.array_equal(lat.cpu().numpy(), kodim14["latents"])  # bit-exact vs the reference
    nn = oracle.decode_nn(d, kodim14["nn_bytes"])
    raw_o = oracle.synthesize(d, nn, kodim14["latents"])
    raw = out[0].cpu().numpy()
    assert np.array_equal(raw, raw_o)  # same canonical fp32 order as the oracle
    g = kodim14["raw_rows"]
    assert np.abs(raw[:, g["rows"], :] - g["data"]).max() <= TOL_FLOAT  # vs the PyTorch reference
    img = ctx.finish_frame(out, 8, "rgb")[0].cpu().numpy()
    assert np.array_equal(img, oracle.finish_frame(raw_o, 8, "rgb"))
    u8 = np.round(img * 255).astype(np.uint8).transpose(1, 2, 0)
    diff = u8.astype(np.int32) - kodim14["image"].astype(np.int32)
    assert np.abs(diff).max() <= 1 and int((diff != 0).sum()) <= 32  # rounding ties only (SURVEY F7)


def test_decode_video_api_and_cli(ctx, kodim14, tmp_path):
    from coolchic_b200.bitstream.decode import decode_frame, decode_video
    from coolchic_b200.io import FrameData

    path = os.path.join(GOLDEN, "kodim14.cool")
    frames = decode_video(path, decoded_path=str(tmp_path / "out.ppm"))
    assert list(frames) == ["0"] and isinstance(frames["0"], FrameData)
    fd = frames["0"]
    assert (fd.bitdepth, fd.frame_data_type, fd.img_size) == (8, "rgb", (512, 768))
    assert fd.data.device.type == "cpu" and fd.data.dtype.is_floating_point and tuple(fd.data.shape) == (1, 3, 512, 768)
    u8 = np.round(fd.data[0].numpy() * 255).astype(np.uint8).transpose(1, 2, 0)
    assert int((u8 != kodim14["image"]).sum()) <= 32
    raw = (tmp_path / "out.ppm").read_bytes()
    assert raw.startswith(b"P6\n768 512\n255\n") and np.array_equal(
        np.frombuffer(raw[len(b"P6\n768 512\n255\n"):], dtype=np.uint8).reshape(512, 768, 3), u8)
    # decode_frame returns the unread tail (decode.py:212)
    frame, rest = decode_frame(kodim14["data"][8:] + b"tail", reference_frames=[])
    assert rest == b"tail" and frame.img_size == (512, 768)
    # the command line
    out_png = tmp_path / "cli.png"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "cc_decode.py"), "-i", path, "-o", str(out_png)],
                       capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    assert "Decoding frame 0" in r.stdout and "seconds." in r.stdout
    from PIL import Image

    assert np.array_equal(np.asarray(Image.open(out_png)), u8)


def test_corrupt_payload_is_reported(ctx, kodim14):
    from coolchic_b200 import _native

    bad = bytearray(kodim14["lat_bytes"])
    bad[0:64] = b"\xff" * 64
    with pytest.raises(_native.CcdError) as e:
        ctx.decode_coolchic(kodim14["desc"], kodim14["nn_bytes"], bytes(bad))
    assert e.value.code == -3  # CCD_ERR_DESYNC
    with pytest.raises(_native.CcdError) as e:
        ctx.decode_coolchic(kodim14["desc"], kodim14["nn_bytes"][:500], kodim14["lat_bytes"])
    assert e.value.code == -2  # CCD_ERR_NN_TRUNCATED
    # an empty payload decodes like the reference does (missing words read as 0): no crash
    ctx.decode_coolchic(kodim14["desc"], kodim14["nn_bytes"], b"")


def test_device_range_encoder_and_sampler(ctx, oracle, kodim14):
    import torch

    d = kodim14["desc"]
    nn = oracle.decode_nn(d, kodim14["nn_bytes"])
    _, payload, slow = ctx.encode_latents(d, nn, latents=torch.from_numpy(kodim14["latents"]).cuda())
    assert payload == kodim14["lat_bytes"] and slow == 0  # byte-exact with real constriction output
    lat_s, payload_s, _ = ctx.encode_latents(d, nn, seed=77)
    lat_o, payload_o = oracle.sample_latents(d, nn, 77)
    assert np.array_equal(lat_s.cpu().numpy(), lat_o) and payload_s == payload_o
    # the sampled stream leaves the 31-symbol window often: exercises the exact-CDF slow path
    dec = ctx.decode_latents(d, nn, payload_s)
    assert np.array_equal(dec.cpu().numpy(), lat_o) and ctx.last_status()[2] > 1000


# ------------------------------------------------------------------------------------------
# synthetic streams: (H, W), latent_resolution, hyperlatent_resolution, header overrides
CASES = [
    ((64, 96), (0, 6), (4, 6), {}),                     # same structure as the sample, tiny
    ((17, 33), (0, 4), None, {}),                       # odd sizes, ceil grids, crops
    ((129, 7), (0, 3), None, {}),                       # w <= 9: raster scan on every grid
    ((40, 250), (0, 6), (4, 6), {}),                    # coarse grids 1 pixel high
    ((96, 64), (0, 2), None, {}),                       # few grids
    ((1, 1), (0, 1), None, {}),                         # degenerate
    ((72, 88), (2, 5), None, {"final_upsampling_type": "nearest"}),  # motion-like: nearest x4 output
    ((60, 100), (0, 6), (4, 6), {"spatial_context_arm": 8}),          # no template: generic int64 kernel
    ((60, 100), (0, 5), None, {"spatial_context_arm": 20}),           # vhop ARM width (20 + 6)
    ((48, 80), (0, 4), None, {"n_hidden_layers_arm": 1, "linear_stabiliser_arm": 0}),
    ((48, 80), (0, 4), None, {"output_feature_ifce": 0}),             # no IFCE at all -> generic
]


@pytest.mark.parametrize("case", CASES, ids=[f"{c[0][0]}x{c[0][1]}-{i}" for i, c in enumerate(CASES)])
def test_synthetic_stream_parity(ctx, oracle, seed_stream, case):
    import torch

    from coolchic_b200 import synth
    from coolchic_b200._desc import desc_from_header

    hw, lr, hr, ov = case
    ov = dict(ov)
    fut = ov.pop("final_upsampling_type", None)
    if ov.get("output_feature_ifce", 1) == 0:
        ov["ifce_resolution"] = None
    cc_bytes, header, lat_dev = synth.make_coolchic(ctx, seed_stream, hw, lr, hr, seed=3, final_upsampling_type=fut,
                                                    overrides=ov)
    if ov.get("output_feature_ifce", 1) == 0:
        assert header.get_value("ifce_resolution") is None
    h2 = type(header)()
    rest = h2.read_header(cc_bytes)
    d = desc_from_header(h2)
    n_nn, n_lat = h2.get_value("nn_n_bytes"), h2.get_value("n_bytes_latent")
    nn_bytes, payload = rest[:n_nn], rest[n_nn:n_nn + n_lat]
    nn = oracle.decode_nn(d, nn_bytes)
    lat_in = lat_dev.cpu().numpy()
    # encoder parity: the device payload is the oracle's payload
    assert payload == oracle.encode_latents(d, nn, lat_in)
    # decoder parity
    out, lat = ctx.decode_coolchic(d, nn_bytes, payload, want_latents=True)
    torch.cuda.synchronize()
    assert ctx.last_status()[0] == 0
    assert np.array_equal(lat.cpu().numpy(), lat_in)                       # round trip
    assert np.array_equal(lat.cpu().numpy(), _decode_ref(oracle, d, nn, payload))  # vs oracle
    assert np.array_equal(out[0].cpu().numpy(), oracle.synthesize(d, nn, lat_in))  # bit-exact float tail
    assert tuple(out.shape) == (1, 3, hw[0], hw[1])


def test_many_streams_concurrently(ctx, oracle, seed_stream):
    """decode_many: one persistent CTA per stream, mixed architectures in one call."""
    import torch

    from coolchic_b200 import synth
    from coolchic_b200._desc import desc_from_header

    items = []
    for i in range(9):
        hw = (48 + 8 * i, 120 - 4 * i)
        ov = {"spatial_context_arm": 8} if i % 4 == 3 else {}
        cc_bytes, header, lat_dev = synth.make_coolchic(ctx, seed_stream, hw, (0, 5), (4, 5) if i % 2 else None,
                                                        seed=10 + i, overrides=ov)
        h2 = type(header)()
        rest = h2.read_header(cc_bytes)
        items.append((desc_from_header(h2), rest[:h2.get_value("nn_n_bytes")],
                      rest[h2.get_value("nn_n_bytes"):][:h2.get_value("n_bytes_latent")], lat_dev.cpu().numpy()))
    outs, lats = ctx.decode_many([x[0] for x in items], [x[1] for x in items], [x[2] for x in items], want_latents=True)
    torch.cuda.synchronize()
    for (d, nnb, _, lat_in), out, lat in zip(items, outs, lats):
        assert np.array_equal(lat.cpu().numpy(), lat_in)
        assert np.array_equal(out[0].cpu().numpy(), oracle.synthesize(d, oracle.decode_nn(d, nnb), lat_in))


@pytest.mark.parametrize("fmt,bitdepth", [("rgb", 8), ("yuv444", 10), ("yuv420", 8), ("yuv420", 10), ("yuv420", 12)])
def test_finish_frame(ctx, oracle, fmt, bitdepth):
    import torch

    rng = np.random.default_rng(5)
    x = rng.uniform(-0.3, 1.3, size=(3, 37, 50)).astype(np.float32)
    # exact ties of the rounding grid as well
    x[0, 0, :8] = (np.arange(8) + 0.5) / (2**bitdepth - 1)
    got = ctx.finish_frame(torch.from_numpy(x[None]).cuda(), bitdepth, fmt)
    want = oracle.finish_frame(x, bitdepth, fmt)
    if fmt == "yuv420":
        for k in "yuv":
            assert np.array_equal(got[k][0, 0].cpu().numpy(), want[k])
    else:
        assert np.array_equal(got[0].cpu().numpy(), want)


def test_laplace_cdf_device_equals_host_exhaustively(ctx, oracle):
    """SURVEY Appendix C.3: the only platform-dependent operation of the entropy model is
    the f64 exp().  Its argument set is finite (32641 numerators x 2561 scales, both CDF
    branches): the device evaluation must equal the host libm one on ALL of it."""
    bad = 0
    step = 128
    for sc in range(0, 2561, step):
        hi_sc = min(2561, sc + step)
        dlo, dhi = ctx.laplace_domain(sc, hi_sc)
        hlo, hhi = oracle.laplace_domain(sc, hi_sc)
        bad += int((dlo != hlo).sum()) + int((dhi != hhi).sum())
    assert bad == 0


# ------------------------------------------------------------------------------------------
# BASELINE.json sizes: size-independent properties (round trip, payload idempotence) + oracle latents
@pytest.mark.parametrize("hw,lr,fmt", [((1080, 1920), (0, 6), "rgb"), ((2160, 3840), (0, 7), "yuv420")],
                         ids=["1080p-7grids-rgb", "4k-8grids-yuv420"])
def test_full_size_parity(ctx, oracle, seed_stream, hw, lr, fmt):
    """BASELINE configs[1] and configs[3] at full size: latents, raw synthesis output and the finished frame are
    IDENTICAL to the oracle's (whole frame, every sample), plus the size-independent properties (every word
    consumed, encode -> decode round trip, payload idempotence)."""
    import torch

    from coolchic_b200 import synth
    from coolchic_b200._desc import desc_from_header

    cc_bytes, header, lat_dev = synth.make_coolchic(ctx, seed_stream, hw, lr, None, seed=1)
    h2 = type(header)()
    rest = h2.read_header(cc_bytes)
    d = desc_from_header(h2)
    nn_bytes = rest[:h2.get_value("nn_n_bytes")]
    payload = rest[h2.get_value("nn_n_bytes"):][:h2.get_value("n_bytes_latent")]
    assert d.n_symbols() == {1080: 2764710, 2160: 11059110}[hw[0]]
    out, lat = ctx.decode_coolchic(d, nn_bytes, payload, want_latents=True)
    torch.cuda.synchronize()
    st = ctx.last_status()
    assert st[0] == 0 and st[1] == len(payload) // 4 + 1  # every word consumed, one over-read
    assert torch.equal(lat, lat_dev)                       # encode -> decode round trip
    nn = oracle.decode_nn(d, nn_bytes)
    _, payload2, _ = ctx.encode_latents(d, nn, latents=lat)
    assert payload2 == payload                             # re-encoding reproduces the payload
    oracle.set_threads(0)
    lat_o = _decode_ref(oracle, d, nn, payload)
    assert np.array_equal(lat.cpu().numpy(), lat_o)        # bit-exact latents vs the oracle
    raw_o = oracle.synthesize(d, nn, lat_o)
    assert np.array_equal(out[0].cpu().numpy(), raw_o)     # the whole float tail, bit for bit
    want = oracle.finish_frame(raw_o, 8, fmt)
    # the production path: library-owned (16-byte aligned) latents -> TMA tile staging, frame tail fused
    fin, _ = ctx.decode_many([d], [nn_bytes], [payload], finish=[(8, fmt)])
    if fmt == "yuv420":
        for k in "yuv":
            assert np.array_equal(fin[0][k][0, 0].cpu().numpy(), want[k]), k
    else:
        assert np.array_equal(fin[0][0].cpu().numpy(), want)
    raw2 = ctx.decode_coolchic(d, nn_bytes, payload)       # same path without the frame tail
    assert torch.equal(raw2, out)


@pytest.mark.parametrize("fmt,bitdepth,hw,lr", [("rgb", 8, (96, 160), (0, 4)), ("yuv420", 8, (96, 160), (0, 4)),
                                                 ("yuv420", 10, (50, 70), (0, 3)), ("yuv444", 10, (33, 47), (0, 2)),
                                                 ("rgb", 8, (64, 64), (0, 1))])
def test_fused_frame_tail_equals_separate_kernels(ctx, oracle, seed_stream, fmt, bitdepth, hw, lr):
    """The frame tail fused into the synthesis kernel (TMA and plain-load tile staging, odd sizes, 2-grid streams)
    against the raw output followed by ccd_finish_frame, and against the oracle."""
    import torch

    from coolchic_b200 import synth
    from coolchic_b200._desc import desc_from_header

    cc, h, _ = synth.make_coolchic(ctx, seed_stream, hw, lr, None, seed=5)
    h2 = type(h)()
    rest = h2.read_header(cc)
    d = desc_from_header(h2)
    nnb = rest[:h2.get_value("nn_n_bytes")]
    lb = rest[h2.get_value("nn_n_bytes"):][:h2.get_value("n_bytes_latent")]
    raw = ctx.decode_coolchic(d, nnb, lb)
    sep = ctx.finish_frame(raw, bitdepth, fmt)
    fin, _ = ctx.decode_many([d], [nnb], [lb], finish=[(bitdepth, fmt)])
    nn = oracle.decode_nn(d, nnb)
    lat_o, _ = oracle.decode_latents(d, nn, lb)
    want = oracle.finish_frame(oracle.synthesize(d, nn, lat_o), bitdepth, fmt)
    if fmt == "yuv420":
        for k in "yuv":
            assert torch.equal(fin[0][k], sep[k]), k
            assert np.array_equal(fin[0][k][0, 0].cpu().numpy(), want[k]), k
    else:
        assert torch.equal(fin[0], sep)
        assert np.array_equal(fin[0][0].cpu().numpy(), want)


def test_148_streams_every_output_checked(ctx, oracle, seed_stream):
    """BASELINE configs[2] on one GPU: 148 Kodak-size streams (24 distinct) in ONE ccd_decode_many call (one SM
    each for the entropy stage, batched float tail): EVERY latent array and EVERY finished frame is compared with
    the oracle's for that stream."""
    import hashlib

    import torch

    from coolchic_b200 import synth
    from coolchic_b200._desc import desc_from_header

    items = []
    for i in range(24):
        cc, h, _ = synth.make_coolchic(ctx, seed_stream, (512, 768), (0, 6), (4, 6), seed=i)
        h2 = type(h)()
        rest = h2.read_header(cc)
        n_nn, n_lat = h2.get_value("nn_n_bytes"), h2.get_value("n_bytes_latent")
        items.append((desc_from_header(h2), rest[:n_nn], rest[n_nn:n_nn + n_lat]))
    oracle.set_threads(0)
    want = []
    for d, nnb, lb in items:
        nn = oracle.decode_nn(d, nnb)
        lat_o, _ = oracle.decode_latents(d, nn, lb)
        img = oracle.finish_frame(oracle.synthesize(d, nn, lat_o), 8, "rgb")
        want.append((hashlib.sha256(lat_o.tobytes()).hexdigest(), hashlib.sha256(np.ascontiguousarray(img).tobytes()).hexdigest()))
    sub = [items[i % 24] for i in range(148)]
    outs, lats = ctx.decode_many([x[0] for x in sub], [x[1] for x in sub], [x[2] for x in sub], want_latents=True,
                                 finish=[(8, "rgb")] * 148)
    torch.cuda.synchronize()
    for i in range(148):
        got = (hashlib.sha256(lats[i].cpu().numpy().tobytes()).hexdigest(),
               hashlib.sha256(np.ascontiguousarray(outs[i][0].cpu().numpy()).tobytes()).hexdigest())
        assert got == want[i % 24], i
    # and without caller-owned latents (library layout: TMA staging)
    outs2, _ = ctx.decode_many([x[0] for x in sub], [x[1] for x in sub], [x[2] for x in sub], finish=[(8, "rgb")] * 148)
    for i in range(148):
        assert torch.equal(outs2[i], outs[i]), i
    # more streams than SMs: the entropy kernel runs 8-warp CTAs, two per SM -- same answers, stream by stream
    n_many = 2 * 148 + 5
    sub = [items[i % 24] for i in range(n_many)]
    outs3, lats3 = ctx.decode_many([x[0] for x in sub], [x[1] for x in sub], [x[2] for x in sub], want_latents=True,
                                   finish=[(8, "rgb")] * n_many)
    torch.cuda.synchronize()
    for i in range(n_many):
        got = (hashlib.sha256(lats3[i].cpu().numpy().tobytes()).hexdigest(),
               hashlib.sha256(np.ascontiguousarray(outs3[i][0].cpu().numpy()).tobytes()).hexdigest())
        assert got == want[i % 24], i


# ------------------------------------------------------------------------------------------
# P/B frames
# sinc coefficients: canonical double-precision sin / cos shared by the oracle and the device (detmath): bit-exact


@pytest.mark.parametrize("is_b,fs", [(False, 8), (True, 8), (True, 6), (False, 12), (False, 2), (True, 2), (False, 4),
                                      (True, 4), (False, 14), (True, 10)])
def test_inter_predict_vs_oracle(ctx, oracle, is_b, fs):
    import torch

    from coolchic_b200.io import FrameData

    rng = np.random.default_rng(11)
    h, w = 45, 70
    residue = rng.normal(0, 0.3, size=(5 if is_b else 4, h, w)).astype(np.float32)
    motion = rng.normal(0, 3.0, size=(4 if is_b else 2, h, w)).astype(np.float32)
    motion[0, :4, :4] = np.array([[0.0, 1.0, -1.0, 2.5]] * 4)  # integer and half-pel flows
    motion[:, 0, 0] = 500.0                                     # far outside the frame: border clamp
    ref0 = rng.uniform(0, 1, size=(3, h, w)).astype(np.float32)
    ref1 = rng.uniform(0, 1, size=(3, h, w)).astype(np.float32)
    gf = [3, -2, -5, 4] if is_b else [6, 1]
    want = oracle.inter_predict(residue, motion, ref0, ref1 if is_b else None, gf, fs)
    refs = [FrameData(8, "rgb", torch.from_numpy(ref0[None]).cuda())]
    if is_b:
        refs.append(FrameData(8, "rgb", torch.from_numpy(ref1[None]).cuda()))
    got = ctx.inter_predict(torch.from_numpy(residue[None]).cuda(), torch.from_numpy(motion[None]).cuda(), refs, is_b,
                            "rgb", gf, fs)
    assert np.array_equal(got[0].cpu().numpy(), want)


def test_unsupported_warp_is_an_error_not_a_fallback(ctx):
    import torch

    from coolchic_b200 import _native
    from coolchic_b200.io import FrameData

    z = torch.zeros((1, 4, 8, 8), device="cuda")
    ref = [FrameData(8, "rgb", z[:, :3].contiguous())]
    with pytest.raises(_native.CcdError) as e:  # 16 taps cannot be signalled by the 4-bit header field: not built
        ctx.inter_predict(z, z[:, :2].contiguous(), ref, False, "rgb", [0, 0], 16)
    assert e.value.code == -4  # CCD_ERR_UNSUPPORTED
    with pytest.raises(_native.CcdError) as e:
        ctx.inter_predict(z, z[:, :2].contiguous(), ref, False, "rgb", [0, 0], 7)
    assert e.value.code == -1  # CCD_ERR_ARG: odd filter size
    # shape errors are raised before any pointer reaches a kernel (the reference raises on them too)
    with pytest.raises(ValueError):  # P-frame residue with 3 channels
        ctx.inter_predict(z[:, :3].contiguous(), z[:, :2].contiguous(), ref, False, "rgb", [0, 0], 8)
    with pytest.raises(ValueError):  # B frame with a 2-channel motion field
        ctx.inter_predict(torch.zeros((1, 5, 8, 8), device="cuda"), z[:, :2].contiguous(), ref + ref, True, "rgb",
                          [0, 0, 0, 0], 8)
    with pytest.raises(ValueError):  # reference of another size
        ctx.inter_predict(z, z[:, :2].contiguous(), [FrameData(8, "rgb", torch.zeros((1, 3, 8, 10), device="cuda"))],
                          False, "rgb", [0, 0], 8)
    with pytest.raises(ValueError):  # B frame, one reference
        ctx.reconstruct_frame(torch.zeros((1, 5, 8, 8), device="cuda"), z, ref, True, "rgb", 8, [0, 0, 0, 0], 8)


@pytest.mark.parametrize("fmt,is_b,fs,bitdepth", [("yuv420", True, 8, 8), ("yuv420", False, 6, 10), ("yuv444", True, 4, 10),
                                                   ("rgb", False, 2, 8), ("yuv420", True, 2, 8)])
def test_reconstruct_frame_vs_oracle(ctx, oracle, fmt, is_b, fs, bitdepth):
    """The one-kernel P/B reconstruction (4:2:0 references read in place, fused frame tail) against the oracle's
    convert_420_to_444 -> inter_predict -> finish_frame sequence: identical samples."""
    import torch

    from coolchic_b200.io import FrameData

    rng = np.random.default_rng(23)
    h, w = 46, 72
    M = 2**bitdepth - 1
    residue = rng.normal(0, 0.3, size=(5 if is_b else 4, h, w)).astype(np.float32)
    motion = rng.normal(0, 2.5, size=(4 if is_b else 2, h, w)).astype(np.float32)

    def make_ref():
        if fmt == "yuv420":
            return {"y": (rng.integers(0, M + 1, size=(h, w)) / M).astype(np.float32),
                    "u": (rng.integers(0, M + 1, size=(h // 2, w // 2)) / M).astype(np.float32),
                    "v": (rng.integers(0, M + 1, size=(h // 2, w // 2)) / M).astype(np.float32)}
        return (rng.integers(0, M + 1, size=(3, h, w)) / M).astype(np.float32)

    refs = [make_ref() for _ in range(2 if is_b else 1)]

    def to444(r):
        if fmt != "yuv420":
            return r
        up = lambda p: np.repeat(np.repeat(p, 2, axis=0), 2, axis=1)  # noqa: E731
        return np.stack([r["y"], up(r["u"]), up(r["v"])])

    gf = [2, -3, -1, 4] if is_b else [-4, 1]
    pre = oracle.inter_predict(residue, motion, to444(refs[0]), to444(refs[1]) if is_b else None, gf, fs)
    want = oracle.finish_frame(pre, bitdepth, fmt)

    def to_fd(r):
        if fmt == "yuv420":
            return FrameData(bitdepth, fmt, {k: torch.from_numpy(v[None, None]).cuda() for k, v in r.items()})
        return FrameData(bitdepth, fmt, torch.from_numpy(r[None]).cuda())

    got = ctx.reconstruct_frame(torch.from_numpy(residue[None]).cuda(), torch.from_numpy(motion[None]).cuda(),
                                [to_fd(r) for r in refs], is_b, fmt, bitdepth, gf, fs)
    if fmt == "yuv420":
        for k in "yuv":
            assert np.array_equal(got[k][0, 0].cpu().numpy(), want[k]), k
    else:
        assert np.array_equal(got[0].cpu().numpy(), want)


@pytest.mark.parametrize("fmt,bitdepth,hw", [("rgb", 8, (37, 53)), ("yuv420", 8, (36, 50)), ("yuv420", 10, (36, 50)),
                                             ("yuv444", 10, (33, 47)), ("rgb", 16, (5, 3))])
def test_pack_frame(ctx, fmt, bitdepth, hw):
    """Device-side output packing (f3): planar and pixel-interleaved integer samples equal numpy's."""
    import torch

    rng = np.random.default_rng(3)
    h, w = hw
    M = 2**bitdepth - 1
    if fmt == "yuv420":
        planes = [rng.integers(0, M + 1, size=s) for s in ((h, w), (h // 2, w // 2), (h // 2, w // 2))]
        data = {k: torch.from_numpy((p / M).astype(np.float32)[None, None]).cuda() for k, p in zip("yuv", planes)}
    else:
        planes = list(rng.integers(0, M + 1, size=(3, h, w)))
        data = torch.from_numpy((np.stack(planes) / M).astype(np.float32)[None]).cuda()
    dt = np.uint8 if bitdepth <= 8 else np.uint16
    got = ctx.pack_frame(data, bitdepth, fmt).cpu().numpy().view(dt)
    assert np.array_equal(got, np.concatenate([p.reshape(-1) for p in planes]).astype(dt))
    if fmt != "yuv420":
        got = ctx.pack_frame(data, bitdepth, fmt, interleaved=True).cpu().numpy().view(dt)
        assert np.array_equal(got, np.stack(planes).transpose(1, 2, 0).reshape(-1).astype(dt))
    # a batch: three copies as consecutive slices of one buffer (one launch) and as separate tensors (fallback)
    want3 = np.concatenate([p.reshape(-1) for p in planes] * 3).astype(dt)
    flat = torch.cat([t.reshape(-1) for t in ((data["y"], data["u"], data["v"]) if fmt == "yuv420" else (data,))] * 3)
    n_fr = flat.numel() // 3
    if fmt == "yuv420":
        ny, nc = h * w, (h // 2) * (w // 2)
        batch = [{"y": flat[i * n_fr:i * n_fr + ny].view(1, 1, h, w),
                  "u": flat[i * n_fr + ny:i * n_fr + ny + nc].view(1, 1, h // 2, w // 2),
                  "v": flat[i * n_fr + ny + nc:(i + 1) * n_fr].view(1, 1, h // 2, w // 2)} for i in range(3)]
        loose = [{k: v.clone() for k, v in data.items()} for _ in range(3)]
    else:
        batch = [flat[i * n_fr:(i + 1) * n_fr].view(1, 3, h, w) for i in range(3)]
        loose = [data.clone() for _ in range(3)]
    launches = ctx.launch_count()
    assert np.array_equal(ctx.pack_frames(batch, bitdepth, fmt).cpu().numpy().view(dt), want3)
    assert ctx.launch_count() == launches + 1
    assert np.array_equal(ctx.pack_frames(loose, bitdepth, fmt).cpu().numpy().view(dt), want3)


@pytest.mark.parametrize("name,fmt", [("gop5_64x96_yuv420", "yuv420"), ("gop3_40x56_rgb", "rgb"),
                                      ("gop3_48x72_yuv420_bilinear", "yuv420"), ("gop3_40x56_rgb_bicubic", "rgb"),
                                      ("gop3_48x72_yuv420_sinc6", "yuv420"), ("gop4_40x56_rgb_sinc12", "rgb")])
def test_gop_decode_video(ctx, name, fmt, tmp_path):
    """decode_video on a P/B stream against frames decoded by the UNMODIFIED reference."""
    from coolchic_b200.bitstream.decode import decode_video

    path = os.path.join(GOLDEN, name + ".cool")
    gold = np.load(os.path.join(GOLDEN, name + "_frames.npz"))
    out = str(tmp_path / ("o.yuv" if fmt == "yuv420" else "o.ppm"))
    frames = decode_video(path, decoded_path=out if fmt == "yuv420" else None)
    n = len(frames)
    assert sorted(frames) == sorted(str(i) for i in range(n))
    bad = tot = 0
    for k, fd in frames.items():
        assert fd.frame_data_type == fmt and fd.bitdepth == 8
        if fmt == "yuv420":
            for c in "yuv":
                a = np.round(fd.data[c][0, 0].numpy() * 255).astype(np.int32)
                b = gold[f"{k}_{c}"].astype(np.int32)
                assert np.abs(a - b).max() <= 1
                bad += int((a != b).sum())
                tot += a.size
        else:
            a = np.round(fd.data[0].numpy() * 255).astype(np.int32)
            b = gold[k].astype(np.int32)
            assert np.abs(a - b).max() <= 1
            bad += int((a != b).sum())
            tot += a.size
    # the oracle itself differs from the reference in at most 1 sample (sinc-6 fixture, tests/test_oracle.py):
    # rounding ties of the fp32 coefficient evaluation; the device equals the oracle
    assert bad <= (1 if name.endswith("sinc6") else 0)
    if fmt == "yuv420":
        h, w = frames["0"].data["y"].shape[-2:]
        assert os.path.getsize(out) == n * (h * w * 3 // 2)  # planar frames appended in display order


def test_gop8_1080p_yuv420_vs_oracle(ctx, oracle, seed_stream, tmp_path):
    """BASELINE configs[4] shape: 1080p YUV420 hierarchical-B GOP with sinc-8 warps, 8 frames (15 Cool-chics: intra
    hop, residue / motion mop): every sample of every frame equals the oracle pipeline's (decode_video on the
    CPU port), and the planar file equals the device-packed samples."""
    import sys

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pipeline  # the oracle's whole-stream decode (test infrastructure)

    from coolchic_b200 import synth
    from coolchic_b200.bitstream.decode import decode_video_bytes

    n = 8
    data = synth.make_video_stream(ctx, seed_stream, 1080, 1920, n, "yuv420", 8, 8, seed=2)
    out = str(tmp_path / "gop.yuv")
    frames = decode_video_bytes(data, decoded_path=out)
    assert sorted(frames, key=int) == [str(i) for i in range(n)]
    oracle.set_threads(0)
    want = pipeline.decode_video(data)
    raw = np.fromfile(out, dtype=np.uint8)
    assert raw.size == n * 1080 * 1920 * 3 // 2
    off = 0
    for i in range(n):
        fmt, bd, planes = want[i]
        assert (fmt, bd) == ("yuv420", 8)
        for c in "yuv":
            got = frames[str(i)].data[c][0, 0].numpy()
            assert np.array_equal(got, planes[c]), (i, c)
            lv = np.round(planes[c] * 255).astype(np.uint8).reshape(-1)
            assert np.array_equal(raw[off:off + lv.size], lv), (i, c)  # written file: planar, display order
            off += lv.size


# ----------------------------------------------------------------------------------------------
# optional branches of the synthesis input / output
@pytest.mark.parametrize("name", ["img_48x72_rgb_common_randomness", "img_50x70_rgb_final_bicubic",
                                  "img_44x60_yuv420_final_bilinear", "img_40x56_yuv444_10bit_arm24",
                                  "img_48x64_rgb_arm8_1hidden"])
def test_optional_synthesis_branches(ctx, oracle, name):
    """Common randomness and bilinear / bicubic final resize on the device: raw synthesis output vs the
    oracle (same fp32 sequence, Box-Muller through the canonical log / cos: bit-exact), decoded image vs the
    UNMODIFIED reference's (oracle/gen_golden_modes.py)."""
    from coolchic_b200 import synth
    from coolchic_b200._desc import desc_from_header
    from coolchic_b200.bitstream.decode import decode_video

    path = os.path.join(GOLDEN, name + ".cool")
    data = open(path, "rb").read()
    _, f, c, nn_bytes, payload = synth.parse_single_image(data)
    desc = desc_from_header(c)
    raw = ctx.decode_coolchic(desc, nn_bytes, payload).cpu().numpy()[0]
    nn = oracle.decode_nn(desc, nn_bytes)
    lat, _ = oracle.decode_latents(desc, nn, payload)
    want = oracle.synthesize(desc, nn, lat)
    assert np.array_equal(raw, want)
    gold = np.load(os.path.join(GOLDEN, name + ".npz"))
    fd = decode_video(path, None)["0"]
    M = 2**fd.bitdepth - 1
    assert fd.bitdepth == (10 if "10bit" in name else 8)
    for k in gold.files:
        got = np.round((fd.data[k][0, 0] if k in "yuv" else fd.data[0]).numpy() * M).astype(np.int32)
        assert np.abs(got - gold[k].astype(np.int32)).max() <= 1
        assert (got != gold[k]).sum() <= 4  # rounding ties only


def test_common_randomness_1080p_properties(ctx, seed_stream):
    """Full-size common-randomness stream: decodes, deterministic, and the noise half of the input matters."""
    from coolchic_b200 import synth
    from coolchic_b200._desc import desc_from_header

    data = synth.make_image_stream(ctx, seed_stream, 1080, 1920, "rgb", 8, (0, 6), None, seed=1,
                                   overrides={"flag_common_randomness": 1})
    _, f, c, nn_bytes, payload = synth.parse_single_image(data)
    desc = desc_from_header(c)
    a = ctx.decode_coolchic(desc, nn_bytes, payload)
    b = ctx.decode_coolchic(desc, nn_bytes, payload)
    assert a.shape == (1, 3, 1080, 1920) and bool((a == b).all()) and bool(a.isfinite().all())
    plain = synth.make_image_stream(ctx, seed_stream, 1080, 1920, "rgb", 8, (0, 6), None, seed=1)
    _, _, c2, nn2, pay2 = synth.parse_single_image(plain)
    p = ctx.decode_coolchic(desc_from_header(c2), nn2, pay2)
    assert float((a - p).abs().mean()) > 1e-3


def test_fused_synthesis_equals_layer_kernels(ctx, seed_stream):
    """The fused synthesis kernel (tile + halo, shared-memory 3x3 stages) against the one-kernel-per-layer
    path: bit-identical on every architecture of the fused family that the streams use (3 / 4 / 5 / 2 output
    channels, 0-2 3x3 layers, with and without stabiliser, common randomness), odd sizes and tiny frames."""
    import torch

    from coolchic_b200 import synth
    from coolchic_b200._desc import desc_from_header

    cases = [
        ((131, 203), (0, 6), None, None),                                   # hop, 3 channels, 2 x 3x3
        ((70, 50), (0, 3), None, synth._syn_overrides(16, 4, 4)),           # P residue: 4 channels
        ((64, 96), (0, 4), None, synth._syn_overrides(16, 5, 3)),           # B residue: 5 channels, one 3x3
        ((48, 80), (2, 5), "nearest", synth._syn_overrides(16, 2, 2)),      # motion: 2 channels, no 3x3, resize
        ((40, 56), (0, 3), None, {"flag_common_randomness": 1}),            # 8 inputs, stabiliser on 4
        ((17, 9), (0, 2), None, None),                                      # smaller than one tile
    ]
    try:
        for size, lat, fin, ov in cases:
            cc, h, _ = synth.make_coolchic(ctx, seed_stream, size, lat, None, seed=2, final_upsampling_type=fin, overrides=ov)
            h2 = type(h)()
            rest = h2.read_header(cc)
            d = desc_from_header(h2)
            nnb = rest[:h2.get_value("nn_n_bytes")]
            lb = rest[h2.get_value("nn_n_bytes"):][:h2.get_value("n_bytes_latent")]
            ctx.set_fused_synthesis(True)
            n0 = ctx.launch_count()
            a = ctx.decode_coolchic(d, nnb, lb)
            n_fused = ctx.launch_count() - n0
            ctx.set_fused_synthesis(False)
            n0 = ctx.launch_count()
            b = ctx.decode_coolchic(d, nnb, lb)
            n_layers = ctx.launch_count() - n0
            assert torch.equal(a, b), (size, lat)
            assert n_fused < n_layers, (size, n_fused, n_layers)  # the fused kernel did run
    finally:
        ctx.set_fused_synthesis(True)


def test_corrupt_streams_fail_cleanly_on_the_device(ctx, seed_stream):
    """Fuzz on the device: bit flips in the NN payload and in the range-coded payload of a small stream.  Every
    decode returns -- an image (garbage is fine) or a CcdError -- and the context keeps working afterwards."""
    import random

    import torch

    from coolchic_b200 import _native, synth
    from coolchic_b200._desc import desc_from_header

    cc, h, _ = synth.make_coolchic(ctx, seed_stream, (96, 160), (0, 4), None, seed=9)
    h2 = type(h)()
    rest = h2.read_header(cc)
    d = desc_from_header(h2)
    n_nn, n_lat = h2.get_value("nn_n_bytes"), h2.get_value("n_bytes_latent")
    nnb, lb = rest[:n_nn], rest[n_nn:n_nn + n_lat]
    good = ctx.decode_coolchic(d, nnb, lb)
    rng = random.Random(3)
    n_err = n_ok = 0
    for trial in range(24):
        a, b = bytearray(nnb), bytearray(lb)
        tgt = a if trial % 3 == 0 else b
        for _ in range(rng.randint(1, 6)):
            tgt[rng.randrange(len(tgt))] ^= 1 << rng.randrange(8)
        if trial % 5 == 4:
            b = b[: rng.randrange(1, len(b))]  # truncated payload: missing words read as zero
        try:
            out = ctx.decode_coolchic(d, bytes(a), bytes(b))
            assert out.shape == good.shape
            n_ok += 1
        except _native.CcdError as e:
            assert e.code in (-1, -2, -3, -4)
            n_err += 1
    assert n_ok + n_err == 24
    assert torch.equal(ctx.decode_coolchic(d, nnb, lb), good)  # the context is still healthy


def test_integration_stub_b_runs_against_the_reference_header(ctx, kodim14):
    """INTEGRATION.md, stub B, executed as documented: the code block is taken from the file, pointed at the in-tree
    library, and driven with what the REFERENCE's own VideoHeader / FrameHeader / CoolChicHeader objects return for
    the sample stream (tests/golden/reference_headers.json, written by oracle/gen_golden_reference_headers.py): its
    output equals this package's decode of the same Cool-chic."""
    import json
    import re
    import types

    import torch

    class RecordedCoolChicHeader:
        """Replays the reference CoolChicHeader's get_value / get_coolchic_parameter for kodim14.cool."""

        def __init__(self, rec):
            self.rec = rec

        def get_value(self, key):
            v = self.rec["values"][key]
            if key in ("nn_q_step", "nn_expgol_cnt"):  # DescriptorCoolChic: get_value(module, "weight" / "bias")
                return types.SimpleNamespace(get_value=lambda m, k: v[m][k])
            return v

        def get_coolchic_parameter(self):
            return types.SimpleNamespace(**self.rec["parameter"])

    rec = json.load(open(os.path.join(GOLDEN, "reference_headers.json")))["kodim14"]
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    code = re.search(r"```python\n(# coolchic/bitstream/component/coolchic_b200_stub\.py.*?)```", text, re.S).group(1)
    code = code.replace('"/path/to/cool-chic_b200/csrc/libccdec.so"', repr(os.path.join(ROOT, "cool-chic_b200", "csrc", "libccdec.so")))
    stub = types.ModuleType("coolchic_b200_stub")
    exec(compile(code, "INTEGRATION.md:stub_b", "exec"), stub.__dict__)
    rest = kodim14["data"][sum(rec["header_bytes"].values()):]  # what the reference's three read_header calls leave
    cc = RecordedCoolChicHeader(rec)
    n_nn, n_lat = cc.get_value("nn_n_bytes"), cc.get_value("n_bytes_latent")
    out, none = stub.encode_decode_coolchic(cc, rest[:n_nn], "decode", rest[n_nn:n_nn + n_lat])
    torch.cuda.synchronize()
    assert none is None
    want = ctx.decode_coolchic(kodim14["desc"], kodim14["nn_bytes"], kodim14["lat_bytes"])
    assert torch.equal(out, want)
