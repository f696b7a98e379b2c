"""The operator's encode half: ``encode_decode_coolchic(mode="encode")`` / ``encode_coolchics`` over
``ccd_encode_many`` (one data-parallel ARM pass, one range-coder warp per job).  Payloads must be byte-identical to
the files the reference wrote, to the wavefront encoder (``ccd_encode_latents`` mode 1) and to the oracle.  The
argument checks of the operator run before the library is touched and are tested without a GPU."""
import ctypes
import glob
import os

import numpy as np
import pytest
from conftest import GOLDEN

gpu = pytest.mark.gpu

# the synthetic architectures of test_gpu_decode.py: (H, W), latent_resolution, hyperlatent_resolution, overrides
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


def _grids(desc, flat):
    """Flat decode-order latents -> the reference encoder's list (finest first, [1, 1, h_i, w_i] int64)."""
    import torch

    from coolchic_b200 import _native

    flat = flat.cpu() if isinstance(flat, torch.Tensor) else torch.from_numpy(np.asarray(flat))
    _, offs = _native.latent_layout(desc)
    return [flat[offs[g]:offs[g] + desc.grid_h[g] * desc.grid_w[g]].to(torch.int64).view(1, 1, desc.grid_h[g], desc.grid_w[g])
            for g in range(desc.n_grids)]


def _stream(ctx, seed_stream, case, seed=3):
    """(desc, nn_bytes, payload, latents on the device) of a synthetic Cool-chic made by the wavefront encoder."""
    from coolchic_b200 import synth
    from coolchic_b200._desc import desc_from_header

    hw, lr, hr, ov = case
    ov = dict(ov)
    fut = ov.pop("final_upsampling_type", None)
    if ov.get("output_feature_ifce", 1) == 0:
        ov["ifce_resolution"] = None
    cc, header, lat = synth.make_coolchic(ctx, seed_stream, hw, lr, hr, seed=seed, final_upsampling_type=fut, overrides=ov)
    h2 = type(header)()
    rest = h2.read_header(cc)
    n_nn, n_lat = h2.get_value("nn_n_bytes"), h2.get_value("n_bytes_latent")
    return desc_from_header(h2), rest[:n_nn], rest[n_nn:n_nn + n_lat], lat


def _encode_raw(ctx, desc, nn_bytes, lat_dev, cap):
    """ccd_encode_many called directly on device int8 latents with a chosen capacity -> (rc, job)."""
    import torch

    from coolchic_b200 import _native

    words = torch.zeros((max(cap, 1),), dtype=torch.int32, device=ctx.torch_device)
    job = (_native.CcdEncodeJob * 1)()
    job[0].desc = ctypes.pointer(desc)
    job[0].nn_bytes = nn_bytes
    job[0].nn_nbytes = len(nn_bytes)
    job[0].d_latents = lat_dev.data_ptr()
    job[0].d_words = words.data_ptr()
    job[0].cap_words = cap
    rc = ctx._lib.ccd_encode_many(ctx._h, job, 1, ctx._stream())
    torch.cuda.synchronize()
    return rc, job[0]


# ------------------------------------------------------------------------------------------
@gpu
def test_kodim14_through_the_operator(ctx, oracle, kodim14):
    import torch

    from coolchic_b200.bitstream.coolchic import encode_decode_coolchic
    from coolchic_b200.bitstream.header import CoolChicHeader

    data = kodim14["data"]
    video, frames, _ = _split_file(data)
    cc_section = data[len(video) + len(frames[0][0]):]  # the Cool-chic section: after the video and frame headers
    h = CoolChicHeader()
    h.read_header(cc_section)
    want_n = h.get_value("n_bytes_latent")
    assert want_n == 30952
    h.set_value("n_bytes_latent", 0)  # the operator must set it
    d = kodim14["desc"]
    out, cc_bytes = encode_decode_coolchic(h, kodim14["nn_bytes"], "encode", enc_quantized_latent=_grids(d, kodim14["latents"]))
    torch.cuda.synchronize()
    assert cc_bytes == cc_section  # header + NN + the 30 952 latent bytes constriction wrote, byte for byte
    assert h.get_value("n_bytes_latent") == want_n
    assert ctx.last_slow == [0]
    assert tuple(out.shape) == (1, 3, 512, 768)
    dec = ctx.decode_coolchic(d, kodim14["nn_bytes"], kodim14["lat_bytes"])
    assert torch.equal(out, dec)
    nn = oracle.decode_nn(d, kodim14["nn_bytes"])
    assert np.array_equal(out[0].cpu().numpy(), oracle.synthesize(d, nn, kodim14["latents"]))


def _split_file(data):
    """video header bytes, [(frame header bytes, [(CoolChicHeader, nn, latent payload)])], trailing bytes"""
    from coolchic_b200.bitstream.decode import _split_coolchic
    from coolchic_b200.bitstream.header import FrameHeader, VideoHeader

    vh = VideoHeader()
    rest = vh.read_header(data)
    video = data[:len(data) - len(rest)]
    frames = []
    for _ in range(vh.get_coding_structure().get_max_coding_order() + 1):
        fh = FrameHeader()
        r2 = fh.read_header(rest)
        fbytes = rest[:len(rest) - len(r2)]
        ccs = []
        for _ in range(2 if fh.get_value("frame_type") in ("P", "B") else 1):
            h, nn, lat, r2 = _split_coolchic(r2)
            ccs.append((h, bytes(nn), bytes(lat)))
        frames.append((fbytes, ccs))
        rest = r2
    return video, frames, rest


GOLDEN_FILES = sorted(os.path.basename(p)[:-5] for p in glob.glob(os.path.join(GOLDEN, "*.cool")))


@gpu
@pytest.mark.parametrize("name", GOLDEN_FILES)
def test_every_golden_file_reencodes_to_itself(ctx, name):
    """Decode every Cool-chic of the file (latents kept), re-encode all of them in ONE encode_coolchics call,
    reassemble video / frame / Cool-chic headers: the file again, byte for byte."""
    from coolchic_b200._desc import desc_from_header
    from coolchic_b200.bitstream.coolchic import encode_coolchics

    data = open(os.path.join(GOLDEN, name + ".cool"), "rb").read()
    video, frames, tail = _split_file(data)
    assert tail == b""
    ccs = [cc for _, f in frames for cc in f]
    descs = [desc_from_header(h) for h, _, _ in ccs]
    outs, lats = ctx.decode_many(descs, [c[1] for c in ccs], [c[2] for c in ccs], want_latents=True)
    for h, _, _ in ccs:
        h.set_value("n_bytes_latent", 0)
    enc = encode_coolchics([c[0] for c in ccs], [c[1] for c in ccs], [_grids(d, lat) for d, lat in zip(descs, lats)])
    it = iter(enc)
    rebuilt = video + b"".join(fb + b"".join(next(it)[1] for _ in f) for fb, f in frames)
    assert rebuilt == data
    for (out, _), dec in zip(enc, outs):
        assert bool((out == dec).all())


@gpu
@pytest.mark.parametrize("case", CASES, ids=[f"{c[0][0]}x{c[0][1]}-{i}" for i, c in enumerate(CASES)])
def test_architectures_equal_mode1_and_oracle(ctx, oracle, seed_stream, case):
    import torch

    d, nnb, payload, lat = _stream(ctx, seed_stream, case)
    nn = oracle.decode_nn(d, nnb)
    _, p1, slow1 = ctx.encode_latents(d, nn, latents=lat)  # the wavefront encoder (mode 1)
    (p,), (out,) = ctx.encode_many([d], [nnb], [lat])
    assert p == p1 == payload == oracle.encode_latents(d, nn, lat.cpu().numpy())
    assert ctx.last_slow == [slow1]
    assert torch.equal(out, ctx.decode_coolchic(d, nnb, payload))


@gpu
def test_slow_path(ctx, oracle, kodim14, seed_stream):
    import torch

    d, nnb = kodim14["desc"], kodim14["nn_bytes"]
    nn = oracle.decode_nn(d, nnb)
    lat_s, payload_s, slow_s = ctx.encode_latents(d, nn, seed=77)  # drawn from the model: far from the mode often
    assert slow_s > 1000
    (p,), _ = ctx.encode_many([d], [nnb], [lat_s], synthesize=False)
    assert p == payload_s and ctx.last_slow == [slow_s]
    # a small grid of alternating extremes: every symbol outside the window, the longest words
    d2, nnb2, _, _ = _stream(ctx, seed_stream, ((24, 40), (0, 3), None, {}))
    m = d2.n_symbols()
    alt = torch.tensor([-64 if i % 2 == 0 else 63 for i in range(m)], dtype=torch.int8, device=ctx.torch_device)
    nn2 = oracle.decode_nn(d2, nnb2)
    (p2,), _ = ctx.encode_many([d2], [nnb2], [alt], synthesize=False)
    _, p1, slow1 = ctx.encode_latents(d2, nn2, latents=alt)
    assert p2 == p1 == oracle.encode_latents(d2, nn2, alt.cpu().numpy())
    assert ctx.last_slow == [slow1] and slow1 > m // 2
    rc, job = _encode_raw(ctx, d2, nnb2, alt, m + 1)
    assert rc == 0 and job.n_words <= m + 1 and job.n_words == len(p2) // 4


@gpu
def test_int64_arm_path_equals_mode1(ctx, oracle, seed_stream):
    """An ARM weight above 2^31 in fixed point: arm_fits_int32 rejects the int32-operand kernel (its first test
    is |W| <= INT32_MAX), both encoders run the int64 path."""
    from coolchic_b200 import synth
    from coolchic_b200._desc import desc_from_header
    from coolchic_b200.bitstream.expgolomb import encode_exp_golomb

    header = synth.make_coolchic_header(seed_stream.header, (48, 80), (0, 4), None)
    d = desc_from_header(header)
    nn = synth.adapt_nn(seed_stream.desc, seed_stream.nn, d)
    shift = 16 + int(d.qshift[0])
    nn[0] = (1 << (31 - shift)) + 1  # first ARM weight: (q << shift) > INT32_MAX
    _, counts = synth.join_nn(d, synth.split_nn(d, nn))
    nn_bytes, pad = encode_exp_golomb(nn.tolist(), counts)
    header.set_value("nn_n_bytes", len(nn_bytes))
    header.set_value("nn_n_bit_pad", pad)
    d = desc_from_header(header)
    assert np.array_equal(oracle.decode_nn(d, nn_bytes), nn)
    lat = synth.tile_latents(seed_stream.desc, seed_stream.latents, d, 4)
    lat_dev, p1, slow1 = ctx.encode_latents(d, nn, latents=lat)
    (p,), _ = ctx.encode_many([d], [nn_bytes], [lat_dev], synthesize=False)
    assert p == p1 == oracle.encode_latents(d, nn, lat_dev.cpu().numpy())
    assert ctx.last_slow == [slow1]


@gpu
@pytest.mark.parametrize("hw,lr", [((1080, 1920), (0, 6)), ((2160, 3840), (0, 7))], ids=["1080p-7grids", "4k-8grids"])
def test_full_size_payload(ctx, seed_stream, hw, lr):
    d, nnb, payload, lat = _stream(ctx, seed_stream, (hw, lr, None, {}), seed=1)
    (p,), _ = ctx.encode_many([d], [nnb], [lat], synthesize=False)
    assert p == payload


@gpu
def test_batch_of_301_mixed_streams(ctx, seed_stream):
    import torch

    items = [_stream(ctx, seed_stream, c, seed=20 + i) for i, c in enumerate(CASES)]
    single = [ctx.encode_many([d], [nnb], [lat]) for d, nnb, _, lat in items]
    sub = [items[i % len(items)] for i in range(301)]
    pays, outs = ctx.encode_many([x[0] for x in sub], [x[1] for x in sub], [x[3] for x in sub])
    for i in range(301):
        (p1,), (o1,) = single[i % len(items)]
        assert pays[i] == p1 == sub[i][2], i
        assert torch.equal(outs[i], o1), i


@gpu
def test_errors_leave_the_context_working(ctx, kodim14, seed_stream):
    import torch

    from coolchic_b200 import _native
    from coolchic_b200.bitstream.coolchic import encode_decode_coolchic

    d, nnb = kodim14["desc"], kodim14["nn_bytes"]
    good = ctx.decode_coolchic(d, nnb, kodim14["lat_bytes"])
    for v in (64, -65):
        grids = _grids(d, kodim14["latents"])
        grids[2][0, 0, 1, 1] = v
        with pytest.raises(ValueError):
            encode_decode_coolchic(kodim14["header"], nnb, "encode", enc_quantized_latent=grids)
        lat = torch.from_numpy(kodim14["latents"]).to(ctx.torch_device).clone()
        lat[1000] = v
        rc, job = _encode_raw(ctx, d, nnb, lat, d.n_symbols() + 1)
        assert rc == -1 and job.status == -1  # CCD_ERR_ARG
        assert torch.equal(ctx.decode_coolchic(d, nnb, kodim14["lat_bytes"]), good)
    lat = torch.from_numpy(kodim14["latents"]).to(ctx.torch_device)
    rc, job = _encode_raw(ctx, d, nnb, lat, 100)  # 7 738 words needed
    assert rc == -1 and job.n_words == len(kodim14["lat_bytes"]) // 4
    with pytest.raises(_native.CcdError):
        _native._check(rc)
    assert torch.equal(ctx.decode_coolchic(d, nnb, kodim14["lat_bytes"]), good)
    rc, job = _encode_raw(ctx, d, nnb, lat, job.n_words)  # exactly enough
    assert rc == 0


@gpu
def test_integration_stub_b_encode_branch(ctx, kodim14):
    """INTEGRATION.md stub B, executed as documented, in encode mode with a header object: the sample's Cool-chic
    section comes back byte for byte."""
    import re
    import types

    import torch

    from conftest import ROOT
    from coolchic_b200.bitstream.header import CoolChicHeader

    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    code = re.search(r"```python\n(# coolchic/bitstream/component/coolchic_b200_stub\.py.*?)```", text, re.S).group(1)
    code = code.replace('"/path/to/cool-chic_b200/csrc/libccdec.so"', repr(os.path.join(ROOT, "cool-chic_b200", "csrc", "libccdec.so")))
    stub = types.ModuleType("coolchic_b200_stub")
    exec(compile(code, "INTEGRATION.md:stub_b", "exec"), stub.__dict__)
    data = kodim14["data"]
    video, frames, _ = _split_file(data)
    cc_section = data[len(video) + len(frames[0][0]):]
    h = CoolChicHeader()
    h.read_header(cc_section)
    h.set_value("n_bytes_latent", 0)
    d = kodim14["desc"]
    out, cc_bytes = stub.encode_decode_coolchic(h, kodim14["nn_bytes"], "encode",
                                                enc_quantized_latent=_grids(d, kodim14["latents"]))
    torch.cuda.synchronize()
    assert cc_bytes == cc_section
    assert torch.equal(out, ctx.decode_coolchic(d, kodim14["nn_bytes"], kodim14["lat_bytes"]))


# ------------------------------------------------------------------------------------------
# host-side checks: no GPU needed
def test_operator_checks_its_arguments_before_the_device(kodim14):
    import torch

    from coolchic_b200.bitstream.coolchic import encode_coolchics, encode_decode_coolchic

    d = kodim14["desc"]
    lat = kodim14["latents"]
    sizes = [(d.grid_h[g], d.grid_w[g]) for g in range(d.n_grids)]
    grids = [torch.zeros((1, 1, h, w), dtype=torch.int32) for h, w in sizes]
    with pytest.raises(ValueError):
        encode_decode_coolchic(kodim14["header"], kodim14["nn_bytes"], "encode", enc_quantized_latent=grids[:-1])
    bad = list(grids)
    bad[0] = torch.zeros((1, 1, sizes[0][0], sizes[0][1] + 1))
    with pytest.raises(ValueError):
        encode_decode_coolchic(kodim14["header"], kodim14["nn_bytes"], "encode", enc_quantized_latent=bad)
    bad = [g.clone() for g in grids]
    bad[-1][0, 0, 0, 0] = 64
    with pytest.raises(ValueError):
        encode_coolchics([kodim14["header"]], [kodim14["nn_bytes"]], [bad])
    with pytest.raises(ValueError):
        encode_decode_coolchic(kodim14["header"], kodim14["nn_bytes"], "encode", enc_quantized_latent=None)
    assert lat.size == d.n_symbols()
    if not torch.cuda.is_available():
        # valid arguments and no device: an error, never a CPU fallback
        with pytest.raises(RuntimeError):
            encode_decode_coolchic(kodim14["header"], kodim14["nn_bytes"], "encode", enc_quantized_latent=grids)


def test_latent_list_to_decode_order(kodim14):
    import torch

    from coolchic_b200.bitstream.coolchic import latents_to_decode_order

    d = kodim14["desc"]
    flat = latents_to_decode_order(d, _grids(d, kodim14["latents"]))
    assert flat.dtype == torch.int8 and np.array_equal(flat.numpy(), kodim14["latents"])
