"""Host-side mirrors of the reference interface: headers, coding structure, writers."""
import json
import os

import numpy as np
import pytest
from conftest import GOLDEN


def test_kodim14_headers(kodim14):
    v, f, c = kodim14["video"], kodim14["frame"], kodim14["header"]
    assert (v.get_value("n_frames"), v.get_value("intra_pos"), v.get_value("p_pos")) == (1, [0], [])
    assert (f.get_value("frame_type"), f.get_value("frame_data_type"), f.get_value("bitdepth")) == ("I", "rgb", 8)
    # SURVEY Appendix E
    assert c.get_value("img_size") == [512, 768] and c.get_value("n_latent_grids") == 10
    assert c.get_value("latent_resolution") == [0, 6] and c.get_value("hyperlatent_resolution") == [4, 6]
    assert [c.get_value(f"syn_layer_{i}") for i in range(4)] == [
        "48-1-linear-relu", "3-1-linear-none", "3-3-residual-relu", "3-3-residual-none"]
    assert (c.get_value("nn_n_bytes"), c.get_value("nn_n_bit_pad"), c.get_value("n_bytes_latent")) == (2020, 6, 30952)
    d = kodim14["desc"]
    assert d.grid_sizes() == [(512, 768), (256, 384), (128, 192), (64, 96), (32, 48), (32, 48), (16, 24), (16, 24),
                              (8, 12), (8, 12)]
    assert list(d.grid_ifce_in)[:10] == [9, 8, 7, 0, 0, 0, 0, 0, 0, 0]
    assert list(d.qshift) == [-7, -6, -6, -5, -8, 0, -10, -11] and list(d.expgol) == [5, 5, 3, 3, 6, 0, 7, 9]
    assert d.n_symbols() == 526272


def test_headers_roundtrip(kodim14):
    data = kodim14["data"]
    v, f, c = kodim14["video"], kodim14["frame"], kodim14["header"]
    assert v.to_bytes() == data[:8] and f.to_bytes() == data[8:13] and c.to_bytes() == data[13:48]


def test_header_errors():
    from coolchic_b200.bitstream.header import BitWriter, CoolChicHeader, FrameHeader

    with pytest.raises(ValueError):
        FrameHeader().read_header(b"\x00")  # truncated
    w = BitWriter()
    with pytest.raises(ValueError):
        w.write(5000, 12, name="display_index")
    with pytest.raises(ValueError):
        w.write(-9000, 14, signed=True, name="global_flow")
    h = CoolChicHeader()
    with pytest.raises(ValueError):
        h.set_value("not_a_field", 1)


def test_pb_frame_header_roundtrip():
    from coolchic_b200.bitstream.header import FrameHeader

    f = FrameHeader()
    f._values.update(display_index=7, frame_type="B", frame_data_type="yuv420", bitdepth=10,
                     index_references=[4, 8], global_flow=[-3, 2, 5, -1], warp_filter_size=8)
    b = f.to_bytes()
    g = FrameHeader()
    rest = g.read_header(b + b"xyz")
    assert rest == b"xyz"
    for k in ("display_index", "frame_type", "frame_data_type", "bitdepth", "index_references", "global_flow",
              "warp_filter_size"):
        assert g.get_value(k) == f.get_value(k)


GOPS = [(1, [0], []), (5, [0], [4]), (9, [0], [8]), (8, [0, 7], []), (8, [0], [1, 2, 3, 4, 5, 6, 7]),
        (33, [0], [32]), (10, [0], [6, 9]), (17, [0, 16], [8])]
# coding order (display indices) of a hierarchical-B GOP of 9: codingstructure.py:398-434
GOLDEN_GOP9 = [0, 8, 4, 2, 1, 3, 6, 5, 7]


def test_coding_structure_golden():
    from coolchic_b200.utils.codingstructure import CodingStructure

    cs = CodingStructure(n_frames=9, intra_pos=[0], p_pos=[8])
    order = [cs.get_frame_from_coding_order(i).display_order for i in range(9)]
    assert order == GOLDEN_GOP9
    assert cs.get_frame_from_display_order(4).index_references == [0, 8]
    assert cs.get_frame_from_display_order(8).frame_type == "P" and cs.get_frame_from_display_order(5).depth == 4
    with pytest.raises(AssertionError):
        CodingStructure(n_frames=4, intra_pos=[1], p_pos=[3])
    with pytest.raises(AssertionError):
        CodingStructure(n_frames=4, intra_pos=[0], p_pos=[2])


def test_against_reference_classes(kodim14):
    """Our host mirrors vs what the reference's own CodingStructure and CoolChicHeader computed for the same inputs
    (tests/golden/reference_headers.json, written by oracle/gen_golden_reference_headers.py)."""
    from coolchic_b200 import synth
    from coolchic_b200.utils.codingstructure import CodingStructure

    gold = json.load(open(os.path.join(GOLDEN, "reference_headers.json")))
    assert [(g["n_frames"], g["intra_pos"], g["p_pos"]) for g in gold["coding_structures"]] == GOPS
    for g in gold["coding_structures"]:
        ours = CodingStructure(n_frames=g["n_frames"], intra_pos=list(g["intra_pos"]), p_pos=list(g["p_pos"]))
        assert len(g["coding_order"]) == g["n_frames"]
        for i, want in enumerate(g["coding_order"]):
            a = ours.get_frame_from_coding_order(i)
            assert [a.display_order, a.index_references, a.frame_type, a.depth] == want
    p_ref, p = gold["kodim14"]["parameter"], kodim14["header"].get_coolchic_parameter()
    assert [tuple(s) for s in p_ref["size_per_latent"]] == p.size_per_latent
    assert p_ref["input_features_ifce"] == p.input_features_ifce and p_ref["flag_is_hyperlatent"] == p.flag_is_hyperlatent
    assert [tuple(g["img_size"]) for g in gold["synthetic_headers"]] == [(1080, 1920), (2160, 3840), (17, 33), (1, 1), (129, 7)]
    for g in gold["synthetic_headers"]:
        h = synth.make_coolchic_header(kodim14["header"], tuple(g["img_size"]), (0, 6), (4, 6))
        assert h.to_bytes().hex() == g["bytes"]  # the header the reference parsed
        assert [tuple(s) for s in g["size_per_latent"]] == h.get_coolchic_parameter().size_per_latent
        assert g["input_features_ifce"] == h.get_coolchic_parameter().input_features_ifce


def test_exp_golomb_python(kodim14, oracle):
    from coolchic_b200 import synth
    from coolchic_b200.bitstream.expgolomb import decode_exp_golomb, encode_exp_golomb

    d = kodim14["desc"]
    nn = oracle.decode_nn(d, kodim14["nn_bytes"])
    _, counts = synth.join_nn(d, synth.split_nn(d, nn))
    payload, pad = encode_exp_golomb(nn.tolist(), counts)
    assert payload == kodim14["nn_bytes"] and pad == 6
    assert decode_exp_golomb(payload, pad, counts) == nn.tolist()
    vals = [0, 1, -1, 2, -2, 65535, -65535, 17]
    for k in (0, 1, 5, 12):
        b, p = encode_exp_golomb(vals, [k] * len(vals))
        assert decode_exp_golomb(b, p, [k] * len(vals)) == vals
    with pytest.raises(ValueError):
        encode_exp_golomb([1, 2], [0])


def test_writers(tmp_path):
    import torch

    from coolchic_b200.io import FrameData, save_frame_data_to_file

    x = torch.linspace(0, 1, 3 * 4 * 6).reshape(1, 3, 4, 6)
    fd = FrameData(8, "rgb", x)
    assert fd.img_size == (4, 6) and fd.n_pixels == 24
    save_frame_data_to_file(fd, str(tmp_path / "a.ppm"))
    raw = (tmp_path / "a.ppm").read_bytes()
    assert raw.startswith(b"P6\n6 4\n255\n") and len(raw) == 11 + 72
    save_frame_data_to_file(fd, str(tmp_path / "a.png"))
    from PIL import Image

    im = np.asarray(Image.open(tmp_path / "a.png"))
    assert np.array_equal(im, np.round(x[0].permute(1, 2, 0).numpy() * 255).astype(np.uint8))
    yuv = {"y": torch.rand(1, 1, 4, 6), "u": torch.rand(1, 1, 2, 3), "v": torch.rand(1, 1, 2, 3)}
    fy = FrameData(10, "yuv420", yuv)
    save_frame_data_to_file(fy, str(tmp_path / "v.yuv"))
    save_frame_data_to_file(fy, str(tmp_path / "v.yuv"), append=True)
    assert (tmp_path / "v.yuv").stat().st_size == 2 * 2 * (24 + 6 + 6)
    with pytest.raises(AssertionError):
        save_frame_data_to_file(fy, str(tmp_path / "v.png"))
    with pytest.raises(AssertionError):
        save_frame_data_to_file(fd, str(tmp_path / "a.bmp"))


def test_synthetic_header_and_nn_layout(kodim14, oracle):
    from coolchic_b200 import synth
    from coolchic_b200._desc import desc_from_header

    d = kodim14["desc"]
    nn = oracle.decode_nn(d, kodim14["nn_bytes"])
    for hw, lr, hr, nsym in [((1080, 1920), (0, 6), None, 2764710), ((2160, 3840), (0, 7), None, 11059110),
                             ((512, 768), (0, 6), (4, 6), 526272)]:
        h = synth.make_coolchic_header(kodim14["header"], hw, lr, hr)
        d2 = desc_from_header(h)
        assert d2.n_symbols() == nsym  # SURVEY 8a/8d symbol counts
        nn2 = synth.adapt_nn(d, nn, d2)
        assert len(nn2) == oracle.nn_counts(d2)[0]
    h = synth.make_coolchic_header(kodim14["header"], (512, 768), (0, 6), (4, 6))
    assert np.array_equal(synth.adapt_nn(d, nn, desc_from_header(h)), nn)


def test_output_shape_from_header_alone():
    """decode.output_shape (used by ranks that did not decode a Cool-chic to allocate the broadcast buffer)
    against the channel counts / sizes of the committed GOP fixture: I residue 3, P residue 4, B residue 5,
    P motion 2, B motion 4 channels, all at frame size."""
    from coolchic_b200.bitstream import decode as dec

    data = open(os.path.join(GOLDEN, "gop5_64x96_yuv420.cool"), "rb").read()
    from coolchic_b200.bitstream.header import VideoHeader

    v = VideoHeader()
    rest = v.read_header(data)
    seen = {}
    for _ in range(5):
        fh, ccs, rest = dec._parse_frame(rest)
        for name, (h, _, _) in ccs.items():
            shp = dec.output_shape(h)
            assert shp[0] == 1 and shp[2:] == (64, 96)
            seen[(fh.get_value("frame_type"), name)] = shp[1]
    assert seen == {("I", "residue"): 3, ("P", "residue"): 4, ("P", "motion"): 2, ("B", "residue"): 5, ("B", "motion"): 4}


def test_corrupt_headers_and_payloads_never_crash():
    """Fuzz: random byte flips in the header / NN-payload region of a real stream.  The host parser either
    raises a Python exception or yields a description that the C-ABI accepts or rejects with an error code --
    never a crash, never a silent out-of-range descriptor (ccd_nn_count / ccd_latent_count validate it)."""
    import ctypes
    import random

    import numpy as np

    from coolchic_b200 import _native
    from coolchic_b200._desc import desc_from_header
    from coolchic_b200.bitstream.header import CoolChicHeader, FrameHeader, VideoHeader

    data = open(os.path.join(GOLDEN, "kodim14.cool"), "rb").read()
    lib = _native.load_library()
    rng = random.Random(7)
    outcomes = {"parse_error": 0, "rejected": 0, "nn_error": 0, "accepted": 0}
    for trial in range(300):
        b = bytearray(data[:4096])
        for _ in range(rng.randint(1, 4)):
            b[rng.randrange(0, 64 if trial % 2 else 2048)] ^= 1 << rng.randrange(8)
        try:
            rest = VideoHeader().read_header(bytes(b))
            rest = FrameHeader().read_header(rest)
            c = CoolChicHeader()
            rest = c.read_header(rest)
            d = desc_from_header(c)
        except Exception:
            outcomes["parse_error"] += 1
            continue
        n = lib.ccd_nn_count(ctypes.byref(d))
        if n < 0 or _native.latent_layout(d)[0] < 0:
            outcomes["rejected"] += 1
            continue
        try:
            ints = _native.decode_nn(d, rest[: max(0, c.get_value("nn_n_bytes"))])
            assert len(ints) == n and np.abs(ints).max() < 2**40
            outcomes["accepted"] += 1
        except _native.CcdError as e:
            assert e.code in (-1, -2, -4)
            outcomes["nn_error"] += 1
    assert sum(outcomes.values()) == 300 and outcomes["accepted"] > 0 and outcomes["parse_error"] + outcomes["rejected"] + outcomes["nn_error"] > 0


def test_corrupt_coolchic_header_raises_value_error():
    """ADVICE r1: impossible header values surface as ValueError (not ZeroDivisionError / IndexError)."""
    import pytest

    from coolchic_b200._desc import desc_from_header
    from coolchic_b200.bitstream.header import CoolChicHeader, FrameHeader, VideoHeader

    data = open(os.path.join(GOLDEN, "kodim14.cool"), "rb").read()
    rest = FrameHeader().read_header(VideoHeader().read_header(data))
    for key, bad in (("img_size", [0, 768]), ("n_layer_synthesis", 0), ("latent_resolution", [6, 0]),
                     ("hyperlatent_resolution", [6, 4])):
        c = CoolChicHeader()
        c.read_header(rest)
        c._values[key] = bad
        with pytest.raises(ValueError):
            desc_from_header(c)


def test_bit_reader_window_grows_on_demand():
    """The header bit reader starts with a 256-byte window (shifting a 64 KB integer per field made batch parsing slow) and
    widens it when a read crosses the end: same values as one big integer, and a clean error on truncated data."""
    import random

    import pytest

    from coolchic_b200.bitstream.header import BitReader

    rng = random.Random(5)
    data = bytes(rng.randrange(256) for _ in range(3000))
    big, n_bits = int.from_bytes(data, "big"), 8 * len(data)
    br, pos = BitReader(data), 0
    while pos + 40 < n_bits:
        n = rng.choice((1, 3, 7, 8, 13, 16, 24, 32, 37))
        want = (big >> (n_bits - pos - n)) & ((1 << n) - 1)
        assert br.read(n) == want, pos
        pos += n
    assert br.pos == pos
    br = BitReader(data[:300])
    br.read(8 * 290)          # one read across the first window
    br.read(8 * 10)
    with pytest.raises(ValueError):
        br.read(1)
    # signed fields: sign-magnitude, as the reference writes them
    assert BitReader(bytes([0b10000101])).read(8, signed=True) == -5 and BitReader(bytes([0b00000101])).read(8, signed=True) == 5
