"""Generate tests/golden/reference_headers.json: what the UNMODIFIED reference's own host classes
(coolchic.utils.codingstructure.CodingStructure, coolchic.bitstream.header.*) compute for the inputs that
tests/test_host_logic.py::test_against_reference_classes and
tests/test_gpu_decode.py::test_integration_stub_b_runs_against_the_reference_header compare against:

* the coding order (display order, references, frame type, depth) of a few GOP structures;
* the parse of kodim14.cool: bytes taken by each header, every CoolChicHeader field, the CoolChicEncoderParameter
  the header yields;
* the reference's parse of Cool-chic headers written by coolchic_b200.synth at other image sizes (the bytes are
  stored too, so that a test can tell whether the writer still emits what the reference parsed).

TEST INFRASTRUCTURE ONLY.  Needs a checkout of the reference (Orange-OpenSource/Cool-Chic 5.0.1):

    python oracle/gen_golden_reference_headers.py PATH_TO_COOL_CHIC_CHECKOUT
"""
import dataclasses
import json
import os
import sys
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "..", "tests", "golden")

# (n_frames, intra_pos, p_pos)
GOPS = [(1, [0], []), (5, [0], [4]), (9, [0], [8]), (8, [0, 7], []), (8, [0], [1, 2, 3, 4, 5, 6, 7]),
        (33, [0], [32]), (10, [0], [6, 9]), (17, [0, 16], [8])]
# image sizes of the synthetic headers (latent_resolution (0, 6), hyperlatent_resolution (4, 6))
SIZES = [(1080, 1920), (2160, 3840), (17, 33), (1, 1), (129, 7)]


def _plain(x):
    """JSON-able copy of a header value / parameter field."""
    if hasattr(x, "arm") and hasattr(x, "get_value"):  # DescriptorCoolChic
        return {m: {k: x.get_value(m, k) for k in ("weight", "bias")} for m in ("arm", "ifce", "upsampling", "synthesis")}
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    if isinstance(x, bool):
        return int(x)
    return x


def main(ref_root):
    sys.path.insert(0, os.path.join(HERE, ".."))
    sys.path.insert(0, os.path.join(HERE, "refshim"))
    sys.path.insert(0, ref_root)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # SyntaxWarning: invalid escape sequences in the reference's docstrings
        from coolchic.bitstream.header.header import CoolChicHeader, FrameHeader, VideoHeader
        from coolchic.utils.codingstructure import CodingStructure
    import coolchic

    if not os.path.abspath(coolchic.__file__).startswith(os.path.abspath(ref_root)):
        raise RuntimeError(f"imported coolchic from {coolchic.__file__}, not from {ref_root}")
    import coolchic_b200  # noqa: F401
    from coolchic_b200 import synth

    gops = []
    for n, ip, pp in GOPS:
        cs = CodingStructure(n_frames=n, intra_pos=list(ip), p_pos=list(pp))
        frames = []
        for i in range(n):
            f = cs.get_frame_from_coding_order(i)
            frames.append([f.display_order, list(f.index_references), f.frame_type, f.depth])
        gops.append({"n_frames": n, "intra_pos": ip, "p_pos": pp, "coding_order": frames})

    data = open(os.path.join(GOLD, "kodim14.cool"), "rb").read()
    sizes = []
    rest = data
    for hdr in (VideoHeader(), FrameHeader()):
        nxt = hdr.read_header(rest)
        sizes.append(len(rest) - len(nxt))
        rest = nxt
    cc = CoolChicHeader()
    nxt = cc.read_header(rest)
    sizes.append(len(rest) - len(nxt))
    param = cc.get_coolchic_parameter()
    kodim14 = {
        "header_bytes": dict(zip(("video", "frame", "coolchic"), sizes)),
        "values": {e.name: _plain(cc.get_value(e.name)) for e in cc._get_all_header_elements()},
        "parameter": {f.name: _plain(getattr(param, f.name)) for f in dataclasses.fields(param)},
    }

    # the synthetic headers are written from our parse of the sample's header, like the test does
    from coolchic_b200.bitstream.header import CoolChicHeader as OurCC
    from coolchic_b200.bitstream.header import FrameHeader as OurFrame
    from coolchic_b200.bitstream.header import VideoHeader as OurVideo

    ours = OurCC()
    ours.read_header(OurFrame().read_header(OurVideo().read_header(data)))
    headers = []
    for hw in SIZES:
        b = synth.make_coolchic_header(ours, hw, (0, 6), (4, 6)).to_bytes()
        r = CoolChicHeader()
        r.read_header(b)
        p = r.get_coolchic_parameter()
        headers.append({"img_size": list(hw), "latent_resolution": [0, 6], "hyperlatent_resolution": [4, 6],
                        "bytes": b.hex(), "size_per_latent": _plain(p.size_per_latent),
                        "input_features_ifce": _plain(p.input_features_ifce),
                        "flag_is_hyperlatent": _plain(p.flag_is_hyperlatent)})

    out = {"source": "Orange-OpenSource/Cool-Chic 5.0.1, unmodified, through oracle/gen_golden_reference_headers.py",
           "coding_structures": gops, "kodim14": kodim14, "synthetic_headers": headers}
    path = os.path.join(GOLD, "reference_headers.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
