"""Per-Cool-chic decode operator.

Mirror of the reference's ``coolchic/bitstream/component/coolchic.py:29-207``
(``encode_decode_coolchic``, both modes): same signature, same errors, same return value
(raw, un-clamped, un-rounded float32 synthesis output ``[1, C, H, W]``, plus the Cool-chic's bytes
in encode mode) -- but every stage (NN parsing, integer ARM + IFCE, range decoding or encoding,
upsampling, synthesis, final resize) runs in ``libccdec.so`` on the GPU.  ``CoolChicDecoder`` is the module-style wrapper (``load`` /
``forward``) named in BASELINE.json; the reference itself has no such class (SURVEY F2).
"""
from typing import List, Literal, Optional, Sequence, Tuple

import torch
from torch import Tensor

from .. import _native
from .._desc import CcdCoolChicDesc, desc_from_header
from .header import CoolChicHeader


def encode_decode_coolchic(
    header: CoolChicHeader,
    bytes_nn: bytes,
    mode: Literal["encode", "decode"],
    dec_bytes_latent: Optional[bytes] = None,
    enc_quantized_latent: Optional[List[Tensor]] = None,
    verbosity: int = 0,
    device: int = 0,
) -> Tuple[Tensor, Optional[bytes]]:
    """One Cool-chic through the reference operator's contract.

    ``mode="decode"``: returns ``(synthesis_output [1, C, H, W] float32 CUDA, None)``.
    ``mode="encode"``: ``enc_quantized_latent`` holds one tensor per grid in ``size_per_latent`` order (finest first,
    hyperlatents included), each ``[1, 1, h_i, w_i]`` of any dtype.  The latents are range-coded on the device,
    ``n_bytes_latent`` is set on ``header`` and the function returns ``(synthesis_output of those latents,
    header.to_bytes() + bytes_nn + latent_bytes)``."""
    if mode == "encode":
        if enc_quantized_latent is None:
            raise ValueError(
                "Trying to encode cool_chic latent without indicating the quantized latent value. "
                "Found enc_quantized_latent=None. It should be a list of integer Tensor."
            )
        (out, cc_bytes), = encode_coolchics([header], [bytes_nn], [enc_quantized_latent], device=device,
                                            verbosity=verbosity)
        return out, cc_bytes
    if mode != "decode":
        raise ValueError(f"Unknown mode {mode}")
    if dec_bytes_latent is None:
        raise ValueError(
            "Trying to encode cool_chic latent with dec_bytes_latent=None. "
            "The argument dec_bytes_latent should represent the bytes of the bitstream."
        )
    dec = CoolChicDecoder(device=device).load(header, bytes_nn, dec_bytes_latent)
    out = dec.forward()
    if verbosity:
        print(header.pretty_string())
    if verbosity >= 2:
        # the reference's per-stage line (component/coolchic.py:199-205): seconds spent on the NN weights, the IFCE
        # contexts, the latents (IFCE included) and upsampling + synthesis.  Here: host parse of the NN payload + staging
        # + H2D | 0 (the IFCE layer is evaluated on the fly inside the entropy kernel) | entropy kernel | float-tail kernels
        t = dec.last_timing
        time_neural_net, time_ifce = t["upload_ms"] / 1e3, 0.0
        time_latent, time_syn = t["entropy_ms"] / 1e3, t["synthesis_ms"] / 1e3
        print(f"{time_neural_net:6.2f} {time_ifce:6.2f} {time_latent:6.2f} {time_syn:6.2f} ")
    return out, None


class CoolChicDecoder:
    """``load(header, bytes_nn, bytes_latent)`` then ``forward() -> Tensor[1, C, H, W]``."""

    def __init__(self, device: int = 0):
        self.device = device
        self.desc: Optional[CcdCoolChicDesc] = None
        self._nn: Optional[bytes] = None
        self._lat: Optional[bytes] = None
        self.latents: Optional[Tensor] = None
        self.last_timing = {}

    def load(self, header: CoolChicHeader, bytes_nn: bytes, bytes_latent: bytes) -> "CoolChicDecoder":
        if bytes_nn is None or bytes_latent is None:
            raise ValueError("CoolChicDecoder.load: bytes_nn and bytes_latent must be bytes objects")
        n_nn, n_lat = header.get_value("nn_n_bytes"), header.get_value("n_bytes_latent")
        if len(bytes_nn) < n_nn or len(bytes_latent) < n_lat:
            raise ValueError(
                f"Cool-chic payload truncated: header announces {n_nn} NN bytes and {n_lat} latent bytes, "
                f"got {len(bytes_nn)} and {len(bytes_latent)}."
            )
        self.desc = desc_from_header(header)
        self._nn = bytes(bytes_nn[:n_nn])
        self._lat = bytes(bytes_latent[:n_lat])
        return self

    @torch.no_grad()
    def forward(self, want_latents: bool = False) -> Tensor:
        if self.desc is None:
            raise RuntimeError("CoolChicDecoder.forward called before load()")
        ctx = _native.get_context(self.device)
        if want_latents:
            out, self.latents = ctx.decode_coolchic(self.desc, self._nn, self._lat, want_latents=True)
        else:
            out = ctx.decode_coolchic(self.desc, self._nn, self._lat)
        self.last_timing = ctx.last_timing()
        return out

    __call__ = forward


def decode_coolchics(headers: Sequence[CoolChicHeader], bytes_nn: Sequence[bytes], bytes_latent: Sequence[bytes],
                     device: int = 0, finish=None) -> List[Tensor]:
    """Decode several independent Cool-chics CONCURRENTLY (one persistent CTA per stream).  ``finish[i]`` =
    (bitdepth, frame_data_type) for the Cool-chic of an I frame: the synthesis kernel then writes the finished
    frame (decode.py:191-206 fused into its epilogue) instead of the raw output."""
    ctx = _native.get_context(device)
    descs = [desc_from_header(h) for h in headers]
    outs, _ = ctx.decode_many(descs, [bytes(b) for b in bytes_nn], [bytes(b) for b in bytes_latent], finish=finish)
    return outs


def latents_to_decode_order(desc: CcdCoolChicDesc, latents: Sequence[Tensor]) -> Tensor:
    """The reference encoder's per-grid latent list (``size_per_latent`` order: finest first, each ``[1, 1, h_i, w_i]``,
    any dtype) -> the flat int8 array in decode order (coarsest grid first, each row-major) that the library codes.
    Raises ValueError for a wrong grid count, a wrong shape or a value outside [-64, 63] (AC_MAX_VAL,
    constants.py:9-11): the reference's range coder has no symbol for it."""
    if len(latents) != desc.n_grids:
        raise ValueError(f"enc_quantized_latent has {len(latents)} grids, the header describes {desc.n_grids}")
    grids = []
    for g in range(desc.n_grids):
        t = latents[g]
        if not isinstance(t, Tensor):
            t = torch.as_tensor(t)
        want = (1, 1, int(desc.grid_h[g]), int(desc.grid_w[g]))
        if tuple(t.shape) != want:
            raise ValueError(f"latent grid {g} has shape {tuple(t.shape)}, expected {want}")
        t = t.detach().to(torch.int64)  # like the reference (FIXED_POINT_DTYPE)
        if t.numel() and (int(t.min()) < -64 or int(t.max()) > 63):
            raise ValueError(f"latent grid {g} holds values in [{int(t.min())}, {int(t.max())}], outside [-64, 63]")
        grids.append(t.reshape(-1))
    return torch.cat(grids[::-1]).to(torch.int8)


def encode_coolchics(headers: Sequence[CoolChicHeader], bytes_nn: Sequence[bytes], latents_lists: Sequence[Sequence[Tensor]],
                     device: int = 0, verbosity: int = 0) -> List[Tuple[Tensor, bytes]]:
    """Encode several independent Cool-chics (all those of a GOP or of a dataset) in ONE library call: the ARM of
    every symbol of every Cool-chic is one data-parallel pass on the GPU, then one range-coder warp per Cool-chic.
    ``latents_lists[i]`` is Cool-chic i's ``enc_quantized_latent``.  Sets ``n_bytes_latent`` on every header and
    returns, per Cool-chic, ``(synthesis_output [1, C, H, W], header.to_bytes() + bytes_nn + latent_bytes)``.
    Every argument is checked before the device is touched."""
    if not (len(headers) == len(bytes_nn) == len(latents_lists)):
        raise ValueError("encode_coolchics: headers, bytes_nn and latents_lists differ in length")
    descs = [desc_from_header(h) for h in headers]
    flat = [latents_to_decode_order(d, lats) for d, lats in zip(descs, latents_lists)]
    ctx = _native.get_context(device)
    payloads, outs = ctx.encode_many(descs, [bytes(b) for b in bytes_nn], flat)
    t = ctx.last_timing()
    res = []
    for h, nn, pay, out in zip(headers, bytes_nn, payloads, outs):
        h.set_value("n_bytes_latent", len(pay))
        res.append((out, h.to_bytes() + bytes(nn) + pay))
        if verbosity:
            print(h.pretty_string())
        if verbosity >= 2:
            # as in decode mode: host parse + staging + H2D | 0 (IFCE inside the ARM pass) | ARM pass + range coder |
            # float tail
            print(f"{t['upload_ms'] / 1e3:6.2f} {0.0:6.2f} {t['entropy_ms'] / 1e3:6.2f} {t['synthesis_ms'] / 1e3:6.2f} ")
    return res
