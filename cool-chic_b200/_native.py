"""ctypes binding of ``csrc/libccdec.so`` (C-ABI in ``include/ccdec.h``).

There is no CPU fallback: if the shared library is missing or no CUDA device is present,
loading / context creation raises ``RuntimeError``.  PyTorch tensors are only used as owners
of device memory (``tensor.data_ptr()``) and of the CUDA stream.
"""
import ctypes
import os
import threading
from typing import List, Optional, Sequence

import numpy as np
import torch

from ._desc import CCD_MAX_GRIDS, CcdCoolChicDesc

_HERE = os.path.dirname(os.path.abspath(__file__))
# CCD_LIB lets a developer load the instrumented build (csrc/libccdec_prof.so)
LIB_PATH = os.environ.get("CCD_LIB") or os.path.join(_HERE, "csrc", "libccdec.so")

CCD_OK = 0
ERROR_NAMES = {
    -1: "CCD_ERR_ARG", -2: "CCD_ERR_NN_TRUNCATED", -3: "CCD_ERR_DESYNC", -4: "CCD_ERR_UNSUPPORTED",
    -5: "CCD_ERR_NOMEM", -6: "CCD_ERR_CUDA", -7: "CCD_ERR_NO_DEVICE",
}

EXPORTS = [
    "ccd_version", "ccd_sizeof_desc", "ccd_last_error", "ccd_create", "ccd_destroy", "ccd_nn_count",
    "ccd_latent_count", "ccd_decode_nn", "ccd_decode_many", "ccd_decode_coolchic", "ccd_decode_latents",
    "ccd_synthesize", "ccd_encode_latents", "ccd_encode_many", "ccd_finish_frame", "ccd_inter_predict", "ccd_reconstruct_frame",
    "ccd_pack_frame",
    "ccd_pack_samples",
    "ccd_debug_laplace_domain", "ccd_debug_last_status", "ccd_debug_launch_count", "ccd_debug_set_producer_mask", "ccd_debug_set_fused_synthesis", "ccd_last_timing",
]


class CcdJob(ctypes.Structure):
    _fields_ = [
        ("desc", ctypes.POINTER(CcdCoolChicDesc)),
        ("nn_bytes", ctypes.c_char_p),
        ("nn_nbytes", ctypes.c_size_t),
        ("latent_bytes", ctypes.c_char_p),
        ("latent_nbytes", ctypes.c_size_t),
        ("d_out", ctypes.c_void_p),
        ("d_latents", ctypes.c_void_p),
        ("status", ctypes.c_int32),
        ("finish_bitdepth", ctypes.c_int32),
        ("finish_type", ctypes.c_int32),
        ("d_out_u", ctypes.c_void_p),
        ("d_out_v", ctypes.c_void_p),
    ]


class CcdEncodeJob(ctypes.Structure):
    _fields_ = [
        ("desc", ctypes.POINTER(CcdCoolChicDesc)),
        ("nn_bytes", ctypes.c_char_p),
        ("nn_nbytes", ctypes.c_size_t),
        ("d_latents", ctypes.c_void_p),
        ("d_words", ctypes.c_void_p),
        ("cap_words", ctypes.c_int64),
        ("d_out", ctypes.c_void_p),
        ("n_words", ctypes.c_int64),
        ("status", ctypes.c_int32),
        ("slow", ctypes.c_int32),
    ]


class CcdError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERROR_NAMES.get(code, code)}: {msg}")
        self.code = code


_lib = None
_lib_lock = threading.Lock()


def load_library():
    """Load libccdec.so (once).  Raises RuntimeError if it has not been built."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C cool-chic_b200/csrc`).  There is no CPU fallback."
            )
        L = ctypes.CDLL(LIB_PATH)
        vp, sz, i64, ci = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int64, ctypes.c_int
        pd = ctypes.POINTER(CcdCoolChicDesc)
        L.ccd_version.restype = ci
        L.ccd_sizeof_desc.restype = ci
        L.ccd_last_error.restype = ctypes.c_char_p
        L.ccd_last_error.argtypes = [vp]
        L.ccd_create.restype = ci
        L.ccd_create.argtypes = [ci, ctypes.POINTER(vp)]
        L.ccd_destroy.restype = None
        L.ccd_destroy.argtypes = [vp]
        L.ccd_nn_count.restype = i64
        L.ccd_nn_count.argtypes = [pd]
        L.ccd_latent_count.restype = i64
        L.ccd_latent_count.argtypes = [pd, vp]
        L.ccd_decode_nn.restype = i64
        L.ccd_decode_nn.argtypes = [pd, ctypes.c_char_p, sz, vp, sz]
        L.ccd_decode_many.restype = ci
        L.ccd_decode_many.argtypes = [vp, ctypes.POINTER(CcdJob), ci, vp]
        L.ccd_decode_coolchic.restype = ci
        L.ccd_decode_coolchic.argtypes = [vp, pd, ctypes.c_char_p, sz, ctypes.c_char_p, sz, vp, vp, vp]
        L.ccd_decode_latents.restype = ci
        L.ccd_decode_latents.argtypes = [vp, pd, vp, ctypes.c_char_p, sz, vp, vp]
        L.ccd_synthesize.restype = ci
        L.ccd_synthesize.argtypes = [vp, pd, vp, vp, vp, vp]
        L.ccd_encode_latents.restype = ci
        L.ccd_encode_latents.argtypes = [vp, pd, vp, ci, ctypes.c_uint64, vp, vp, i64, vp, vp, vp]
        L.ccd_encode_many.restype = ci
        L.ccd_encode_many.argtypes = [vp, ctypes.POINTER(CcdEncodeJob), ci, vp]
        L.ccd_finish_frame.restype = ci
        L.ccd_finish_frame.argtypes = [vp, vp, ci, ci, ci, ci, vp, vp, vp, vp]
        L.ccd_inter_predict.restype = ci
        L.ccd_inter_predict.argtypes = [vp, vp, ci, vp, ci, vp, vp, ci, ci, ci, vp, ci, vp, vp]
        L.ccd_reconstruct_frame.restype = ci
        L.ccd_reconstruct_frame.argtypes = [vp, vp, ci, vp, ci, vp, vp, ci, ci, ci, ci, ci, vp, ci, vp, vp]
        L.ccd_pack_frame.restype = ci
        L.ccd_pack_frame.argtypes = [vp, vp, ci, ci, ci, ci, ci, ci, vp, vp]
        L.ccd_pack_samples.restype = ci
        L.ccd_pack_samples.argtypes = [vp, vp, ctypes.c_size_t, ci, ci, vp, vp]
        L.ccd_debug_laplace_domain.restype = ci
        L.ccd_debug_laplace_domain.argtypes = [vp, ci, ci, vp, vp]
        L.ccd_debug_last_status.restype = ci
        L.ccd_debug_last_status.argtypes = [vp, vp]
        L.ccd_debug_launch_count.restype = ctypes.c_uint64
        L.ccd_debug_launch_count.argtypes = []
        L.ccd_debug_set_producer_mask.restype = ci
        L.ccd_debug_set_producer_mask.argtypes = [vp, ctypes.c_uint32]
        L.ccd_debug_set_fused_synthesis.restype = ci
        L.ccd_debug_set_fused_synthesis.argtypes = [vp, ci]
        L.ccd_last_timing.restype = ci
        L.ccd_last_timing.argtypes = [vp, vp]
        if L.ccd_sizeof_desc() != ctypes.sizeof(CcdCoolChicDesc):
            raise RuntimeError("CcdCoolChicDesc layout mismatch between Python and libccdec.so")
        _lib = L
        return _lib


def _check(rc: int) -> None:
    if rc != CCD_OK:
        msg = load_library().ccd_last_error(None)
        raise CcdError(rc, msg.decode() if msg else "")


def decode_nn(desc: CcdCoolChicDesc, nn_bytes: bytes) -> np.ndarray:
    """Host exp-Golomb decode of the NN payload -> int64 array (module/param order)."""
    L = load_library()
    n = L.ccd_nn_count(ctypes.byref(desc))
    if n < 0:
        _check(int(n))
    out = np.zeros(int(n), dtype=np.int64)
    got = L.ccd_decode_nn(ctypes.byref(desc), nn_bytes, len(nn_bytes), out.ctypes.data_as(ctypes.c_void_p), out.size)
    if got < 0:
        _check(int(got))
    return out


def latent_layout(desc: CcdCoolChicDesc):
    L = load_library()
    offs = (ctypes.c_int64 * CCD_MAX_GRIDS)()
    n = L.ccd_latent_count(ctypes.byref(desc), offs)
    if n < 0:
        _check(int(n))
    return int(n), [int(offs[i]) for i in range(desc.n_grids)]


class Context:
    """One decoder context per CUDA device (``ccd_create`` / ``ccd_destroy``)."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        if not torch.cuda.is_available():
            raise RuntimeError("cool-chic_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback.")
        self.device = int(device)
        h = ctypes.c_void_p()
        _check(self._lib.ccd_create(self.device, ctypes.byref(h)))
        self._h = h
        self.torch_device = torch.device("cuda", self.device)
        self.last_slow: List[int] = []  # encode_many: symbols outside the 31-symbol window, per job

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.ccd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.torch_device).cuda_stream)

    # ---- whole Cool-chic(s) -----------------------------------------------------------
    def decode_many(self, descs: Sequence[CcdCoolChicDesc], nn_bytes: Sequence[bytes],
                    latent_bytes: Sequence[bytes], want_latents: bool = False, finish=None):
        """Decode n independent Cool-chics concurrently.  Returns (outputs, latents) where
        outputs[i] is a float32 CUDA tensor [1, C, H, W] (raw synthesis output).
        ``finish[i] = (bitdepth, frame_data_type)`` (or None) asks for decode_frame's frame tail fused into the
        synthesis kernel: outputs[i] is then the FINISHED frame in FrameData layout ([1, 3, H, W], or the
        y / u / v dictionary for yuv420)."""
        n = len(descs)
        jobs = (CcdJob * n)()
        outs, lats = [], []
        # all outputs are slices of ONE buffer, frame after frame, plane after plane: a batch of finished planar frames
        # is then already in output order (pack_frames: one launch, one copy to the host for the whole batch)
        sizes = []
        for i in range(n):
            d = descs[i]
            fin = finish[i] if finish is not None else None
            if fin is not None and fin[1] == "yuv420":
                sizes.append(d.img_h * d.img_w + 2 * (d.img_h // 2) * (d.img_w // 2))
            else:
                sizes.append(d.n_out_channels * d.img_h * d.img_w)
        slab = torch.empty((sum(sizes),), dtype=torch.float32, device=self.torch_device)
        off = 0
        for i in range(n):
            d = descs[i]
            fin = finish[i] if finish is not None else None
            jobs[i].desc = ctypes.pointer(d)
            jobs[i].nn_bytes = nn_bytes[i]
            jobs[i].nn_nbytes = len(nn_bytes[i])
            jobs[i].latent_bytes = latent_bytes[i]
            jobs[i].latent_nbytes = len(latent_bytes[i])
            if fin is not None and fin[1] == "yuv420":
                h, w = d.img_h, d.img_w
                ny, nc = h * w, (h // 2) * (w // 2)
                out = {"y": slab[off:off + ny].view(1, 1, h, w),
                       "u": slab[off + ny:off + ny + nc].view(1, 1, h // 2, w // 2),
                       "v": slab[off + ny + nc:off + ny + 2 * nc].view(1, 1, h // 2, w // 2)}
                jobs[i].d_out = out["y"].data_ptr()
                jobs[i].d_out_u = out["u"].data_ptr()
                jobs[i].d_out_v = out["v"].data_ptr()
            else:
                out = slab[off:off + sizes[i]].view(1, d.n_out_channels, d.img_h, d.img_w)
                jobs[i].d_out = out.data_ptr()
            off += sizes[i]
            if fin is not None:
                jobs[i].finish_bitdepth = int(fin[0])
                jobs[i].finish_type = _frame_type_code(fin[1])
            outs.append(out)
            if want_latents:
                lat = torch.empty((d.n_symbols(),), dtype=torch.int8, device=self.torch_device)
                lats.append(lat)
                jobs[i].d_latents = lat.data_ptr()
            else:
                jobs[i].d_latents = None
        rc = self._lib.ccd_decode_many(self._h, jobs, n, self._stream())
        _check(rc)
        return outs, (lats if want_latents else None)

    def decode_coolchic(self, desc, nn_bytes: bytes, latent_bytes: bytes, want_latents: bool = False):
        outs, lats = self.decode_many([desc], [nn_bytes], [latent_bytes], want_latents)
        return (outs[0], lats[0]) if want_latents else outs[0]

    # ---- stages -----------------------------------------------------------------------
    def decode_latents(self, desc, nn_ints: np.ndarray, latent_bytes: bytes) -> torch.Tensor:
        nn_ints = np.ascontiguousarray(nn_ints, dtype=np.int64)
        lat = torch.empty((desc.n_symbols(),), dtype=torch.int8, device=self.torch_device)
        _check(self._lib.ccd_decode_latents(self._h, ctypes.byref(desc), nn_ints.ctypes.data_as(ctypes.c_void_p),
                                            latent_bytes, len(latent_bytes), lat.data_ptr(), self._stream()))
        return lat

    def synthesize(self, desc, nn_ints: np.ndarray, latents: torch.Tensor) -> torch.Tensor:
        nn_ints = np.ascontiguousarray(nn_ints, dtype=np.int64)
        assert latents.dtype == torch.int8 and latents.is_cuda and latents.is_contiguous()
        out = torch.empty((1, desc.n_out_channels, desc.img_h, desc.img_w), dtype=torch.float32,
                          device=self.torch_device)
        _check(self._lib.ccd_synthesize(self._h, ctypes.byref(desc), nn_ints.ctypes.data_as(ctypes.c_void_p),
                                        latents.data_ptr(), out.data_ptr(), self._stream()))
        return out

    def encode_latents(self, desc, nn_ints: np.ndarray, latents: Optional[torch.Tensor] = None,
                       seed: Optional[int] = None):
        """Range-encode ``latents`` (mode 1) or draw them from the ARM with ``seed`` (mode 2).
        Returns (latents int8 CUDA tensor, payload bytes, slow_path_count)."""
        nn_ints = np.ascontiguousarray(nn_ints, dtype=np.int64)
        n = desc.n_symbols()
        if latents is None:
            assert seed is not None
            lat = torch.zeros((n,), dtype=torch.int8, device=self.torch_device)
            mode = 2
        else:
            lat = latents.to(self.torch_device, torch.int8).contiguous().clone()
            mode, seed = 1, 0
        cap = n // 2 + 1024
        words = torch.zeros((cap,), dtype=torch.int32, device=self.torch_device)
        n_words = ctypes.c_int64(0)
        slow = ctypes.c_int32(0)
        _check(self._lib.ccd_encode_latents(self._h, ctypes.byref(desc), nn_ints.ctypes.data_as(ctypes.c_void_p),
                                            mode, ctypes.c_uint64(seed), lat.data_ptr(), words.data_ptr(), cap,
                                            ctypes.byref(n_words), ctypes.byref(slow), self._stream()))
        payload = words[: n_words.value].cpu().numpy().astype("<u4").tobytes()
        return lat, payload, int(slow.value)

    def encode_many(self, descs: Sequence[CcdCoolChicDesc], nn_bytes: Sequence[bytes], latents: Sequence,
                    synthesize: bool = True):
        """Range-encode n independent Cool-chics from their latents (``ccd_encode_many``): one data-parallel ARM pass
        over all symbols of all jobs, then one range-coder warp per job.  ``latents[i]``: the job's latents in decode
        order (coarsest grid first, each grid row-major), a tensor or array of any integer dtype with values in
        [-64, 63].  Returns ``(payloads, outputs)``: the latent payload bytes of every job and, with ``synthesize``,
        the raw synthesis output [1, C, H, W] of the given latents (slices of one buffer, as in ``decode_many``),
        else None."""
        n = len(descs)
        dev = self.torch_device
        lats = []
        for i in range(n):
            t = latents[i] if isinstance(latents[i], torch.Tensor) else torch.from_numpy(np.ascontiguousarray(latents[i]))
            if t.numel() != descs[i].n_symbols():
                raise ValueError(f"job {i}: {t.numel()} latents, the descriptor has {descs[i].n_symbols()} symbols")
            if t.dtype != torch.int8 and t.numel() and (int(t.min()) < -64 or int(t.max()) > 63):
                # checked before the int8 conversion, which would wrap such a value (int8 values are checked on the device)
                raise ValueError(f"job {i}: latent value outside [-64, 63]")
            lats.append(t.reshape(-1).to(dev, torch.int8).contiguous())
        caps = [d.n_symbols() + 1 for d in descs]  # at most one word per symbol, plus the seal
        words = torch.empty((sum(caps),), dtype=torch.int32, device=dev)
        outs = []
        if synthesize:
            sizes = [d.n_out_channels * d.img_h * d.img_w for d in descs]
            slab = torch.empty((sum(sizes),), dtype=torch.float32, device=dev)
        jobs = (CcdEncodeJob * n)()
        w_off, o_off = [], 0
        off = 0
        for i in range(n):
            d = descs[i]
            jobs[i].desc = ctypes.pointer(d)
            jobs[i].nn_bytes = nn_bytes[i]
            jobs[i].nn_nbytes = len(nn_bytes[i])
            jobs[i].d_latents = lats[i].data_ptr()
            jobs[i].d_words = words.data_ptr() + 4 * off
            jobs[i].cap_words = caps[i]
            w_off.append(off)
            off += caps[i]
            if synthesize:
                out = slab[o_off:o_off + sizes[i]].view(1, d.n_out_channels, d.img_h, d.img_w)
                jobs[i].d_out = out.data_ptr()
                o_off += sizes[i]
                outs.append(out)
            else:
                jobs[i].d_out = None
        _check(self._lib.ccd_encode_many(self._h, jobs, n, self._stream()))
        # the word counts are on the host now: gather the payloads on the device, then ONE copy to the host
        counts = [int(jobs[i].n_words) for i in range(n)]
        self.last_slow = [int(jobs[i].slow) for i in range(n)]
        flat = torch.cat([words[w_off[i]:w_off[i] + counts[i]] for i in range(n)]) if n else words[:0]
        host = flat.cpu().numpy().astype("<u4").tobytes()
        payloads, at = [], 0
        for c in counts:
            payloads.append(host[4 * at:4 * (at + c)])
            at += c
        return payloads, (outs if synthesize else None)

    def finish_frame(self, raw: torch.Tensor, bitdepth: int, frame_data_type: str):
        """decode_frame tail: round / (420 average) / clamp / round.  raw: [1, 3, H, W] CUDA."""
        assert raw.is_cuda and raw.dtype == torch.float32 and raw.dim() == 4 and raw.size(1) == 3
        raw = raw.contiguous()
        h, w = raw.shape[-2:]
        code = _frame_type_code(frame_data_type)
        if code == 1:
            y = torch.empty((1, 1, h, w), dtype=torch.float32, device=raw.device)
            u = torch.empty((1, 1, h // 2, w // 2), dtype=torch.float32, device=raw.device)
            v = torch.empty_like(u)
            _check(self._lib.ccd_finish_frame(self._h, raw.data_ptr(), h, w, bitdepth, code, y.data_ptr(),
                                              u.data_ptr(), v.data_ptr(), self._stream()))
            return {"y": y, "u": u, "v": v}
        out = torch.empty_like(raw)
        _check(self._lib.ccd_finish_frame(self._h, raw.data_ptr(), h, w, bitdepth, 2 if code == 3 else code,
                                          out.data_ptr(), None, None, self._stream()))
        return out

    @staticmethod
    def _check_inter_shapes(residue, motion, refs, is_b, frame_data_type):
        """The reference fails with a shape error when the Cool-chic outputs or the references do not fit the
        frame (decode.py:159-189); the kernels read raw pointers, so the same conditions are checked here."""
        if residue.dim() != 4 or motion.dim() != 4 or residue.size(0) != 1 or motion.size(0) != 1:
            raise ValueError(f"residue / motion must be [1, C, H, W], found {tuple(residue.shape)} / {tuple(motion.shape)}")
        h, w = residue.shape[-2:]
        if tuple(motion.shape[-2:]) != (h, w):
            raise ValueError(f"motion is {tuple(motion.shape[-2:])}, residue is {(h, w)}")
        n_ref = 2 if is_b else 1
        if residue.size(1) != 3 + n_ref:
            raise ValueError(f"{'B' if is_b else 'P'}-frame residue needs {3 + n_ref} channels, found {residue.size(1)}")
        if motion.size(1) != 2 * n_ref:
            raise ValueError(f"{'B' if is_b else 'P'}-frame motion needs {2 * n_ref} channels, found {motion.size(1)}")
        if len(refs) < n_ref:
            raise ValueError(f"{'B' if is_b else 'P'} frame with {len(refs)} reference frame(s)")
        for r in refs[:n_ref]:
            if r.frame_data_type != frame_data_type:
                raise ValueError(f"reference is {r.frame_data_type}, frame is {frame_data_type}")
            if frame_data_type == "yuv420":
                shapes = [tuple(r.data[k].shape) for k in ("y", "u", "v")]
                if (h | w) & 1 or shapes != [(1, 1, h, w), (1, 1, h // 2, w // 2), (1, 1, h // 2, w // 2)]:
                    raise ValueError(f"yuv420 reference planes {shapes} do not fit a {h}x{w} frame")
            elif tuple(r.data.shape) != (1, 3, h, w):
                raise ValueError(f"reference is {tuple(r.data.shape)}, frame is {(1, 3, h, w)}")
        return h, w

    @staticmethod
    def _ref_planes(r, frame_data_type):
        """(keep-alive tensors, c_void_p[3]) of a reference frame's planes."""
        if frame_data_type == "yuv420":
            ts = [r.data[k].contiguous() for k in ("y", "u", "v")]
        else:
            t = r.data.contiguous()
            ts = [t[0, c] for c in range(3)]
        assert all(t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() for t in ts)
        return ts, (ctypes.c_void_p * 3)(*[t.data_ptr() for t in ts])

    def inter_predict(self, residue, motion, refs, is_b, frame_data_type, global_flow, warp_filter_size):
        """decode_frame P/B branch (bitstream/decode.py:156-189) -> PRE-ROUNDING frame [1,3,H,W] (stage entry
        point for tests; decode_frame uses reconstruct_frame).  References are 4:4:4 here."""
        if frame_data_type == "yuv420":
            raise ValueError("inter_predict takes 4:4:4 references; use reconstruct_frame for yuv420 frames")
        h, w = self._check_inter_shapes(residue, motion, refs, is_b, frame_data_type)
        residue, motion = residue.contiguous(), motion.contiguous()
        r0 = refs[0].data.contiguous()
        r1 = refs[1].data.contiguous() if is_b else None
        out = torch.empty((1, 3, h, w), dtype=torch.float32, device=self.torch_device)
        gf = (ctypes.c_int32 * 4)(*(list(global_flow) + [0, 0, 0, 0])[:4])
        _check(self._lib.ccd_inter_predict(
            self._h, residue.data_ptr(), residue.size(1), motion.data_ptr(), motion.size(1), r0.data_ptr(),
            r1.data_ptr() if is_b else None, h, w, int(is_b), gf, int(warp_filter_size), out.data_ptr(), self._stream()))
        return out

    def reconstruct_frame(self, residue, motion, refs, is_b, frame_data_type, bitdepth, global_flow, warp_filter_size):
        """Whole P/B reconstruction in one kernel (bitstream/decode.py:156-206): prediction from the finished
        reference frames (4:2:0 planes read in place), blending, residue, frame tail.  Returns the finished frame
        in FrameData layout ([1,3,H,W], or the y / u / v dictionary)."""
        h, w = self._check_inter_shapes(residue, motion, refs, is_b, frame_data_type)
        residue, motion = residue.contiguous(), motion.contiguous()
        keep0, p0 = self._ref_planes(refs[0], frame_data_type)
        keep1, p1 = self._ref_planes(refs[1], frame_data_type) if is_b else (None, None)
        dev = self.torch_device
        if frame_data_type == "yuv420":
            data = {"y": torch.empty((1, 1, h, w), dtype=torch.float32, device=dev),
                    "u": torch.empty((1, 1, h // 2, w // 2), dtype=torch.float32, device=dev),
                    "v": torch.empty((1, 1, h // 2, w // 2), dtype=torch.float32, device=dev)}
            outs = [data[k] for k in ("y", "u", "v")]
        else:
            data = torch.empty((1, 3, h, w), dtype=torch.float32, device=dev)
            outs = [data[0, c] for c in range(3)]
        po = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in outs])
        gf = (ctypes.c_int32 * 4)(*(list(global_flow) + [0, 0, 0, 0])[:4])
        _check(self._lib.ccd_reconstruct_frame(
            self._h, residue.data_ptr(), residue.size(1), motion.data_ptr(), motion.size(1), p0, p1,
            _frame_type_code(frame_data_type), int(bitdepth), h, w, int(is_b), gf, int(warp_filter_size), po,
            self._stream()))
        del keep0, keep1
        return data

    def pack_frame(self, data, bitdepth: int, frame_data_type: str, interleaved: bool = False,
                   sample_bytes: Optional[int] = None) -> torch.Tensor:
        """Finished frame (FrameData.data on the device) -> integer samples on the device, uint8 / uint16:
        planar (y, u, v one after the other: the .yuv file order) or pixel-interleaved HWC (PPM / PNG order)."""
        if frame_data_type == "yuv420":
            planes = [data[k].contiguous() for k in ("y", "u", "v")]
            h, w = planes[0].shape[-2:]
            cs = 1
        else:
            t = data.contiguous()
            h, w = t.shape[-2:]
            planes = [t[0, c] for c in range(3)]
            cs = 0
        if sample_bytes is None:
            sample_bytes = 1 if bitdepth <= 8 else 2
        n = h * w + 2 * (h >> cs) * (w >> cs)
        out = torch.empty((n,), dtype=torch.uint8 if sample_bytes == 1 else torch.int16, device=self.torch_device)
        pp = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in planes])
        _check(self._lib.ccd_pack_frame(self._h, pp, h, w, cs, int(bitdepth), sample_bytes, int(bool(interleaved)),
                                        out.data_ptr(), self._stream()))
        return out

    def pack_frames(self, frames, bitdepth: int, frame_data_type: str, sample_bytes: Optional[int] = None) -> torch.Tensor:
        """A batch of finished frames (what decode_many returns with ``finish``) -> the planar integer samples of all
        of them, frame after frame, in ONE device tensor.  Frames that are consecutive slices of one buffer (decode_many
        allocates them so) are converted by a single launch; anything else falls back to one pack_frame per frame."""
        if sample_bytes is None:
            sample_bytes = 1 if bitdepth <= 8 else 2
        dt = torch.uint8 if sample_bytes == 1 else torch.int16

        def first_last(fr):
            if frame_data_type == "yuv420":
                return fr["y"], (fr["y"], fr["u"], fr["v"])
            return fr, (fr,)

        total, base, contiguous = 0, None, len(frames) > 0
        for fr in frames:
            head, parts = first_last(fr)
            for t in parts:
                if base is None:
                    base = t.data_ptr()
                contiguous = contiguous and t.is_contiguous() and t.dtype == torch.float32 and t.data_ptr() == base + 4 * total
                total += t.numel()
        if not contiguous:
            return torch.cat([self.pack_frame(fr, bitdepth, frame_data_type, False, sample_bytes) for fr in frames])
        out = torch.empty((total,), dtype=dt, device=self.torch_device)
        _check(self._lib.ccd_pack_samples(self._h, ctypes.c_void_p(base), total, int(bitdepth), sample_bytes, out.data_ptr(),
                                          self._stream()))
        return out

    def last_timing(self):
        ms = (ctypes.c_float * 4)()
        _check(self._lib.ccd_last_timing(self._h, ms))
        return {"entropy_ms": ms[0], "synthesis_ms": ms[1], "upload_ms": ms[2], "upload_bytes": int(ms[3])}

    def launch_count(self) -> int:
        return int(self._lib.ccd_debug_launch_count())

    def set_fused_synthesis(self, on: bool) -> None:
        """Debug switch: fused synthesis kernel (default) vs one kernel per layer; results are bit-identical."""
        _check(self._lib.ccd_debug_set_fused_synthesis(self._h, int(bool(on))))

    def last_status(self):
        st = (ctypes.c_int32 * 16)()
        _check(self._lib.ccd_debug_last_status(self._h, st))
        return list(st)

    def laplace_domain(self, sc_lo: int, sc_hi: int):
        n = (sc_hi - sc_lo) * 32641
        lo = np.zeros(n, dtype=np.uint32)
        hi = np.zeros(n, dtype=np.uint32)
        _check(self._lib.ccd_debug_laplace_domain(self._h, sc_lo, sc_hi, lo.ctypes.data_as(ctypes.c_void_p),
                                                  hi.ctypes.data_as(ctypes.c_void_p)))
        return lo, hi


def _frame_type_code(frame_data_type: str) -> int:
    """io/types.py:12 order: rgb, yuv420, yuv444, flow.  'flow' frames take the generic (4:4:4) tail like the
    reference's decode.py:191-206 does."""
    try:
        return {"rgb": 0, "yuv420": 1, "yuv444": 2, "flow": 3}[frame_data_type]
    except KeyError:
        raise ValueError(f"unknown frame_data_type {frame_data_type!r}") from None


_contexts = {}
_contexts_lock = threading.Lock()


def get_context(device: int = 0) -> Context:
    with _contexts_lock:
        if device not in _contexts:
            _contexts[device] = Context(device)
        return _contexts[device]
