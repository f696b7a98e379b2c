#!/usr/bin/env python
"""Benchmark of the decode hot path (BASELINE.json): decoded Mpixel/s (bit-exact).

    python bench.py --gpus N --steps K --warmup W [--workload NAME]      # this repository (B200)
    python bench.py ... --dump-outputs DIR                                # + the frames of the last timed step, as .npy
    python bench.py --impl reference --gpus N --steps K --warmup W        # CPU arm: the reference's own decode_video

Workloads (synthetic streams fabricated from the shipped sample, coolchic_b200.synth: the sample's latents TILED to
the target grids -- "kodim14 tiled" -- and range-encoded; networks re-shaped from the sample's):
  1080p_rgb_7grids      BASELINE configs[1]: one 1920x1080 RGB frame, 7 grids, HOP widths      (default for --gpus 1)
  4k_yuv420_8grids      configs[3]
  kodak_768x512_10grids configs[0]-shaped single frame
  kodak24_batch         configs[2]: 24 distinct 768x512 streams x 49 copies = 1176 frames, dealt to the ranks
                        (frame i -> rank i mod N), STRONG scaling                                 (default for --gpus > 1)
  gop32_1080p_yuv420    configs[4]: 32-frame hierarchical-B GOP, frame ownership per rank, exchange of reconstructed frames

A "step" = one pass of the hot path over the whole workload.  Printed JSON (one line, rank 0):
  value    : Mpixel/s from DEVICE time (CUDA events inside the library around the entropy and float-tail kernels; the
             bitstream upload is outside); for the video workload the wall clock of decode_video_bytes with frames left
             on the device;
  e2e      : the same metric through the public API with HOST buffers in and out: bitstream bytes in host memory (for
             N > 1 the NCCL broadcast of the bytes from rank 0 is inside the timed region) -> frames as packed integer
             samples (uint8) in pinned host memory;
  roofline : dominant kernel (k_entropy): algorithmic bytes / its CUDA-event duration against the measured HBM peak (tiny
             by construction: one serial dependency chain per stream), next to the figures that can bind it: ns / symbol,
             the serial floor measured on this box by tools/ubench/steps (tier-1 chain of the coder, one warp), and their
             ratio;  roofline_synthesis: the float tail against the HBM and the FP32 roofs;
  cpu_baseline: the reference's own decode_video on this box's host cores (oracle/_ref), the C port beside it.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "1080p_rgb_7grids": dict(kind="image", h=1080, w=1920, fmt="rgb", lat_res=(0, 6), hyp_res=None),
    "4k_yuv420_8grids": dict(kind="image", h=2160, w=3840, fmt="yuv420", lat_res=(0, 7), hyp_res=None),
    "kodak_768x512_10grids": dict(kind="image", h=512, w=768, fmt="rgb", lat_res=(0, 6), hyp_res=(4, 6)),
    "kodak24_batch": dict(kind="batch", h=512, w=768, fmt="rgb", lat_res=(0, 6), hyp_res=(4, 6), distinct=24, copies=49),
    "gop32_1080p_yuv420": dict(kind="video", h=1080, w=1920, fmt="yuv420", n_frames=32),
}
METRIC = "decoded Mpixel/s (bit-exact)"
UNIT = "Mpixel/s"
DUMP_LIMIT = 60 << 20  # bytes of samples written by --dump-outputs (the files stay under 64 MB with their headers)
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12  # CUDA-core FMA roof of a B200 at its maximum SM clock (74.5)


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.proc = None

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:  # noqa: BLE001
                self.proc.kill()

    def summary(self):
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        reasons = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for i, n in enumerate(names):
                if len(s) > 2 + i and s[2 + i].lower().startswith("active") and n not in reasons:
                    reasons.append(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def workload_pixels(wl):
    if wl["kind"] == "batch":
        return wl["h"] * wl["w"] * wl["distinct"] * wl["copies"]
    if wl["kind"] == "video":
        return wl["h"] * wl["w"] * wl["n_frames"]
    return wl["h"] * wl["w"]


def config_of(name, wl, world):
    cfg = {"workload": name, "height": wl["h"], "width": wl["w"], "frame_data_type": wl["fmt"], "bitdepth": 8,
           "latents": "kodim14 tiled (the shipped sample's decoded latents tiled to the target grids, range-encoded)",
           "l2_policy": "L2 flushed (256 MiB write) between timed iterations"}
    if wl["kind"] == "image":
        cfg.update(latent_resolution=list(wl["lat_res"]), hyperlatent_resolution=list(wl["hyp_res"]) if wl["hyp_res"] else None,
                   arm="14 ctx + 6 IFCE, 2 hidden", synthesis="48-1,3-1,3-3r,3-3r + stabiliser", frames_per_step=world,
                   parallelism=f"one frame per rank x{world} (a single stream cannot be split)", streams_per_gpu=1, sms_busy_entropy=1)
    elif wl["kind"] == "batch":
        n = wl["distinct"] * wl["copies"]
        cfg.update(latent_resolution=list(wl["lat_res"]), hyperlatent_resolution=list(wl["hyp_res"]),
                   arm="14 ctx + 6 IFCE, 2 hidden", synthesis="48-1,3-1,3-3r,3-3r + stabiliser", frames_per_step=n,
                   distinct_streams=wl["distinct"], parallelism=f"frame i -> rank i mod {world}",
                   streams_per_gpu=(n + world - 1) // world,
                   sms_busy_entropy="one SM per stream in flight: min(148, streams_per_gpu) per GPU")
    else:
        cfg.update(n_frames=wl["n_frames"], gop="I + P + hierarchical B, sinc-8 warps; intra hop, residue / motion mop",
                   frames_per_step=wl["n_frames"], coolchics=2 * wl["n_frames"] - 1,
                   parallelism=f"frame (coding order) i -> rank i mod {world}; reconstructed frames broadcast by their owner",
                   streams_per_gpu=(2 * wl["n_frames"] - 1 + world - 1) // world,
                   sms_busy_entropy="one SM per Cool-chic in flight",
                   floor="one I-frame stream is a single serial chain (~0.2 s at 1080p) whatever the number of GPUs")
    return cfg


# ----------------------------------------------------------------------------------------------------------------
def serial_floor(sm_mhz):
    """tools/ubench/steps on this box: cycles / symbol of the coder's tier-1 chain (one warp, 14 noise warps)."""
    exe = os.path.join(ROOT, "tools", "ubench", "steps")
    if not os.path.exists(exe):
        return None
    try:
        out = subprocess.run([exe, "floor"], capture_output=True, text=True, timeout=60).stdout
        m = re.search(r"mode only, lagged check\s+K=4 noise=14 :\s+([0-9.]+) cycles", out)
        if not m:
            return None
        cyc = float(m.group(1))
        return {"cycles_per_symbol": cyc, "ns_per_symbol": cyc / (sm_mhz or 1965.0) * 1e3,
                "what": "tools/ubench/steps: branch-free mode-only step of the range recursion, blocks of 4, one warp"}
    except Exception:  # noqa: BLE001
        return None


def run_reference_arm(args, name, wl, config):
    """CPU arm: the reference's own decode_video (oracle/_ref staged by oracle/make_ref.sh) on this box's host cores;
    inputs fabricated on the CPU by the oracle-backed writer.  Rank 0 only."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import reference_arm as ra

    if wl["kind"] == "image":
        sample_wl, n_px, what = dict(wl, seed=0), wl["h"] * wl["w"], "one full frame of the workload"
        n_rep = 1
    elif wl["kind"] == "batch":
        sample_wl, n_px, what = dict(wl, kind="image", seed=0), wl["h"] * wl["w"], "frames of the batch, decoded one after the other (the reference has no frame parallelism)"
        n_rep = 2
    else:
        sample_wl = dict(wl, n_frames=3, seed=0)
        n_px, what = 3 * wl["h"] * wl["w"], "a 3-frame GOP (I, P, B) of the workload's format"
        n_rep = 1
    data = ra.fabricate(sample_wl)
    ra.time_port(ra.fabricate(dict(kind="image", h=64, w=96, fmt="rgb", lat_res=(0, 4), hyp_res=None)), 64 * 96, 1)  # warm
    port = ra.time_port(data, n_px, os.cpu_count() or 1)
    steps = max(1, min(args.steps, n_rep if ra.reference_available() else 2))
    runs = []
    for _ in range(steps):
        runs.append(ra.time_reference(data, n_px) if ra.reference_available() else ra.time_port(data, n_px, os.cpu_count() or 1))
    best = max(runs, key=lambda r: r["value"])
    best["sample"] = what + "; " + best["sample"]
    line = {"impl": "reference", "metric": METRIC, "value": best["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": len(runs), "warmup": 0, "ms_per_step": best["seconds"] * 1e3, "higher_is_better": True,
            "scaling": "strong" if wl["kind"] != "image" else "weak", "vs_baseline": None,
            "dtype": "int64 entropy model + fp32 synthesis", "data": "synthetic", "config": config,
            "cpu_baseline": best, "cpu_baseline_port": port,
            "e2e": {"value": best["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the informational extra measurements (148 streams, batch workload at N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the frames the last timed step decoded (rank 0) to DIR/<name>.npy, "
                         f"float32, at most {DUMP_LIMIT >> 20} MiB (a seeded sample of whole frames when they are larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    name = args.workload or ("1080p_rgb_7grids" if world == 1 else "kodak24_batch")
    wl = WORKLOADS[name]
    n_pixels = workload_pixels(wl) * (world if wl["kind"] == "image" else 1)
    config = config_of(name, wl, world)

    if args.impl == "reference":
        if rank == 0:
            run_reference_arm(args, name, wl, config)
        return

    import torch

    import coolchic_b200  # noqa: F401
    from coolchic_b200 import _native, synth
    from coolchic_b200._desc import desc_from_header
    from coolchic_b200.bitstream.decode import decode_frame, decode_video_bytes
    from coolchic_b200.dist import broadcast_byte_strings

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = _native.get_context(local_rank)
    dev = ctx.torch_device
    warmup = max(3, args.warmup)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def split_cc(cc_bytes, header):
        h2 = type(header)()
        rest = h2.read_header(cc_bytes)
        n_nn, n_lat = h2.get_value("nn_n_bytes"), h2.get_value("n_bytes_latent")
        return desc_from_header(h2), rest[:n_nn], rest[n_nn:n_nn + n_lat]

    # ---- inputs: rank 0 fabricates the workload's streams (outside the timed region)
    streams = None  # list of complete single-frame bitstreams (image / batch), or [video bitstream]
    if rank == 0:
        ss = synth.SeedStream(ctx)
        if wl["kind"] == "image":
            streams = [synth.make_image_stream(ctx, ss, wl["h"], wl["w"], wl["fmt"], 8, wl["lat_res"], wl["hyp_res"], seed=0)]
        elif wl["kind"] == "batch":
            distinct = [synth.make_image_stream(ctx, ss, wl["h"], wl["w"], wl["fmt"], 8, wl["lat_res"], wl["hyp_res"], seed=i)
                        for i in range(wl["distinct"])]
            streams = [distinct[i % wl["distinct"]] for i in range(wl["distinct"] * wl["copies"])]
        else:
            streams = [synth.make_video_stream(ctx, ss, wl["h"], wl["w"], wl["n_frames"], wl["fmt"], 8, 8, seed=0)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    n_sym_total = [0]
    alg_bytes = [0]

    def parse_image(data):
        _, f, c, nn_bytes, payload = synth.parse_single_image(data)
        return desc_from_header(c), nn_bytes, payload

    # ---- the step of each kind.  Returns (device_ms or None, h2d_bytes, d2h_bytes) of this rank
    pinned = {}

    def pinned_buf(n):
        if pinned.get("n", 0) < n:
            pinned["t"] = torch.empty((n,), dtype=torch.uint8).pin_memory()
            pinned["n"] = n
        return pinned["t"]

    def pack_to_host(frames_data, fmt):
        """finished frames on the device -> packed uint8 samples in pinned host memory (the frames of one decode_many
        call are slices of one buffer: one packing launch and one copy for the whole batch)"""
        packed = ctx.pack_frames(frames_data, 8, fmt)
        n = int(packed.numel())
        pinned_buf(n)[:n].copy_(packed, non_blocking=True)
        torch.cuda.synchronize()
        return n

    if wl["kind"] == "image":
        data0 = broadcast_byte_strings(streams, src=0, device=dev)[0] if world > 1 else streams[0]
        desc, nn_bytes, payload = parse_image(data0)
        n_sym_total[0] = desc.n_symbols()
        alg_bytes[0] = len(payload) + len(nn_bytes) + desc.n_symbols()
        frame_bytes = data0[8:]  # after the video header (1 intra frame)

        def device_step():
            outs, _ = ctx.decode_many([desc], [nn_bytes], [payload], finish=[(8, wl["fmt"])])
            t = ctx.last_timing()
            return t["entropy_ms"], t["synthesis_ms"], [("frame", outs[0])]

        def e2e_step():
            frame, _ = decode_frame(frame_bytes, reference_frames=[], device=local_rank)
            h2d = ctx.last_timing()["upload_bytes"]
            return h2d, pack_to_host([frame.data], wl["fmt"])
    elif wl["kind"] == "batch":
        resident = broadcast_byte_strings(streams, src=0, device=dev) if world > 1 else streams
        mine = list(range(rank, len(resident), world))
        def my_jobs(all_streams):
            # (header parsing of this rank's share is part of the end-to-end path)
            return [parse_image(all_streams[i]) for i in mine]

        jobs0 = my_jobs(resident)
        n_sym_total[0] = sum(j[0].n_symbols() for j in jobs0)
        alg_bytes[0] = sum(len(j[1]) + len(j[2]) + j[0].n_symbols() for j in jobs0)

        def device_step():
            outs, _ = ctx.decode_many([j[0] for j in jobs0], [j[1] for j in jobs0], [j[2] for j in jobs0], finish=[(8, wl["fmt"])] * len(jobs0))
            t = ctx.last_timing()
            return t["entropy_ms"], t["synthesis_ms"], [(f"frame{i:04d}", o) for i, o in zip(mine, outs)]

        def e2e_step():
            got = broadcast_byte_strings(streams, src=0, device=dev, want=mine) if world > 1 else streams
            jobs = my_jobs(got)
            outs, _ = ctx.decode_many([j[0] for j in jobs], [j[1] for j in jobs], [j[2] for j in jobs], finish=[(8, wl["fmt"])] * len(jobs))
            h2d = ctx.last_timing()["upload_bytes"]
            return h2d, pack_to_host(outs, wl["fmt"])
    else:
        import contextlib
        import io

        data0 = broadcast_byte_strings(streams, src=0, device=dev)[0] if world > 1 else streams[0]

        def decode_gop(data):
            with contextlib.redirect_stdout(io.StringIO()):  # (one timing line per frame, like the reference)
                return decode_video_bytes(data, device=local_rank, output_device="cuda")

        def device_step():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            frames = decode_gop(data0)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3
            return ms, 0.0, [(f"frame{int(k):02d}", frames[k].data) for k in sorted(frames, key=int)]

        def e2e_step():
            data = broadcast_byte_strings(streams, src=0, device=dev)[0] if world > 1 else streams[0]
            frames = decode_gop(data)
            own = [frames[k].data for k in sorted(frames, key=int) if int(k) % world == rank]
            return len(data), pack_to_host(own, wl["fmt"])

    for _ in range(warmup):
        device_step()
        e2e_step()

    # ---- timed region 1: K steps, device time; L2 flushed between steps
    ent_ms, syn_ms = [], []
    launches0 = ctx.launch_count()
    with ClockSampler(local_rank) as clocks:
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(args.steps):
            flush.zero_()
            outputs = None  # release the previous step's frames before this step allocates its own
            a, b, outputs = device_step()
            ent_ms.append(a)
            syn_ms.append(b)
        ev1.record()
        barrier()
        launches = (ctx.launch_count() - launches0) // max(1, args.steps)
        total_ms = ev0.elapsed_time(ev1)
        dev_ms = (sum(ent_ms) + sum(syn_ms)) / args.steps
        # ---- timed region 2: K end-to-end steps (host bytes in, packed samples in pinned host memory out)
        h2d = d2h = 0
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            flush.zero_()
            h2d, d2h = e2e_step()
        barrier()
        e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)
    stats = torch.tensor([dev_ms, total_ms / args.steps, e2e_ms, sum(ent_ms) / args.steps], dtype=torch.float64, device=dev)
    sums = torch.tensor([float(h2d), float(d2h), float(n_sym_total[0]), float(alg_bytes[0])], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    dev_ms, step_ms, e2e_ms, ent_avg = [float(x) for x in stats.tolist()]
    h2d_all, d2h_all, n_sym_all, alg_all = [float(x) for x in sums.tolist()]

    if rank == 0:
        peak, peak_kind = hbm_peak()
        clk = clocks.summary()
        line = {"metric": METRIC, "value": n_pixels / dev_ms / 1e3, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": warmup, "ms_per_step": step_ms, "higher_is_better": True,
                "scaling": "weak" if wl["kind"] == "image" else "strong", "vs_baseline": None,
                "dtype": "int64 entropy model + fp32 synthesis", "data": "synthetic", "config": config,
                "device_ms_per_step": dev_ms,
                "e2e": {"value": n_pixels / e2e_ms / 1e3, "unit": UNIT, "ms_per_step": e2e_ms,
                        "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all),
                        "output": "packed uint8 samples in pinned host memory (device-side packing)"},
                "gpu_launches": int(launches), "clocks": clk}
        if wl["kind"] != "video":
            ent_s = ent_avg / 1e3
            per_gpu_sym = n_sym_all / world
            # one persistent CTA per stream: the serial chain of ONE stream bounds the launch (streams run concurrently)
            chain_sym = per_gpu_sym if wl["kind"] == "image" else desc_from_header(synth.parse_single_image(streams[0])[2]).n_symbols() * \
                max(1, -(-config["streams_per_gpu"] // 148))
            roof = {"bound": "hbm", "kernel": "k_entropy (wavefront ARM + range decoder, one persistent CTA per stream)",
                    "achieved": alg_all / world / ent_s / 1e9, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                    "frac": alg_all / world / ent_s / 1e9 / peak,
                    # DRAM bytes per launch from the committed ncu --set full capture of the default command
                    # (profiles/r02_*): quoted for the default workload only
                    "traffic": None,
                    "algorithmic_bytes_per_launch": int(alg_all / world), "kernel_ms": ent_avg, "share_of_step": ent_avg / dev_ms,
                    "ns_per_symbol": ent_avg * 1e6 / chain_sym, "symbols_on_the_serial_chain": int(chain_sym),
                    "note": "serial-latency-bound kernel (one range-coded stream = one dependency chain; the streams of a "
                            "batch run concurrently, one SM each): HBM is not the limiting resource, see DESIGN.md"}
            prof = os.path.join(ROOT, "profiles", "r02_traffic.json")
            if name == "1080p_rgb_7grids" and os.path.exists(prof):
                try:
                    roof["traffic"] = json.load(open(prof)).get("k_entropy_dram_bytes_per_launch")
                except Exception:  # noqa: BLE001
                    pass
            fl = serial_floor(clk.get("sm_mhz"))
            if fl and wl["kind"] == "image":
                roof["serial_floor_ns_per_symbol"] = fl["ns_per_symbol"]
                roof["serial_floor"] = fl
                roof["frac_of_serial_floor"] = fl["ns_per_symbol"] / roof["ns_per_symbol"]
            line["roofline"] = roof
            syn_avg = max(dev_ms - ent_avg, 1e-6)
            px_gpu = n_pixels / world
            px_bytes = per_gpu_sym + (12 if wl["fmt"] != "yuv420" else 6) * px_gpu
            flops = 1724.0 * px_gpu  # 2 x (672 synthesis + 190 upsampling MAC) per pixel at HOP widths (SURVEY 8d)
            line["roofline_synthesis"] = {
                "bound": "fp32", "kernel": "cascade levels + k_tail_syn (last level + synthesis + frame tail, TMA tile staging)",
                "kernel_ms": syn_avg, "algorithmic_bytes": int(px_bytes),
                "achieved_gbs": px_bytes / (syn_avg / 1e3) / 1e9, "hbm_frac": px_bytes / (syn_avg / 1e3) / 1e9 / peak,
                "achieved_tflops": flops / (syn_avg / 1e3) / 1e12, "fp32_peak_tflops": FP32_PEAK_TFLOPS,
                "fp32_frac": flops / (syn_avg / 1e3) / 1e12 / FP32_PEAK_TFLOPS}
        if not args.no_extras and world == 1 and name == "1080p_rgb_7grids":
            # informational extras, outside the timed region; they must never cost the headline line
            try:
                line["many_streams"] = many_streams(ctx, synth, parse_image)
            except Exception as e:  # noqa: BLE001
                line["many_streams"] = {"error": str(e)[:200]}
            try:
                # the N = 1 point of the workload the multi-GPU runs use by default (strong scaling: same 1176 frames)
                bw = WORKLOADS["kodak24_batch"]
                line["scale_workload_at_n1"] = many_streams(ctx, synth, parse_image, n=bw["distinct"] * bw["copies"], distinct=bw["distinct"],
                                                            label="kodak24_batch", reps=2)
            except Exception as e:  # noqa: BLE001
                line["scale_workload_at_n1"] = {"error": str(e)[:200]}
        if not args.no_cpu_baseline and world == 1:
            try:
                sys.path.insert(0, os.path.join(ROOT, "oracle"))
                import reference_arm as ra

                sample = streams[0]
                px = wl["h"] * wl["w"] * (wl.get("n_frames", 1) if wl["kind"] == "video" else 1)
                if wl["kind"] == "video":  # bounded sample: a 3-frame GOP
                    sample = ra.fabricate(dict(wl, n_frames=3, seed=0))
                    px = 3 * wl["h"] * wl["w"]
                ra.time_port(ra.fabricate(dict(kind="image", h=64, w=96, fmt="rgb", lat_res=(0, 4), hyp_res=None)), 64 * 96, 1)
                line["cpu_baseline_port"] = ra.time_port(sample, px, os.cpu_count() or 1)
                line["cpu_baseline"] = ra.time_reference(sample, px) if ra.reference_available() else line["cpu_baseline_port"]
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"error": str(e)[:200], "kind": "reference", "cores": 0}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(dirname, frames):
    """Write the decoded frames, as returned to the caller, to ``dirname/<name>.npy`` (float32; a yuv420 frame is three
    files <name>_y / _u / _v).  When all of them exceed DUMP_LIMIT bytes, a fixed seeded sample of whole frames is written,
    so that two builds run with the same arguments can be compared file by file."""
    import numpy as np

    units = []
    for name, data in frames:
        planes = [(f"{name}_{c}", data[c]) for c in ("y", "u", "v")] if isinstance(data, dict) else [(name, data)]
        units.append((planes, sum(4 * t.numel() for _, t in planes)))
    keep = list(range(len(units)))
    if sum(n for _, n in units) > DUMP_LIMIT:
        keep, total = [], 0
        for i in np.random.default_rng(0).permutation(len(units)):
            if total + units[i][1] <= DUMP_LIMIT:
                keep.append(int(i))
                total += units[i][1]
        keep.sort()
    os.makedirs(dirname, exist_ok=True)
    for i in keep:
        for name, t in units[i][0]:
            np.save(os.path.join(dirname, name + ".npy"), t.detach().float().cpu().numpy())


def many_streams(ctx, synth, parse_image, n=148, distinct=24, label=None, reps=3):
    """Informational: BASELINE configs[2] on ONE GPU in one call -- 148 Kodak-size frames decoded concurrently (one
    persistent CTA, i.e. one SM, per stream; batched float tail).  Outputs verified by
    tests/test_gpu_decode.py::test_148_streams_every_output_checked."""
    import torch

    ss = synth.SeedStream(ctx)
    items = [parse_image(synth.make_image_stream(ctx, ss, 512, 768, "rgb", 8, (0, 6), (4, 6), seed=i)) for i in range(distinct)]
    sub = (items * ((n + distinct - 1) // distinct))[:n]
    best = None
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ctx.decode_many([x[0] for x in sub], [x[1] for x in sub], [x[2] for x in sub], finish=[(8, "rgb")] * n)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    tm = ctx.last_timing()
    out = {"workload": f"{n} x 768x512 RGB, 7 grids + 3 hyperlatent grids ({distinct} distinct streams), one ccd_decode_many call",
           "streams": n, "ms": best * 1e3, "entropy_ms": tm["entropy_ms"], "synthesis_ms": tm["synthesis_ms"],
           "value": n * 512 * 768 / best / 1e6, "unit": UNIT,
           "device_value": n * 512 * 768 / (tm["entropy_ms"] + tm["synthesis_ms"]) / 1e3,
           "includes": "host staging + H2D of the bitstreams, finished fp32 frames left on the device; device_value = from the "
                       "library's CUDA events only (what `value` of the kodak24_batch workload reports)"}
    if label:
        out["name"] = label
    return out


if __name__ == "__main__":
    main()
