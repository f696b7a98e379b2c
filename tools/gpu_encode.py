"""Measurement of the data-parallel encoder (ccd_encode_many) against the wavefront encoder (ccd_encode_latents
mode 1) and the oracle's CPU encoder, on the same inputs, in one process.

    python tools/gpu_encode.py [--reps 3] [--out DIR] [--only NAME,...] [--mode1-batch]

Workloads: 1080p 7-grid RGB, 4K 8-grid, 148 Kodak-size streams in one call, kodak24_batch (1176 streams: latents,
intervals and payload words of the batch exceed the 126 MB L2).  Per workload: device time (CUDA events in the
library: ARM pass + range coder) and end-to-end time (host list of int8 latents -> payload bytes in host memory),
both paths alternated rep by rep, payloads compared byte for byte; then, in a separate profiled pass, the kernel times
of k_enc_arm and k_enc_range (torch.profiler), the coder's ns / symbol next to tools/ubench/steps' serial floor, and
the ARM pass in symbols/s and integer MAC/s counted from the architecture.  Needs a GPU: no CPU fallback.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import coolchic_b200  # noqa: E402,F401
from coolchic_b200 import _native, synth  # noqa: E402
from coolchic_b200._desc import desc_from_header  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # noqa: BLE001
        info["power_limit"] = f"not read ({e})"
    return info


def serial_floor():
    """Cycles / symbol of the decoder's mode-only range step (tools/ubench/steps, built by build()); None if absent."""
    exe = os.path.join(ROOT, "tools", "ubench", "steps")
    if not os.path.exists(exe):
        return None
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120).stdout
    m = re.search(r"mode only, lagged check\s+K=4 noise=14 :\s+([0-9.]+) cycles", out)
    return float(m.group(1)) if m else None


def stream(ctx, ss, hw, lr, hr, seed):
    cc, h, lat = synth.make_coolchic(ctx, ss, hw, lr, hr, seed=seed)
    h2 = type(h)()
    rest = h2.read_header(cc)
    n_nn, n_lat = h2.get_value("nn_n_bytes"), h2.get_value("n_bytes_latent")
    return desc_from_header(h2), rest[:n_nn], rest[n_nn:n_nn + n_lat], lat


def arm_macs(d):
    """Integer multiply-accumulates of the ARM (+ IFCE) per Cool-chic, counted from the architecture."""
    dim = d.n_ctx + d.n_ifce_out
    per = d.arm_hidden * dim * dim + 2 * dim + (2 * dim if d.arm_stab else 0)
    total = 0
    for g in range(d.n_grids):
        n = d.grid_h[g] * d.grid_w[g]
        ifce = d.n_ifce_out * d.grid_ifce_in[g] if d.flag_ifce else 0
        total += n * (per + ifce)
    return total


NAMES = ["1080p_rgb_7grids", "4k_8grids", "kodak_148", "kodak24_batch"]


def workloads(ctx, ss, names=NAMES):
    W = {}
    k24 = [stream(ctx, ss, (512, 768), (0, 6), (4, 6), seed=i) for i in range(24)] if any("kodak" in n for n in names) else []
    for n in names:
        if n == "1080p_rgb_7grids":
            W[n] = [stream(ctx, ss, (1080, 1920), (0, 6), None, seed=1)]
        elif n == "4k_8grids":
            W[n] = [stream(ctx, ss, (2160, 3840), (0, 7), None, seed=1)]
        else:
            W[n] = [k24[i % 24] for i in range(148 if n == "kodak_148" else 24 * 49)]
    return W


def run_new(ctx, items, host_lat):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pays, _ = ctx.encode_many([x[0] for x in items], [x[1] for x in items], host_lat, synthesize=False)
    t1 = time.perf_counter()  # encode_many returns host bytes: the device work is complete
    return pays, ctx.last_timing()["entropy_ms"], (t1 - t0) * 1e3


def run_mode1(ctx, items, nn_ints):
    torch.cuda.synchronize()
    dev_ms, pays = 0.0, []
    t0 = time.perf_counter()
    for i, ((d, _, _, lat), nn) in enumerate(zip(items, nn_ints)):
        _, p, _ = ctx.encode_latents(d, nn, latents=lat)
        dev_ms += ctx.last_timing()["entropy_ms"]
        pays.append(p)
        if i % 200 == 199:
            print(f"  mode 1: {i + 1} / {len(items)} streams", flush=True)
    torch.cuda.synchronize()
    return pays, dev_ms, (time.perf_counter() - t0) * 1e3


def profile_one(ctx, items, out_dir, name):
    """Kernel times of one encode_many call under torch.profiler (run in a process of its own per workload)."""
    from torch.profiler import ProfilerActivity, profile as tprof

    args = ([x[0] for x in items], [x[1] for x in items], [x[3] for x in items])
    ctx.encode_many(*args, synthesize=False)
    torch.cuda.synchronize()
    with tprof(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.encode_many(*args, synthesize=False)
        torch.cuda.synchronize()
    path = os.path.join(out_dir or ".", f"encode_{name}.pt.trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        ev = [e for e in json.load(f)["traceEvents"] if e.get("cat") == "kernel"]
    if not out_dir:
        os.remove(path)
    arm = sum(e["dur"] for e in ev if "k_enc_arm" in e["name"]) / 1e3
    rng = sum(e["dur"] for e in ev if "k_enc_range" in e["name"]) / 1e3
    n_sym = sum(x[0].n_symbols() for x in items)
    macs = sum(arm_macs(x[0]) for x in items)
    return {"k_enc_arm_ms": round(arm, 3) if arm else "not captured", "k_enc_range_ms": round(rng, 3) if rng else "not captured",
            "coder_ns_per_symbol": round(rng * 1e6 / max(x[0].n_symbols() for x in items), 3) if rng else None,
            "arm_gsymbols_per_s": round(n_sym / (arm * 1e-3) / 1e9, 3) if arm else None,
            "arm_int_tmac_per_s": round(macs / (arm * 1e-3) / 1e12, 3) if arm else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None, help=argparse.SUPPRESS)  # one workload under torch.profiler
    ap.add_argument("--only", default=",".join(NAMES), help="comma-separated workloads")
    ap.add_argument("--mode1-batch", action="store_true",
                    help="also run mode 1 (once) on kodak24_batch: one stream after the other, ~6 min")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_encode.py needs a CUDA device: there is no CPU fallback")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
    ctx = _native.get_context(0)
    ss = synth.SeedStream(ctx)
    if args.profile:
        print(json.dumps(profile_one(ctx, workloads(ctx, ss, [args.profile])[args.profile], args.out, args.profile)))
        return
    res = {"card": card()}
    print("card:", res["card"], flush=True)
    sm_mhz = float(re.sub(r"[^0-9.]", "", res["card"].get("max_sm_clock", "1965")) or 1965)
    floor_cyc = serial_floor()
    res["serial_floor"] = {"cycles_per_symbol": floor_cyc,
                           "ns_per_symbol": floor_cyc / sm_mhz * 1e3 if floor_cyc else None,
                           "what": "tools/ubench/steps: mode-only step of the decoder's range recursion, one warp"}
    print("serial floor:", res["serial_floor"], flush=True)
    W = workloads(ctx, ss, args.only.split(","))
    res["workloads"] = {}
    for name, items in W.items():
        n_sym = sum(x[0].n_symbols() for x in items)
        host_lat = [x[3].cpu().numpy() for x in items]
        nn_ints = [_native.decode_nn(x[0], x[1]) for x in items]
        run_new(ctx, items[:2], host_lat[:2])  # warm-up: module load, allocations
        new, old = [], []
        same = True
        for r in range(args.reps):
            pays, dev, e2e = run_new(ctx, items, host_lat)
            new.append((dev, e2e))
            same = same and all(p == x[2] for p, x in zip(pays, items))
            if name == "kodak24_batch":
                run1 = args.mode1_batch and r == 0
            else:
                run1 = r < 2 or len(items) == 1
            if run1:
                p1, dev1, e2e1 = run_mode1(ctx, items, nn_ints)
                old.append((dev1, e2e1))
                same = same and p1 == pays
        w = {
            "streams": len(items), "symbols": n_sym, "payload_bytes": sum(len(x[2]) for x in items),
            "payloads_identical_new_mode1_fabricated": same,
            "new_device_ms": [round(a, 3) for a, _ in new], "new_e2e_ms": [round(b, 3) for _, b in new],
            "mode1_device_ms": [round(a, 3) for a, _ in old] or "not measured",
            "mode1_e2e_ms": [round(b, 3) for _, b in old] or "not measured",
        }
        if old:
            w["speedup_device"] = round(min(a for a, _ in old) / min(a for a, _ in new), 2)
            w["speedup_e2e"] = round(min(b for _, b in old) / min(b for _, b in new), 2)
        res["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
    # kernel times: torch.profiler, one process per workload (a later profiling session in the same process lost
    # kernel records)
    for name in W:
        cmd = [sys.executable, "-W", "ignore", os.path.abspath(__file__), "--profile", name] + (["--out", args.out] if args.out else [])
        r = subprocess.run(cmd, capture_output=True, text=True)
        k = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": r.stderr[-500:]}
        res["workloads"][name].update(k)
        print(name, "kernels", json.dumps(k), flush=True)
    # the oracle's CPU encoder (all host threads it uses), one 1080p and one Kodak stream
    import ccoracle

    ccoracle.build()
    cpu = {}
    for name, key in (("1080p_rgb_7grids", "1080p_rgb_7grids"), ("kodak_1_stream", "kodak_148")):
        if key not in W:
            continue
        d, nnb, pay, lat = W[key][0]
        nn = ccoracle.decode_nn(d, nnb)
        ln = lat.cpu().numpy()
        t0 = time.perf_counter()
        p = ccoracle.encode_latents(d, nn, ln)
        cpu[name] = {"ms": round((time.perf_counter() - t0) * 1e3, 3), "identical": p == pay}
    res["oracle_cpu_encoder"] = cpu
    print("oracle cpu:", cpu, flush=True)
    if args.out:
        tag = "" if args.only == ",".join(NAMES) else "_" + args.only.replace(",", "_")
        with open(os.path.join(args.out, f"encode{tag}.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
