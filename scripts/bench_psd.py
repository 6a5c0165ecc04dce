"""Averaged power spectra (sdr_psd) throughput on one GPU: one JSON line per config.

For each config: check spot spectra of a fresh handle's first call against the f64 reference (so a fast wrong answer
cannot be reported), then time >= 20 back-to-back process_dev calls on device-resident data with CUDA events,
ALTERNATING with the composition users have without sdr_psd: for H = N, FftPlan(N, fmt, shift, norm).exec_dev into a
c64 buffer, then torch real^2 + imag^2 and .view(G, K, N).mean(1); for overlapped frames WindowFft instead of FftPlan
(WindowFft has no taper, so the composition skips the Hann multiply, which favours it).  Three rounds of each; the best
round of each is reported.  The per-kernel split of one call comes from torch.profiler in a separate run.

Bytes per input sample are algorithmic: 2 (u8 IQ) or 8 (c64) in, plus the chunk partials (4 N bytes per chunk of up to
32 frames, written and read back, when a group spans several chunks) and the output rows.  "frac_hbm" is that traffic
over the call time against 6552.3 GB/s, the HBM rate the rest of the project quotes as measured peak.  "frac_issue"
(fused path) is the transforms per second against the instruction-issue bound of DESIGN K8: about 1400 warp
instructions per 1024-point transform, 4 issued per cycle per SM, 148 SMs at the card's maximum SM clock.
"composed.intermediate_bytes" is the composition's c64 spectra plus their f32 powers, the memory it needs beyond its
input and output.

    python scripts/bench_psd.py [--calls 20] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "unnamed-rust-sdr_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

PEAK_GBS = 6552.3
INSTR_PER_1K = 1400  # warp instructions per fused 1024-point transform (DESIGN K8)
SMS = 148
S = 32


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        name, power, clk = [s.strip() for s in out.strip().split(",")[:3]]
        return name, power + " W", float(clk) * 1e6
    except Exception as e:  # the numbers still stand; say the card could not be read
        return "unknown (%s)" % e, "unknown", float("nan")


def make_input(torch, dev, fmt, n, seed):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    if fmt == "u8iq":
        return torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    return torch.complex(torch.rand(n, device=dev, generator=g) * 2 - 1, torch.rand(n, device=dev, generator=g) * 2 - 1)


def spot_check(d_in, d_out, fmt, N, H, K, w, G):
    import oracle_lib as O
    import psd_ref as R
    worst = 0.0
    for g in sorted({0, G // 2, G - 1}):
        lo = (g * K + 1) * H - N  # first sample of the group's first frame (< 0: the stream's initial zeros)
        s0, s1 = max(0, lo), (g + 1) * K * H
        raw = d_in[2 * s0:2 * s1] if fmt == "u8iq" else d_in[s0:s1]
        x = O.unpack_u8iq(raw.cpu().numpy()) if fmt == "u8iq" else raw.cpu().numpy()
        x = np.concatenate([np.zeros(s0 - lo, np.complex128), x.astype(np.complex128)])  # x[0] is sample lo
        fr = np.stack([x[r * H:r * H + N] for r in range(K)])
        P = (np.abs(np.fft.fft(fr * (1.0 if w is None else w), axis=1)) ** 2).mean(axis=0) / N
        want = np.roll(P, N // 2)
        got = d_out[g].cpu().numpy().astype(np.float64)
        worst = max(worst, float(np.abs(got - want).max() / want.max()))
    if not worst <= R.bar(N):
        raise SystemExit("spot spectra differ from f64 truth: %.3g of max P > %.3g" % (worst, R.bar(N)))
    return worst


def events_ms(torch, st, fn, calls):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(calls):
        fn()
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b) / calls


def kernel_split(torch, fn):
    """device time (ms) per kernel / copy name of one call, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    split = {}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        name = e.name
        for key in ("psd1024_kernel", "psd_reduce_kernel", "psd_gather_kernel", "psd_accum_kernel",
                    "fft1024_warp_kernel", "window_gather", "fft_", "bluestein", "Memcpy", "reduce", "mean", "mul",
                    "pow", "abs"):
            if key.lower() in name.lower():
                name = key
                break
        else:
            name = name[:40]
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        split[name] = split.get(name, 0.0) + us / 1000.0
    return {k: round(v, 4) for k, v in split.items()}


def bench_config(sdr, torch, dev, fmt, n, N, H, K, hann, general, calls, name, power, clk):
    st = torch.cuda.current_stream(dev)
    d_in = make_input(torch, dev, fmt, n, 1234 + N + H + K)
    G = (n // H) // K
    F = G * K
    d_out = torch.empty((G, N), dtype=torch.float32, device=dev)
    w = np.hanning(N).astype(np.float32) if hann else None
    psd = sdr.Psd(N, H, K, window=w, fmt=fmt, shift=True, norm=True, general=general, stream=st)

    def call():
        psd.reset()
        return psd.process_dev(d_in, n, d_out, G)
    assert call() == G
    torch.cuda.synchronize()
    err = spot_check(d_in, d_out, fmt, N, H, K, None if w is None else w.astype(np.float64), G)
    path = psd.last_path

    # the composition
    c_spec = torch.empty((F, N), dtype=torch.complex64, device=dev)
    if H == N:
        plan = sdr.FftPlan(N, fmt, shift=True, norm=True, stream=st)
        transform = lambda: plan.exec_dev(d_in, F, c_spec)  # noqa: E731
        what = "FftPlan(%d).exec_dev + torch |.|^2 + mean over K" % N
    else:
        wf = sdr.WindowFft(N, H, fmt, shift=True, norm=True, stream=st)

        def transform():
            wf.reset()
            wf.process_dev(d_in, n, c_spec, F)
        what = "WindowFft(%d, %d).process_dev (no taper) + torch |.|^2 + mean over K" % (N, H)
    c_out = torch.empty((G, N), dtype=torch.float32, device=dev)

    def composed():
        transform()
        r = torch.view_as_real(c_spec)
        torch.mean((r[..., 0] * r[..., 0] + r[..., 1] * r[..., 1]).view(G, K, N), dim=1, out=c_out)
    composed()
    torch.cuda.synchronize()
    diff = float((c_out - d_out).abs().max() / d_out.abs().max())

    ms_r, cms_r = [], []
    for _ in range(3):
        ms_r.append(events_ms(torch, st, call, calls))
        cms_r.append(events_ms(torch, st, composed, calls))
    ms, cms = min(ms_r), min(cms_r)
    split = kernel_split(torch, call)
    comp_split = kernel_split(torch, composed)
    es = 2 if fmt == "u8iq" else 8
    cpg = -(-K // S)
    chunks = G * cpg
    part_bytes = 2 * 4 * N * chunks if cpg > 1 else 0
    bps = es + (part_bytes + 4 * N * G) / n
    gs = n / (ms * 1e-3) / 1e9
    rec = {"bench": "psd", "fmt": fmt, "n_samples": n, "N": N, "H": H, "K": K, "taper": "hann" if hann else "rect",
           "path": path, "calls": calls, "ms_per_call": round(ms, 4), "ms_rounds": [round(v, 4) for v in ms_r],
           "gsamples_per_s": round(gs, 2), "bytes_per_sample": round(bps, 4), "gb_per_s": round(gs * bps, 1),
           "frac_hbm": round(gs * bps / PEAK_GBS, 4), "kernels_ms": split, "spot_err_rel": err}
    if path == 2:
        transforms_per_s = F / (ms * 1e-3)
        bound = SMS * 4 * clk / INSTR_PER_1K
        rec["issue"] = {"instr_per_transform": INSTR_PER_1K, "sm_clock_max_mhz": clk / 1e6,
                        "bound_transforms_per_s": round(bound, 1), "frac_issue": round(transforms_per_s / bound, 4),
                        "bound_gsamples_per_s": round(bound * H / 1e9, 1)}
    rec["composed"] = {"what": what, "ms_per_call": round(cms, 4), "ms_rounds": [round(v, 4) for v in cms_r],
                       "gsamples_per_s": round(n / (cms * 1e-3) / 1e9, 2), "kernels_ms": comp_split,
                       "intermediate_bytes": F * N * (8 + 4), "max_diff_vs_psd_rel": diff}
    rec["speedup_vs_composed"] = round(cms / ms, 2)
    rec["gpu"], rec["power_limit"] = name, power
    psd.close()
    del d_in, d_out, c_out, c_spec
    torch.cuda.empty_cache()
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--quick", action="store_true", help="2^22 samples per config (a rehearsal, not a measurement)")
    args = ap.parse_args()
    import torch
    import sdr_b200 as sdr
    if not torch.cuda.is_available() or sdr.device_count() < 1:
        raise SystemExit("bench_psd: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    big = 1 << 22 if args.quick else 1 << 28
    mid = 1 << 22 if args.quick else 1 << 26
    # (fmt, n, N, H, K, hann, general)
    configs = [("u8iq", big, 1024, 1024, 256, False, False), ("u8iq", big, 1024, 1024, 1, False, False),
               ("u8iq", big, 1024, 512, 512, True, False), ("c64", mid, 1024, 1024, 256, False, False),
               ("u8iq", big, 1000, 1000, 256, False, False), ("u8iq", big, 4096, 4096, 64, False, False)]
    for fmt, n, N, H, K, hann, general in configs:
        bench_config(sdr, torch, dev, fmt, n, N, H, K, hann, general, max(20, args.calls), name, power, clk)


if __name__ == "__main__":
    main()
