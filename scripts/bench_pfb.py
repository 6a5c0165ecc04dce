"""Polyphase filter bank (sdr_pfb) throughput on one GPU: one JSON line per config.

For each config: warm up, check spot frames of a fresh handle's first call against the f64 polyphase form (so a fast
wrong answer cannot be reported), time >= 20 back-to-back process_dev calls on device-resident data with CUDA events,
then split one call into stages (front end / FFT / transpose / copies) with torch.profiler in a separate run.
Bytes per input sample are algorithmic: 2 (u8 IQ) or 8 (c64) in, plus 8 M / D out.  "frac_peak" is that traffic over
the call time against 6552.3 GB/s, the HBM rate the rest of the project quotes as measured peak.

The composed alternative users have without the bank -- one Fir(g_k) with Decimate(D) per channel -- is timed for one
channel on a shorter input and reported times M (and scaled to the bank's input length): an extrapolation, labelled so.

    python scripts/bench_pfb.py [--calls 20] [--quick]
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


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception as e:  # the numbers still stand; say the card could not be read
        return "unknown (%s)" % e, "unknown"


def make_input(torch, dev, fmt, n, seed):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    if fmt == "u8iq":
        return torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    return torch.complex(torch.rand(n, device=dev, generator=g) * 2 - 1, torch.rand(n, device=dev, generator=g) * 2 - 1)


def host_samples(d_in, fmt, lo, hi):
    """c64 values of stream samples [lo, hi) of the device input"""
    import oracle_lib as O
    if fmt == "u8iq":
        return O.unpack_u8iq(d_in[2 * lo:2 * hi].cpu().numpy())
    return d_in[lo:hi].cpu().numpy()


def spot_check(d_in, d_out, fmt, h, M, D, cmajor, nf):
    import pfb_ref as R
    L = h.size
    worst = 0.0
    for j in (0, nf // 2, nf - 1):
        s0 = max(0, ((j + 1) * D - L) // D * D)
        x = host_samples(d_in, fmt, s0, (j + 1) * D)
        want = R.polyphase_f64(h, x, M, D, frames=[j - s0 // D])[0]
        got = (d_out[:, j] if cmajor else d_out[j]).cpu().numpy()
        worst = max(worst, float(np.abs(got - want).max() / np.abs(want).max()))
    bar = 1e-5 * np.log2(M)
    if not worst <= bar:
        raise SystemExit("spot frames differ from f64 truth: %.3g of max|y| > %.3g" % (worst, bar))
    return worst


def stage_times(torch, fn):
    """per-stage device time (ms) of one call, from torch.profiler kernel / copy records"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    stages = {"front_end": 0.0, "fft": 0.0, "transpose": 0.0, "copy": 0.0, "other": 0.0}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        name = e.name.lower()
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        if "pfb_front" in name:
            key = "front_end"
        elif "pfb_transpose" in name:
            key = "transpose"
        elif "memcpy" in name:
            key = "copy"
        elif "fft" in name or "bluestein" in name:
            key = "fft"
        else:
            key = "other"
        stages[key] += us / 1000.0
    return {k: round(v, 4) for k, v in stages.items()}


def events_ms(torch, st, fn, calls):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(calls):
        fn()
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b) / calls


def bench_config(sdr, torch, dev, fmt, n, M, D, cmajor, calls, name, power, composed_n):
    import gen
    T = 16
    h = gen.lowpass_taps(T * M, 0.5 / M, 1.0)
    st = torch.cuda.current_stream(dev)
    d_in = make_input(torch, dev, fmt, n, 1234 + M + D)
    nf = n // D
    d_out = torch.empty((M, nf) if cmajor else (nf, M), dtype=torch.complex64, device=dev)
    bank = sdr.Pfb(h, M, D, fmt, channel_major=cmajor, stream=st)
    call = lambda: bank.process_dev(d_in, n, d_out, nf)  # noqa: E731
    assert call() == nf  # first call of a fresh handle: the frames spot_check recomputes
    torch.cuda.synchronize()
    err = spot_check(d_in, d_out, fmt, h, M, D, cmajor, nf)
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    ms = events_ms(torch, st, call, calls)
    stages = stage_times(torch, call)
    es = 2 if fmt == "u8iq" else 8
    bps = es + 8.0 * M / D
    gs = n / (ms * 1e-3) / 1e9
    rec = {"bench": "pfb", "fmt": fmt, "n_samples": n, "M": M, "D": D, "taps": T * M,
           "layout": "channel_major" if cmajor else "frame_major", "calls": calls, "ms_per_call": round(ms, 4),
           "gsamples_per_s": round(gs, 2), "bytes_per_sample": bps, "gb_per_s": round(gs * bps, 1),
           "frac_peak": round(gs * bps / PEAK_GBS, 4), "stages_ms": stages, "spot_err_rel": err,
           "gpu": name, "power_limit": power}
    if composed_n:
        # one channel of the composition users have today: Fir(g_k, L taps) + Decimate(D), on a shorter input
        k = 1
        g = (h.astype(np.float64) * np.exp(2j * np.pi * k * np.arange(h.size) / M)).astype(np.complex64)
        fir = sdr.Fir(g, fmt, decimation=D, stream=st)
        c_out = torch.empty(composed_n // D + 2, dtype=torch.complex64, device=dev)
        c_in = d_in[:(2 if fmt == "u8iq" else 1) * composed_n]
        fcall = lambda: fir.process_dev(c_in, composed_n, c_out, c_out.shape[0])  # noqa: E731
        fcall()
        torch.cuda.synchronize()
        c_ms = events_ms(torch, st, fcall, 3)
        rec["composed_extrapolated"] = {
            "what": "one Fir(g_k)+Decimate channel timed on %d samples, times M=%d channels, scaled to %d samples"
                    % (composed_n, M, n),
            "fir_path": fir.last_path, "one_channel_ms": round(c_ms, 4),
            "ms_per_call_extrapolated": round(c_ms * M * n / composed_n, 1),
            "speedup_extrapolated": round(c_ms * M * n / composed_n / ms, 1)}
        fir.close()
    bank.close()
    del d_in, d_out
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
        raise SystemExit("bench_pfb: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power = card()
    big = 1 << 22 if args.quick else 1 << 28
    mid = 1 << 22 if args.quick else 1 << 26
    configs = [("u8iq", big, 1024, 1024, False, 1 << 22), ("u8iq", big, 1024, 1024, True, 0),
               ("u8iq", big, 1024, 512, False, 1 << 22), ("u8iq", big, 1024, 512, True, 0),
               ("u8iq", big, 4096, 4096, False, 1 << 20), ("u8iq", big, 4096, 2048, False, 0),
               ("c64", mid, 1024, 1024, False, 1 << 20), ("c64", mid, 1024, 512, False, 0)]
    for fmt, n, M, D, cm, comp_n in configs:
        bench_config(sdr, torch, dev, fmt, n, M, D, cm, max(20, args.calls), name, power, comp_n)


if __name__ == "__main__":
    main()
