"""Down-converter bank (sdr_ddc) throughput on one GPU: one JSON line per config.

For each config: check output windows of a fresh handle's first call against the f64 rotated-taps form (so a fast wrong
answer cannot be reported), then time >= 20 back-to-back process_dev calls on device-resident data with CUDA events,
ALTERNATING with the composition users have without the bank: C x Fir(g_k, decimation=D) (complex taps
g_k = h e^{+2 pi i j Delta_k}) followed by a torch elementwise multiply with a precomputed derotation row
e^{-2 pi i phi_k(N_m)} per channel (the table is built before timing, which favours the composition).  Three rounds of
each; the best round of each is reported.  The per-kernel split of one call comes from torch.profiler in a separate run.

Bytes per input sample are algorithmic: 2 (u8 IQ) or 8 (c64) in, plus 8 C / D out; "frac_hbm" is that traffic over the
call time against 6552.3 GB/s, the HBM rate the rest of the project quotes as measured peak.  On the tensor path the
int8 MACs the kernel issues per input sample follow from its geometry (Ng columns x KS k-steps of 32 bytes x groups:
128 rows x 32 samples per tile = 4096 samples), and "frac_tensor" is that work over the call time against the
8192 int8 MAC / cycle / SM measured in scripts/probes/umma_rate_probe.cu, at the card's maximum SM clock.

    python scripts/bench_ddc.py [--calls 20] [--quick]
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
MAC_PER_CYCLE_SM = 8192
RATE = 2.4e6


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        name, power, clk = [s.strip() for s in out.strip().split(",")[:3]]
        return name, power + " W", float(clk) * 1e6
    except Exception as e:  # the numbers still stand; say the card could not be read
        return "unknown (%s)" % e, "unknown", float("nan")


def tc_geometry(C, D, L):
    """ddc.cu ddc_tc_geometry: (Ng, KS, groups) of the tensor path, or None for the CUDA-core kernel"""
    if 32 % D or L > 511:
        return None
    PC = 32 // D
    KS = (L + 7 + 32 - D + 15) // 16
    Nc8 = -(-(6 * PC) // 8) * 8
    stage = (64 * 127 + 32 * KS + 1023) // 1024 * 1024
    cmax = 0
    for c in range(1, C + 1):
        Ng = -(-(c * Nc8) // 16) * 16
        if c * Nc8 > 256 or KS * Ng * 32 + 2 * stage + 1280 > 220 * 1024:
            break
        cmax = c
    if not cmax:
        return None
    groups = -(-C // cmax)
    Cg = -(-C // groups)
    return -(-(Cg * Nc8) // 16) * 16, KS, groups


def make_input(torch, dev, fmt, n, seed):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    if fmt == "u8iq":
        return torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    return torch.complex(torch.rand(n, device=dev, generator=g) * 2 - 1, torch.rand(n, device=dev, generator=g) * 2 - 1)


def spot_check(d_in, d_out, fmt, h, incs, D, nf):
    import ddc_ref as R
    import oracle_lib as O
    L = h.size
    worst = 0.0
    for j0 in (0, nf // 2, nf - 40):
        outs = np.arange(j0, j0 + 40)
        s0 = max(0, (j0 + 1) * D - L) // D * D  # a multiple of D: the window keeps the decimation phase
        s1 = (j0 + 40) * D
        raw = d_in[2 * s0:2 * s1] if fmt == "u8iq" else d_in[s0:s1]
        x = O.unpack_u8iq(raw.cpu().numpy()) if fmt == "u8iq" else raw.cpu().numpy()
        # the window's own first sample is stream sample s0: first_sample = s0 places the phase, and x[< s0] (never
        # needed except at j0 = 0, where s0 = 0) reads as zero
        want = R.rotated_f64(h, x, incs, D, first=s0, outputs=outs - s0 // D)
        got = d_out[:, j0:j0 + 40].cpu().numpy()
        worst = max(worst, max(float(np.abs(got[k] - want[k]).max() / np.abs(want[k]).max()) for k in range(len(incs))))
    if not worst <= 1e-5:
        raise SystemExit("spot outputs differ from f64 truth: %.3g of max|y| > 1e-5" % worst)
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
        for key in ("ddc_tc_kernel", "ddc_general_kernel", "fir_umma", "fir_", "Memcpy", "mul"):
            if key.lower() in name.lower():
                name = key
                break
        else:
            name = name[:40]
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        split[name] = split.get(name, 0.0) + us / 1000.0
    return {k: round(v, 4) for k, v in split.items()}


def bench_config(sdr, torch, dev, fmt, n, C, D, calls, name, power, clk):
    import ddc_ref as R
    import gen
    L = 255
    h = gen.lowpass_taps(L, 100e3 * 10 / D, RATE)  # C3's 255 taps (100 kHz at D = 10) scaled to the output rate
    freqs = [-1.1e6 + 2.2e6 * (k + 0.5) / C for k in range(C)]
    st = torch.cuda.current_stream(dev)
    d_in = make_input(torch, dev, fmt, n, 4321 + C + D)
    nf = n // D
    cap = nf + 1  # later calls of a stream whose length is not a multiple of D complete nf or nf + 1 outputs
    d_out = torch.empty((C, cap), dtype=torch.complex64, device=dev)
    bank = sdr.Ddc(h, freqs, RATE, D, fmt, stream=st)
    incs = [int(v) for v in bank.phase_inc]
    call = lambda: bank.process_dev(d_in, n, d_out, cap)  # noqa: E731
    assert call() == nf
    torch.cuda.synchronize()
    err = spot_check(d_in, d_out, fmt, h, incs, D, nf)
    path = bank.last_path

    # the composition: C x Fir(g_k) + Decimate(D), then out *= derotation row (precomputed)
    firs = [sdr.Fir(R.rotated_taps(h, inc).astype(np.complex64), fmt, decimation=D, stream=st) for inc in incs]
    c_out = torch.empty((C, cap), dtype=torch.complex64, device=dev)
    N = (np.arange(nf, dtype=np.uint64) + np.uint64(1)) * np.uint64(D) - np.uint64(1)
    derot = torch.stack([torch.from_numpy(R.rot(R.phases(0, N, inc)).astype(np.complex64)) for inc in incs]).to(dev)

    def composed():
        for k, f in enumerate(firs):
            f.process_dev(d_in, n, c_out[k], cap)
        c_out[:, :nf].mul_(derot)
    composed()
    torch.cuda.synchronize()
    diff = float((c_out[:, :nf] - d_out[:, :nf]).abs().max() / d_out[:, :nf].abs().max())
    for f in firs:
        f.reset()
    fir_path = firs[0].last_path

    bank_ms, comp_ms = [], []
    for _ in range(3):
        bank_ms.append(events_ms(torch, st, call, calls))
        for f in firs:
            f.reset()
        comp_ms.append(events_ms(torch, st, composed, calls))
    ms, cms = min(bank_ms), min(comp_ms)
    split = kernel_split(torch, call)
    comp_split = kernel_split(torch, composed)
    es = 2 if fmt == "u8iq" else 8
    bps = es + 8.0 * C / D
    gs = n / (ms * 1e-3) / 1e9
    rec = {"bench": "ddc", "fmt": fmt, "n_samples": n, "C": C, "D": D, "taps": L, "path": path, "calls": calls,
           "ms_per_call": round(ms, 4), "ms_rounds": [round(v, 4) for v in bank_ms],
           "gsamples_per_s": round(gs, 2), "bytes_per_sample": bps, "gb_per_s": round(gs * bps, 1),
           "frac_hbm": round(gs * bps / PEAK_GBS, 4), "kernels_ms": split, "spot_err_rel": err}
    geo = tc_geometry(C, D, L) if fmt == "u8iq" else None
    if path == 2 and geo:
        Ng, KS, groups = geo
        macs = Ng * KS * 32 * 128 * groups / 4096  # int8 MACs issued per input sample
        rec["tensor"] = {"Ng": Ng, "KS": KS, "groups": groups, "int8_mac_per_sample": macs,
                         "frac_tensor": round(macs * gs * 1e9 / (MAC_PER_CYCLE_SM * 148 * clk), 4),
                         "sm_clock_max_mhz": clk / 1e6}
    rec["composed"] = {"what": "%d x Fir(g_k, decimation=%d) + torch derotation multiply, same input, alternating"
                               % (C, D),
                       "fir_path": fir_path, "ms_per_call": round(cms, 4), "ms_rounds": [round(v, 4) for v in comp_ms],
                       "gsamples_per_s": round(n / (cms * 1e-3) / 1e9, 2), "kernels_ms": comp_split,
                       "max_diff_vs_bank_rel": diff}
    rec["speedup_vs_composed"] = round(cms / ms, 2)
    rec["gpu"], rec["power_limit"] = name, power
    for f in firs:
        f.close()
    bank.close()
    del d_in, d_out, c_out, derot
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
        raise SystemExit("bench_ddc: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    big = 1 << 22 if args.quick else 1 << 28
    mid = 1 << 22 if args.quick else 1 << 26
    configs = [("u8iq", big, 1, 8), ("u8iq", big, 4, 8), ("u8iq", big, 8, 8), ("u8iq", big, 16, 8),
               ("u8iq", big, 16, 16), ("u8iq", big, 8, 10), ("c64", mid, 8, 8)]
    for fmt, n, C, D in configs:
        bench_config(sdr, torch, dev, fmt, n, C, D, max(20, args.calls), name, power, clk)


if __name__ == "__main__":
    main()
