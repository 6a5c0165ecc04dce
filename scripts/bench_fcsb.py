"""Fast-convolution synthesis bank (sdr_fcsb) throughput on one GPU: one JSON line per config.

For each config: check spot outputs of a fresh handle's first call against the f64 definition (so a fast wrong answer
cannot be reported), then alternate, three rounds, 20 back-to-back process_dev calls of the bank on device-resident
rows with the comparison in the same run -- sdr_duc when every I_k is equal, else one sdr_duc per distinct I_k plus a
torch sum -- each timed with CUDA events; the best round counts.  Stage times of one call come from a separate
torch.profiler run.  Rates are output positions per second.  Per output the script reports the algorithmic HBM traffic
(8 sum_k 1 / I_k bytes of rows in, 8 out; "frac_hbm" against 6552.3 GB/s, the HBM rate the rest of the project quotes
as measured peak), the traffic of the stages between the kernels (mostly through L2) and the flops of the two
transforms and the unfold.  The card's name, power limit and max SM clock are read in the same run.  The last config
is the fcfb -> fcsb round trip on 2^28 u8 IQ samples.

    python scripts/bench_fcsb.py [--calls 20] [--quick]
"""
import argparse
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "unnamed-rust-sdr_b200"), os.path.join(ROOT, "tests"), os.path.dirname(__file__)):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench_duc import card, taps_for  # noqa: E402
from bench_pfb import PEAK_GBS, events_ms  # noqa: E402

F0 = (1 << 40) + 12345
TWO64 = 1 << 64


def stage_times(torch, fn):
    """per-stage device time (ms) of one call, from torch.profiler kernel / copy records"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    keys = ("fcsb_gather", "fcsb_unfold", "fcsb_store", "fcsb_carry", "fcfb", "duc_kernel", "fft")
    stages = {k: 0.0 for k in keys + ("copy", "other")}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        name = e.name.lower()
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        key = next((k for k in keys if k in name), "copy" if "memcpy" in name else "other")
        stages[key] += us / 1000.0
    return {k: round(v, 4) for k, v in stages.items() if v > 0}


def budget(Is, N, P):
    """per output: HBM bytes, bytes between the stages and flops of one block (small DFTs, unfold, N-point DFT)"""
    C = len(Is)
    g = [int(I) & -int(I) for I in Is]
    M = [N // gk for gk in g]
    hbm = 8.0 + 8.0 * sum(1.0 / int(I) for I in Is)
    # gather writes v, the small plans read v and write V, the unfold reads V and G' (once per 4 blocks) and writes S,
    # the N-point plan reads S and writes X, the store reads the last P of X
    l2 = 8.0 * (4 * sum(M) + C * N / 4 + 3 * N + P) / P
    flop = (sum(5 * m * math.log2(m) for m in M) + 8 * C * N + 5 * N * math.log2(N)) / P
    return hbm, l2, flop


def spot_check(d_y, d_out, h, incs, Is, first, cnt):
    import fcsb_ref as Q
    L = h.shape[-1]
    Il = Q.lcm_of(Is)
    worst = 0.0
    for t0 in (0, cnt // 2 + 5, cnt - 2048):
        lo = max(0, (t0 - L) // Il * Il)
        hi = -(-(t0 + 2048) // Il) * Il
        rows = [d_y[k, lo // int(I):hi // int(I)].cpu().numpy() for k, I in enumerate(Is)]
        want = Q.definition_f64(h.astype(np.float64), rows, incs, Is, (first + lo) % TWO64)[t0 - lo:t0 - lo + 2048]
        got = d_out[t0:t0 + 2048].cpu().numpy()
        worst = max(worst, float(np.abs(got - want).max() / np.abs(want).max()))
    N, _ = Q.geometry(L, Is)
    if not worst <= 2e-5 * math.log2(N):
        raise SystemExit("spot outputs differ from f64 truth: %.3g of max|x| > %.3g" % (worst, 2e-5 * math.log2(N)))
    return worst


class DucPerRate:
    """the composition a user writes today: one sdr_duc per distinct I over its consecutive channels, summed in torch"""

    def __init__(self, sdr, h, freqs, Is, first, st):
        self.groups = []
        k0 = 0
        while k0 < len(Is):
            k1 = k0
            while k1 < len(Is) and Is[k1] == Is[k0]:
                k1 += 1
            self.groups.append((k0, k1, int(Is[k0]), sdr.Duc(np.ascontiguousarray(h[k0:k1]), freqs[k0:k1], 1.0,
                                                              int(Is[k0]), first_sample=first, stream=st)))
            k0 = k1

    def __call__(self, torch, d_y, n, d_out, d_tmp):
        for q, (k0, k1, I, duc) in enumerate(self.groups):
            dst = d_out if q == 0 else d_tmp
            duc.process_dev(d_y[k0:], n // I, dst, n, d_y.stride(0))
            if q:
                d_out += d_tmp


def bench_config(sdr, torch, dev, n, Is, L, calls, name, power, clk):
    st = torch.cuda.current_stream(dev)
    C_ = len(Is)
    Imin = min(Is)
    h = np.concatenate([taps_for(1, L, I) for I in Is]).astype(np.float32)
    freqs = np.linspace(-0.4, 0.4, C_)
    g = torch.Generator(device=dev).manual_seed(99 + C_ + L)
    d_y = torch.randn((C_, n // Imin), dtype=torch.complex64, device=dev, generator=g)
    bank = sdr.Fcsb(h, freqs, 1.0, Is, first_sample=F0, stream=st)
    N, P = bank.geometry
    cap = n + P
    d_out = torch.empty(cap, dtype=torch.complex64, device=dev)
    incs = [int(v) for v in bank.phase_inc]
    call = lambda: bank.process_dev(d_y, n, d_out, cap)  # noqa: E731
    cnt = call()
    torch.cuda.synchronize()
    err = spot_check(d_y, d_out, h, incs, Is, F0, cnt)
    comp = DucPerRate(sdr, h, freqs, Is, F0, st)
    d_ref = torch.empty(n, dtype=torch.complex64, device=dev)
    d_tmp = torch.empty(n, dtype=torch.complex64, device=dev) if len(comp.groups) > 1 else None
    comp(torch, d_y, n, d_ref, d_tmp)
    torch.cuda.synchronize()
    diff = float((d_ref[:cnt] - d_out[:cnt]).abs().max() / d_ref[:cnt].abs().max())
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    bank_ms, comp_ms = [], []
    for _ in range(3):  # alternate the two in one run
        bank_ms.append(events_ms(torch, st, call, calls))
        comp_ms.append(events_ms(torch, st, lambda: comp(torch, d_y, n, d_ref, d_tmp), calls))
    ms, cms = min(bank_ms), min(comp_ms)
    gs = n / (ms * 1e-3) / 1e9
    hbm, l2, flop = budget(Is, N, P)
    rec = {"bench": "fcsb", "n_outputs": n, "C": C_, "I": sorted(set(int(i) for i in Is)), "taps": L, "N": N, "P": P,
           "calls": calls, "spot_err_rel": err, "ms_per_call": round(ms, 4), "gsamples_per_s": round(gs, 2),
           "hbm_bytes_per_output": round(hbm, 2), "stage_bytes_per_output": round(l2, 1),
           "flop_per_output": round(flop, 1), "frac_hbm": round(gs * hbm / PEAK_GBS, 4),
           "frac_fp32": round(gs * 1e9 * flop / (148 * 128 * 2 * clk * 1e6), 3),
           "duc_comparison": {"handles": len(comp.groups), "ms_per_call": round(cms, 3), "max_rel_diff": diff,
                              "ratio": round(cms / ms, 2)},
           "rounds_ms": [round(v, 4) for v in bank_ms], "stages_ms": stage_times(torch, call),
           "gpu": name, "power_limit": power, "max_sm_clock_mhz": clk}
    bank.close()
    del d_y, d_out, d_ref, d_tmp, comp
    torch.cuda.empty_cache()
    print(json.dumps(rec), flush=True)
    return rec


def bench_round_trip(sdr, torch, dev, n, calls, name, power):
    """u8 IQ -> Fcfb(h) -> Fcsb(f = D h) on the device, C = 8, D = I = 8, L = 4095"""
    import pfs_ref
    C_, D, L = 8, 8, 4095
    h = pfs_ref.kaiser_lowpass(L, 0.5 / D, 8.0).astype(np.float32)
    f = (D * h).astype(np.float32)
    freqs = np.linspace(-0.4, 0.4, C_)
    st = torch.cuda.current_stream(dev)
    g = torch.Generator(device=dev).manual_seed(7)
    d_in = torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    ana = sdr.Fcfb(h, freqs, 1.0, [D] * C_, "u8iq", first_sample=F0, stream=st)
    syn = sdr.Fcsb(f, freqs, 1.0, [D] * C_, first_sample=F0 - (L - 1), stream=st)
    N, P = ana.geometry
    stride = n // D + P
    d_y = torch.empty((C_, stride), dtype=torch.complex64, device=dev)
    d_x = torch.empty(n + 2 * P, dtype=torch.complex64, device=dev)

    def call():
        got = ana.process_dev(d_in, n, d_y, stride, stride)
        syn.process_dev(d_y, int(got[0]) * D, d_x, n + 2 * P, stride)
    call()
    torch.cuda.synchronize()
    assert bool(torch.isfinite(torch.view_as_real(d_x[n // 2:n // 2 + 4096])).all())
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    ms = min(events_ms(torch, st, call, calls) for _ in range(3))
    gs = n / (ms * 1e-3) / 1e9
    rec = {"bench": "fcfb_fcsb_round_trip", "fmt": "u8iq", "n_samples": n, "C": C_, "D": D, "taps": L, "N": N, "P": P,
           "calls": calls, "ms_per_call": round(ms, 4), "gsamples_per_s": round(gs, 2),
           "stages_ms": stage_times(torch, call), "gpu": name, "power_limit": power}
    ana.close()
    syn.close()
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--quick", action="store_true", help="2^22 outputs per config (a rehearsal, not a measurement)")
    args = ap.parse_args()
    import torch
    import sdr_b200 as sdr
    if not torch.cuda.is_available() or sdr.device_count() < 1:
        raise SystemExit("bench_fcsb: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    big = 1 << 22 if args.quick else 1 << 28
    calls = max(20, args.calls)
    for Is, L in [([8] * 8, 255), ([8] * 8, 4095), ([8, 8, 16, 16, 32, 32, 64, 64], 4095), ([10] * 8, 255)]:
        Il = int(np.lcm.reduce(Is))
        bench_config(sdr, torch, dev, big // Il * Il, Is, L, calls, name, power, clk)
    bench_round_trip(sdr, torch, dev, big, calls, name, power)


if __name__ == "__main__":
    main()
