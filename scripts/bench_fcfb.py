"""Fast-convolution channel bank (sdr_fcfb) throughput on one GPU: one JSON line per config, plus one accuracy line.

For each config: check spot outputs of a fresh handle's first call against the f64 rotated-taps form (so a fast wrong
answer cannot be reported), then time 20 back-to-back process_dev calls on device-resident data with CUDA events,
ALTERNATING with the comparison (sdr_ddc, one sdr_ddc per distinct D, sdr_fir, or C x Fir + a torch derotation
multiply) in the same run.  Three rounds of each; the best round of each is reported.  A comparison whose call takes
longer than 100 ms is timed over fewer back-to-back calls (at least 3) so that a round stays near 2 s; "cmp_calls"
says how many.  The stage split of one call (gather, forward FFT, fold, inverse FFTs, store) comes from torch.profiler
in a separate run, with kernels assigned to stages by their order in the call.

Bytes per input sample are algorithmic: 2 (u8 IQ) or 8 (c64) in, plus 8 sum_k 1/D_k out.  The fold's L2 traffic is
8 C N / P bytes of spectra per input sample plus the G'_k reads (8 sum_k N / P per sample, shared by 4 blocks).

    python scripts/bench_fcfb.py [--calls 20] [--quick]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "unnamed-rust-sdr_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

RATE = 2.4e6


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        name, power = [s.strip() for s in out.strip().split(",")[:2]]
        return name, power + " W"
    except Exception as e:  # the numbers still stand; say the card could not be read
        return "unknown (%s)" % e, "unknown"


def make_input(torch, dev, fmt, n, seed):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    if fmt == "u8iq":
        return torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    return torch.complex(torch.rand(n, device=dev, generator=g) * 2 - 1, torch.rand(n, device=dev, generator=g) * 2 - 1)


def spot_check(d_in, d_out, cnt, fmt, h, incs, ds, N):
    """windows of 40 outputs at the start, middle and end of every channel against the f64 rotated-taps form, relative
    to the channel's largest output (the per-channel bar: FFT round-off follows the block, not a window's own level,
    which is small in the filter's start-up)"""
    import ddc_ref as R
    import oracle_lib as O
    L = h.size
    worst = 0.0
    for k, (inc, D) in enumerate(zip(incs, ds)):
        nf = int(cnt[k])
        peak = float(d_out[k, :nf].abs().max())
        for j0 in (0, nf // 2, nf - 40):
            outs = np.arange(j0, j0 + 40)
            s0 = max(0, (j0 + 1) * D - L) // D * D
            s1 = (j0 + 40) * D
            raw = d_in[2 * s0:2 * s1] if fmt == "u8iq" else d_in[s0:s1]
            x = O.unpack_u8iq(raw.cpu().numpy()) if fmt == "u8iq" else raw.cpu().numpy()
            want = R.rotated_f64(h, x, [inc], D, first=s0, outputs=outs - s0 // D)[0]
            got = d_out[k, j0:j0 + 40].cpu().numpy()
            worst = max(worst, float(np.abs(got - want).max() / peak))
    bar = 2e-5 * math.log2(N)
    if not worst <= bar:
        raise SystemExit("spot outputs differ from f64 truth: %.3g of max|y| > %.3g" % (worst, bar))
    return worst


def events_ms(torch, st, fn, calls):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(calls):
        fn()
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b) / calls


def _events(torch, fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    evs = [e for e in prof.events() if e.device_type.name == "CUDA"]
    evs.sort(key=lambda e: e.time_range.start)
    return evs


def _us(e):
    return e.device_time if hasattr(e, "device_time") else e.cuda_time


def stage_split(torch, fn):
    """device ms per stage of one bank call: kernels between gather and fold are the forward FFT, between fold and
    store the inverse FFTs"""
    split, stage = {}, "other"
    for e in _events(torch, fn):
        nm = e.name
        if "fcfb_gather" in nm:
            stage, key = "fft_forward", "gather"
        elif "fcfb_fold" in nm:
            stage, key = "fft_inverse", "fold"
        elif "fcfb_store" in nm:
            stage, key = "other", "store"
        elif "Memcpy" in nm or "memcpy" in nm.lower():
            key = "memcpy"
        else:
            key = stage
        split[key] = split.get(key, 0.0) + _us(e) / 1000.0
    return {k: round(v, 4) for k, v in split.items()}


def kernel_split(torch, fn):
    split = {}
    for e in _events(torch, fn):
        key = e.name[:40]
        split[key] = split.get(key, 0.0) + _us(e) / 1000.0
    return {k: round(v, 4) for k, v in split.items()}


def bench_config(sdr, torch, dev, row, fmt, n, ds, L, compare, calls, name, power, zero_freq=False):
    import ddc_ref as R
    import gen
    C = len(ds)
    h = gen.lowpass_taps(L, 100e3 * 10 / max(ds), RATE)
    freqs = [0.0] if zero_freq else [-1.1e6 + 2.2e6 * (k + 0.5) / C for k in range(C)]
    st = torch.cuda.current_stream(dev)
    d_in = make_input(torch, dev, fmt, n, 4321 + C + L + sum(ds))
    bank = sdr.Fcfb(h, freqs, RATE, ds, fmt, stream=st)
    N, P = bank.geometry
    incs = [int(v) for v in bank.phase_inc]
    cnt = bank.output_count(n)
    cap = int(cnt.max()) + P  # later calls complete up to one block more
    d_out = torch.empty((C, cap), dtype=torch.complex64, device=dev)
    call = lambda: bank.process_dev(d_in, n, d_out, cap)  # noqa: E731
    got = call()
    torch.cuda.synchronize()
    assert list(got) == list(cnt)
    err = spot_check(d_in, d_out, cnt, fmt, h, incs, ds, N)

    # the comparison, checked against the bank on the outputs both have released
    cmp_objs, cmp_info = [], {}
    if compare == "ddc":
        dd = sdr.Ddc(h, freqs, RATE, ds[0], fmt, stream=st)
        c_out = torch.empty((C, n // ds[0] + 1), dtype=torch.complex64, device=dev)
        cmp_objs.append(dd)

        def cmp_call():
            dd.process_dev(d_in, n, c_out, n // ds[0] + 1)
        cmp_call()
        torch.cuda.synchronize()
        cmp_info["path"] = dd.last_path
        rows = [(k, k) for k in range(C)]
    elif compare == "ddc_per_d":
        outs = []
        for D in sorted(set(ds)):
            ks = [k for k in range(C) if ds[k] == D]
            dd = sdr.Ddc(h, [freqs[k] for k in ks], RATE, D, fmt, stream=st)
            o = torch.empty((len(ks), n // D + 1), dtype=torch.complex64, device=dev)
            outs.append((dd, o, D, ks))
            cmp_objs.append(dd)

        def cmp_call():
            for dd, o, D, _ in outs:
                dd.process_dev(d_in, n, o, n // D + 1)
        cmp_call()
        torch.cuda.synchronize()
        cmp_info["paths"] = [dd.last_path for dd, _, _, _ in outs]
        cmp_info["handles"] = len(outs)
    elif compare == "fir":
        f = sdr.Fir(h, fmt, decimation=ds[0], stream=st)
        c_out = torch.empty((1, n // ds[0] + 1), dtype=torch.complex64, device=dev)
        cmp_objs.append(f)

        def cmp_call():
            f.reset()
            f.process_dev(d_in, n, c_out[0], n // ds[0] + 1)
        cmp_call()
        torch.cuda.synchronize()
        cmp_info["fir_path"] = f.last_path
        rows = [(0, 0)]
    else:  # "firs": C x Fir(g_k, decimation=D) + torch derotation multiply (table precomputed)
        D = ds[0]
        nf = n // D
        firs = [sdr.Fir(R.rotated_taps(h, inc).astype(np.complex64), fmt, decimation=D, stream=st) for inc in incs]
        c_out = torch.empty((C, nf + 1), dtype=torch.complex64, device=dev)
        Nm = (np.arange(nf, dtype=np.uint64) + np.uint64(1)) * np.uint64(D) - np.uint64(1)
        derot = torch.stack([torch.from_numpy(R.rot(R.phases(0, Nm, inc)).astype(np.complex64)) for inc in incs]).to(dev)
        cmp_objs.extend(firs)

        def cmp_call():
            for k, f in enumerate(firs):
                f.reset()
                f.process_dev(d_in, n, c_out[k], nf + 1)
            c_out[:, :nf].mul_(derot)
        cmp_call()
        torch.cuda.synchronize()
        cmp_info["fir_path"] = firs[0].last_path
        rows = [(k, k) for k in range(C)]
    if compare == "ddc_per_d":
        diff = 0.0
        for dd, o, D, ks in outs:
            for i, k in enumerate(ks):
                m = int(cnt[k])
                diff = max(diff, float((o[i, :m] - d_out[k, :m]).abs().max() / d_out[k, :m].abs().max()))
    else:
        diff = max(float((c_out[j, :int(cnt[k])] - d_out[k, :int(cnt[k])]).abs().max()
                         / d_out[k, :int(cnt[k])].abs().max()) for k, j in rows)

    bank.reset()
    ms0 = events_ms(torch, st, call, 1)
    cms0 = events_ms(torch, st, cmp_call, 1)
    ccalls = calls if cms0 <= 100 else max(3, int(2000 / cms0))
    bank_ms, cmp_ms = [], []
    for _ in range(3):
        bank.reset()
        bank_ms.append(events_ms(torch, st, call, calls))
        cmp_ms.append(events_ms(torch, st, cmp_call, ccalls))
    ms, cms = min(bank_ms), min(cmp_ms)
    bank.reset()
    split = stage_split(torch, call)
    cmp_split = kernel_split(torch, cmp_call)
    es = 2 if fmt == "u8iq" else 8
    bps = es + 8.0 * sum(1.0 / d for d in ds)
    gs = n / (ms * 1e-3) / 1e9
    rec = {"bench": "fcfb", "row": row, "fmt": fmt, "n_samples": n, "C": C, "D": ds, "taps": L, "N": N, "P": P,
           "calls": calls, "ms_per_call": round(ms, 4), "ms_rounds": [round(v, 4) for v in bank_ms],
           "gsamples_per_s": round(gs, 2), "bytes_per_sample": round(bps, 3),
           "fold_l2_bytes_per_sample": round(8.0 * C * N / P + 8.0 * C * N / P / 4, 1),
           "stages_ms": split, "spot_err_rel": err}
    cmp_info.update({"what": compare, "cmp_calls": ccalls, "ms_per_call": round(cms, 4),
                     "ms_rounds": [round(v, 4) for v in cmp_ms], "gsamples_per_s": round(n / (cms * 1e-3) / 1e9, 2),
                     "kernels_ms": cmp_split, "max_diff_vs_bank_rel": diff})
    rec["compared"] = cmp_info
    rec["speedup"] = round(cms / ms, 2)
    rec["gpu"], rec["power_limit"] = name, power
    for o in cmp_objs:
        o.close()
    bank.close()
    del d_in, d_out
    torch.cuda.empty_cache()
    print(json.dumps(rec), flush=True)
    return rec


def accuracy(sdr, name, power):
    """error of the bank and of sdr_ddc on the same inputs: random u8 (every channel carries signal) and a channel
    holding only noise 60 dB below an out-of-band tone (error over eps log2(N) ||h||_2 rms, eps = 2^-24)"""
    import gen
    from scipy import signal as S
    import ddc_ref as R
    import oracle_lib as O

    def truth(h, x, incs, D):
        rows = []
        for inc in incs:
            z = np.asarray(x, np.complex128) * R.rot(R.phases(0, np.arange(x.size), inc))
            rows.append(S.fftconvolve(z, h.astype(np.float64))[:x.size][(np.arange(x.size // D) + 1) * D - 1])
        return rows

    rec = {"bench": "fcfb_accuracy", "gpu": name, "power_limit": power}
    # every channel carries signal
    L, D, n = 255, 8, 1 << 20
    h = gen.lowpass_taps(L, 100e3, RATE)
    raw = gen.random_u8(2 * n, 3)
    x = O.unpack_u8iq(raw)
    freqs = [-1.1e6 + 2.2e6 * (k + 0.5) / 8 for k in range(8)]
    b = sdr.Fcfb(h, freqs, RATE, D, "u8iq")
    N, _ = b.geometry
    y = b.process(raw)
    yd = sdr.Ddc(h, freqs, RATE, D, "u8iq").process(raw)
    yg = sdr.Ddc(h, freqs, RATE, D, "u8iq", general=True).process(raw)
    t = truth(h, x, list(b.phase_inc), D)
    rec["signal"] = {"L": L, "D": D, "N": N, "bar": 2e-5 * math.log2(N),
                     "fcfb_err_rel": max(float(np.abs(y[k] - t[k][:y[k].size]).max() / np.abs(t[k]).max())
                                         for k in range(8)),
                     "ddc_tc_err_rel": max(float(np.abs(yd[k] - t[k]).max() / np.abs(t[k]).max()) for k in range(8)),
                     "ddc_general_err_rel": max(float(np.abs(yg[k] - t[k]).max() / np.abs(t[k]).max())
                                                for k in range(8))}
    # the interferer case of tests/test_gpu_fcfb.py
    L, D, n = 1023, 8, 1 << 18
    h = gen.lowpass_taps(L, 50e3, RATE)
    tt = np.arange(n)
    rng = np.random.default_rng(5)
    x = (0.9 * np.exp(2j * np.pi * 700e3 / RATE * tt)
         + 0.9e-3 / math.sqrt(2) * (rng.standard_normal(n) + 1j * rng.standard_normal(n))).astype(np.complex64)
    b = sdr.Fcfb(h, [-300e3], RATE, D, "c64")
    N, _ = b.geometry
    y = b.process(x)[0]
    yd = sdr.Ddc(h, [-300e3], RATE, D, "c64").process(x)[0]
    t = truth(h, x, list(b.phase_inc), D)[0]
    rms = math.sqrt(float(np.mean(np.abs(x.astype(np.complex128)) ** 2)))
    unit = 2.0 ** -24 * math.log2(N) * float(np.linalg.norm(h.astype(np.float64))) * rms
    e, ed = float(np.abs(y - t[:y.size]).max()), float(np.abs(yd - t).max())
    rec["interferer"] = {"L": L, "D": D, "N": N, "fcfb_err": e, "fcfb_err_over_unit": round(e / unit, 3),
                         "ddc_err": ed, "ddc_err_over_unit": round(ed / unit, 3),
                         "fcfb_err_rel_channel": e / float(np.abs(t).max()),
                         "ddc_err_rel_channel": ed / float(np.abs(t).max()), "channel_rms": float(np.abs(t).std())}
    print(json.dumps(rec), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--quick", action="store_true", help="2^22 samples per config (a rehearsal, not a measurement)")
    ap.add_argument("--rows", default="1,2,3,4,5,6")
    args = ap.parse_args()
    import torch
    import sdr_b200 as sdr
    if not torch.cuda.is_available() or sdr.device_count() < 1:
        raise SystemExit("bench_fcfb: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power = card()
    big = 1 << 22 if args.quick else 1 << 28
    mid = 1 << 22 if args.quick else 1 << 26
    rows = {1: ("c64", mid, [8] * 8, 255, "ddc", False),
            2: ("u8iq", big, [10] * 8, 255, "ddc", False),
            3: ("u8iq", big, [8] * 8, 4095, "ddc", False),
            4: ("u8iq", big, [8, 8, 16, 16, 32, 32, 64, 64], 4095, "ddc_per_d", False),
            5: ("c64", mid, [1], 4095, "fir", True),
            6: ("u8iq", big, [8] * 8, 255, "ddc", False)}
    for r in [int(v) for v in args.rows.split(",")]:
        fmt, n, ds, L, cmp, zf = rows[r]
        bench_config(sdr, torch, dev, r, fmt, n, ds, L, cmp, max(20, args.calls), name, power, zero_freq=zf)
        if r == 2:  # the same row against C x Fir + derotation
            bench_config(sdr, torch, dev, r, fmt, n, ds, L, "firs", max(20, args.calls), name, power)
    accuracy(sdr, name, power)


if __name__ == "__main__":
    main()
