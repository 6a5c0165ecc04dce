"""Polyphase synthesis bank (sdr_pfs) throughput on one GPU: one JSON line per config.

For each config: check spot outputs of a fresh handle's first call against the f64 polyphase form (so a fast wrong
answer cannot be reported), time 20 back-to-back process_dev calls on device-resident frames with CUDA events, and
split one call into stages (gather / FFT / back end / copies) with torch.profiler in a separate run.  Bytes per output
sample are algorithmic: 8 M / D of frames in plus 8 out.  "frac_peak" is that traffic over the call time against
6552.3 GB/s, the HBM rate the rest of the project quotes as measured peak.

Alternating with the bank, the composition a user would write in torch -- torch.fft.fft over the frames, then the
polyphase sum as a gather and an einsum, in chunks of frames -- is timed on the same frames and checked against the
bank.  The last config is the Pfb -> Pfs round trip on u8 IQ, with its SNR against the delayed input.

    python scripts/bench_pfs.py [--calls 20] [--quick]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "unnamed-rust-sdr_b200"), os.path.join(ROOT, "tests"), os.path.dirname(__file__)):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench_pfb import PEAK_GBS, card, events_ms  # noqa: E402


def stage_times(torch, fn):
    """per-stage device time (ms) of one call, from torch.profiler kernel / copy records"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    stages = {"gather": 0.0, "fft": 0.0, "back_end": 0.0, "pfb_front_end": 0.0, "copy": 0.0, "other": 0.0}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        name = e.name.lower()
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        if "pfs_gather" in name:
            key = "gather"
        elif "pfs_back" in name:
            key = "back_end"
        elif "pfb_front" in name:
            key = "pfb_front_end"
        elif "memcpy" in name:
            key = "copy"
        elif "fft" in name or "bluestein" in name:
            key = "fft"
        else:
            key = "other"
        stages[key] += us / 1000.0
    return {k: round(v, 4) for k, v in stages.items()}


class TorchComposition:
    """torch.fft.fft over the frames, V = Y[:, (-r) mod M], and xh[m D + j] = sum_i w[j, i] V[m + off[j, i], col[j, i]]
    by gather + einsum, in chunks of frames (the frames before the stream are zero)"""

    def __init__(self, torch, dev, f, M, D, chunk):
        L = f.size
        self.torch, self.M, self.D, self.chunk = torch, M, D, chunk
        self.H = -(-(L - 1) // D)
        I = -(-L // D)
        j = np.arange(D)[:, None]
        i = np.arange(I)[None, :]
        c = (j + 1) % D
        n = c + i * D
        # frame of tap i relative to the chunk's first frame, + H; taps past L (weight 0) point anywhere valid
        off = np.maximum((j + 1) // D - 1 - i + self.H, 0)
        col = (-(n % M)) % M                                  # V[n mod M] = Y[(-n) mod M]
        w = np.where(n < L, np.asarray(f, np.float64)[np.minimum(n, L - 1)], 0.0)
        self.idx = torch.from_numpy(off * M + col).to(dev)
        self.w = torch.from_numpy(w.astype(np.float32)).to(dev).to(torch.complex64)
        self.pad = torch.zeros((self.H, M), dtype=torch.complex64, device=dev)

    def __call__(self, d_y, nf, d_out):
        torch, M, D, H = self.torch, self.M, self.D, self.H
        for f0 in range(0, nf, self.chunk):
            cnt = min(self.chunk, nf - f0)
            lo = f0 - H
            src = d_y[max(lo, 0):f0 + cnt]
            if lo < 0:
                src = torch.cat([self.pad[:-lo], src])
            Y = torch.fft.fft(src, dim=1).reshape(-1)
            g = Y[torch.arange(cnt, device=Y.device)[:, None, None] * M + self.idx[None]]
            d_out[f0 * D:(f0 + cnt) * D] = torch.einsum("mji,ji->mj", g, self.w).reshape(-1)


def spot_check(d_y, d_out, f, M, D, cmajor, nf):
    import pfs_ref as R
    L = f.size
    worst = 0.0
    n = nf * D
    for t0 in (0, n // 2 + 5, n - 2048):
        f0 = max(0, t0 // D - (L // D + 2))
        f1 = (t0 + 2048) // D + 1
        y = (d_y[:, f0:f1].T if cmajor else d_y[f0:f1]).cpu().numpy()
        want = R.polyphase_f64(f, y, M, D, outputs=np.arange(t0, t0 + 2048) - f0 * D)
        got = d_out[t0:t0 + 2048].cpu().numpy()
        worst = max(worst, float(np.abs(got - want).max() / np.abs(want).max()))
    bar = 1e-5 * np.log2(M)
    if not worst <= bar:
        raise SystemExit("spot outputs differ from f64 truth: %.3g of max|x| > %.3g" % (worst, bar))
    return worst


def bench_config(sdr, torch, dev, n_out, M, D, cmajor, calls, name, power, compare):
    import pfs_ref as R
    T = 12
    f = R.prototype_pair(M, D, T)[1].astype(np.float32)
    st = torch.cuda.current_stream(dev)
    nf = n_out // D
    g = torch.Generator(device=dev).manual_seed(99 + M + D)
    d_y = torch.randn((M, nf) if cmajor else (nf, M), dtype=torch.complex64, device=dev, generator=g)
    d_out = torch.empty(nf * D, dtype=torch.complex64, device=dev)
    bank = sdr.Pfs(f, M, D, channel_major=cmajor, stream=st)
    call = lambda: bank.process_dev(d_y, nf, d_out, nf * D)  # noqa: E731
    assert call() == nf * D
    torch.cuda.synchronize()
    err = spot_check(d_y, d_out, f, M, D, cmajor, nf)
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    rec = {"bench": "pfs", "n_outputs": nf * D, "M": M, "D": D, "taps": f.size,
           "layout": "channel_major" if cmajor else "frame_major", "calls": calls, "spot_err_rel": err,
           "gpu": name, "power_limit": power}
    if compare:
        comp = TorchComposition(torch, dev, f, M, D, max(1, (1 << 21) // D))
        d_ref = torch.empty_like(d_out)
        comp(d_y, nf, d_ref)
        bank.reset()  # the warm-up calls continued the stream: compare a fresh one
        call()
        torch.cuda.synchronize()
        diff = float((d_ref - d_out).abs().max() / d_ref.abs().max())
        bank_ms, comp_ms = [], []
        for _ in range(3):  # alternate the two in one run
            bank_ms.append(events_ms(torch, st, call, calls))
            comp_ms.append(events_ms(torch, st, lambda: comp(d_y, nf, d_ref), 2))
        ms = float(np.median(bank_ms))
        rec["torch_composition"] = {"ms_per_call": round(float(np.median(comp_ms)), 3), "max_rel_diff": diff,
                                    "ratio": round(float(np.median(comp_ms)) / ms, 2)}
        del d_ref
    else:
        ms = events_ms(torch, st, call, calls)
    bpo = 8.0 * M / D + 8
    gs = nf * D / (ms * 1e-3) / 1e9
    rec.update({"ms_per_call": round(ms, 4), "gsamples_per_s": round(gs, 2), "bytes_per_output": bpo,
                "gb_per_s": round(gs * bpo, 1), "frac_peak": round(gs * bpo / PEAK_GBS, 4),
                "stages_ms": stage_times(torch, call)})
    bank.close()
    del d_y, d_out
    torch.cuda.empty_cache()
    print(json.dumps(rec), flush=True)
    return rec


def bench_round_trip(sdr, torch, dev, n, calls, name, power):
    """u8 IQ -> Pfb(h) -> Pfs(f) on the device, M = 1024, D = 512, T = 12; SNR against x[t - T M]"""
    import oracle_lib as O
    import pfs_ref as R
    M, D, T = 1024, 512, 12
    h, f = R.prototype_pair(M, D, T)
    h, f = h.astype(np.float32), f.astype(np.float32)
    st = torch.cuda.current_stream(dev)
    g = torch.Generator(device=dev).manual_seed(7)
    d_in = torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    nf = n // D
    d_y = torch.empty((nf, M), dtype=torch.complex64, device=dev)
    d_x = torch.empty(n, dtype=torch.complex64, device=dev)
    ana, syn = sdr.Pfb(h, M, D, "u8iq", stream=st), sdr.Pfs(f, M, D, stream=st)

    def call():
        ana.process_dev(d_in, n, d_y, nf)
        syn.process_dev(d_y, nf, d_x, n)
    call()
    torch.cuda.synchronize()
    d = T * M
    sig = err = 0.0
    for a in (4 * d, n // 2, n - (1 << 16)):
        x = O.unpack_u8iq(d_in[2 * (a - d):2 * (a - d + (1 << 16))].cpu().numpy()).astype(np.complex128)
        xr = d_x[a:a + (1 << 16)].cpu().numpy()
        sig += float(np.sum(np.abs(x) ** 2))
        err += float(np.sum(np.abs(xr - x) ** 2))
    snr = 10 * np.log10(sig / err)
    if not snr > 60:
        raise SystemExit("round trip SNR %.1f dB" % snr)
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    ms = events_ms(torch, st, call, calls)
    gs = n / (ms * 1e-3) / 1e9
    rec = {"bench": "pfb_pfs_round_trip", "fmt": "u8iq", "n_samples": n, "M": M, "D": D, "taps": h.size,
           "calls": calls, "ms_per_call": round(ms, 4), "gsamples_per_s": round(gs, 2),
           "bytes_per_sample": 2 + 2 * 8.0 * M / D + 8, "snr_db_vs_delayed_input": round(snr, 1),
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
        raise SystemExit("bench_pfs: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power = card()
    big = 1 << 22 if args.quick else 1 << 28
    calls = max(20, args.calls)
    for M, D, cm, comp in [(1024, 512, False, True), (1024, 512, True, False), (1024, 1024, False, True),
                           (4096, 2048, False, True)]:
        bench_config(sdr, torch, dev, big, M, D, cm, calls, name, power, comp)
    bench_round_trip(sdr, torch, dev, big, calls, name, power)


if __name__ == "__main__":
    main()
