"""Adaptive equalizer bank (sdr_eq) throughput on one GPU: one JSON line per config.

For each config (C, N, adaptation): first a fresh handle's first call of 2048 symbols per channel is checked against
eq_ref.model (every y, e and the final taps of the first and last channel, bit for bit), so that a fast wrong answer
cannot be reported; then, on device-resident rows of QPSK through a 3-tap multipath channel (so that the taps adapt
rather than diverge; rows larger than the 126 MB L2 from C = 8 on, and by choice not at C = 1), three alternating rounds of 20 back-to-back
process_dev calls continuing the same stream, with, in the same run:
  - "fir": the fixed-tap FIR in torch (a grouped conv1d over re / im), the HBM price of the filter without adaptation;
  - "block_cma": the composition a user would write in torch, CMA with one averaged-gradient update per 64-symbol block
    (the gradient summed over the block, so that the step per symbol matches), timed on the same rows.
Each is timed with CUDA events; the best round counts.  Bytes are algorithmic: 24 per symbol (8 in, 8 y, 8 e), 16
without e.  "frac_hbm" is that traffic over the call time against 6552.3 GB/s, the HBM rate the rest of the project
quotes as measured peak; "cycles_per_symbol" is the call time at the card's max SM clock over the symbols of one channel
(channels run side by side).  The card's name, power limit and max SM clock are read in the same run.  Then the ISI of
the bank and of block CMA on the multipath workload of tests/test_eq_host.py (64 QPSK channels, CMA only), and last
the sdr_ddc -> sdr_tsync -> sdr_eq -> sdr_csync chain on 2^26 u8 IQ samples at C = 8, with the chain without sdr_eq
timed beside it for the equalizer's share.

    python scripts/bench_eq.py [--quick]
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

from bench_duc import card  # noqa: E402
from bench_pfb import PEAK_GBS, events_ms  # noqa: E402

CALLS = 20
BLOCK = 64
MU, RADIUS, EMAX = 5e-3, 1.0, 2.0


def multipath_qpsk(torch, dev, C_, S, seed):
    """QPSK through a 0.25 / 1 / 0.4 symbol-spaced channel with fixed phases, normalised, plus a little noise"""
    g = torch.Generator(device=dev).manual_seed(seed)
    k = torch.randint(0, 4, (C_, S), device=dev, generator=g)
    a = torch.polar(torch.ones(C_, S, device=dev), (math.pi / 4) * (2 * k + 1).float())
    h = [0.25 * complex(math.cos(0.7), math.sin(0.7)), 1.0, 0.4 * complex(math.cos(-1.1), math.sin(-1.1))]
    nrm = math.sqrt(sum(abs(v) ** 2 for v in h))
    x = (h[0] * torch.roll(a, -1, 1) + h[1] * a + h[2] * torch.roll(a, 1, 1)) / nrm
    noise = torch.randn((C_, S), dtype=torch.complex64, device=dev, generator=g)
    return (x + 0.03 * noise).to(torch.complex64)


def spot_check(sdr, torch, d_x, N, adapt, C_, st):
    """a fresh handle's first call of 2048 symbols per channel: channels 0 and C - 1 equal the model bit for bit"""
    import eq_ref as R
    n0 = min(2048, d_x.shape[1])
    b = sdr.Eq(N, adapt, n_channels=C_, stream=st)
    d_y = torch.empty((C_, n0), dtype=torch.complex64, device=d_x.device)
    d_e = torch.empty_like(d_y)
    b.process_dev(d_x, n0, d_x.shape[1], d_y, n0, d_e)
    torch.cuda.synchronize()
    for k in sorted({0, C_ - 1}):
        x = d_x[k:k + 1, :n0].cpu().numpy()
        y, e, w = R.model(x, N, adapt)
        ok = (np.array_equal(y[0].view(np.uint32), d_y[k].cpu().numpy().view(np.uint32))
              and np.array_equal(e[0].view(np.uint32), d_e[k].cpu().numpy().view(np.uint32))
              and np.array_equal(w[0].view(np.uint32), b.taps(k).view(np.uint32)))
        if not ok:
            raise SystemExit("sdr_eq differs from the model on channel %d of (C, N) = (%d, %d)" % (k, C_, N))
    b.close()


def fir_torch(torch, x, w):
    """y_s = sum_j w[j] x_{s-j} per channel: a grouped real conv1d over (re, im) with the taps flipped"""
    C_, N = w.shape
    xr = torch.view_as_real(x).permute(0, 2, 1).reshape(1, 2 * C_, -1)
    wf = torch.flip(w, dims=[1])
    k = torch.stack([torch.stack([wf.real, -wf.imag], 1), torch.stack([wf.imag, wf.real], 1)], 1)  # [C, 2, 2, N]
    y = torch.nn.functional.conv1d(torch.nn.functional.pad(xr, (N - 1, 0)), k.reshape(2 * C_, 2, N), groups=C_)
    return torch.view_as_complex(y.reshape(C_, 2, -1).permute(0, 2, 1).contiguous())


def block_cma(torch, x, w, mu=MU, R=RADIUS * RADIUS, B=BLOCK):
    """CMA with the gradient of each B-symbol block summed and applied once per block; returns (y, final w)"""
    C_, S = x.shape
    N = w.shape[1]
    xp = torch.nn.functional.pad(x, (N - 1, 0))
    w = w.clone()
    ys = []
    for b0 in range(0, S, B):
        nb = min(B, S - b0)
        xb = xp[:, b0:b0 + nb + N - 1].unfold(1, N, 1).flip(-1)  # [C, nb, N]: [..., j] = x_{s-j}
        y = (xb * w[:, None, :]).sum(-1)
        e = (y.real ** 2 + y.imag ** 2 - R) * y
        w = w - mu * (e[:, :, None] * xb.conj()).sum(1)
        ys.append(y)
    return torch.cat(ys, 1), w


def bench_config(sdr, torch, dev, C_, N, S, S_cma, name, power, clk):
    import eq_ref as R
    st = torch.cuda.current_stream(dev)
    adapt = (4, MU, RADIUS, EMAX, S_cma)
    d_x = multipath_qpsk(torch, dev, C_, S, 99 + C_ + N)
    spot_check(sdr, torch, d_x, N, adapt, C_, st)
    bank = sdr.Eq(N, adapt, n_channels=C_, stream=st)
    d_y = torch.empty_like(d_x)
    d_e = torch.empty_like(d_x)
    w0 = torch.from_numpy(np.tile(R.centre_spike(N), (C_, 1))).to(dev)
    out = {}

    def call():
        bank.process_dev(d_x, S, S, d_y, S, d_e)

    def fcall():
        out["f"] = fir_torch(torch, d_x, w0)

    def bcall():
        out["b"] = block_cma(torch, d_x, w0)
    for fn in (call, fcall, bcall):
        fn()
    torch.cuda.synchronize()
    # the torch FIR against the bank at mu = 0 (the same filter): a wrong comparison would not be a price
    fx = sdr.Eq(N, (4, 0.0, 1.0, 2.0, None), n_channels=C_, stream=st)
    d_f = torch.empty_like(d_x)
    fx.process_dev(d_x, S, S, d_f, S)
    torch.cuda.synchronize()
    ferr = float((out["f"] - d_f).abs().max())
    t_ms, f_ms, b_ms = [], [], []
    for _ in range(3):  # alternate in one run
        t_ms.append(events_ms(torch, st, call, CALLS))
        f_ms.append(events_ms(torch, st, fcall, CALLS))
        b_ms.append(events_ms(torch, st, bcall, 2))
    ms, fms, bms = min(t_ms), min(f_ms), min(b_ms)
    total = C_ * S
    rec = {"bench": "eq", "C": C_, "N": N, "adaptation": "CMA" if S_cma is None else "CMA->DD at %d" % S_cma,
           "symbols_per_channel": S, "calls": CALLS, "ms_per_call": round(ms, 4), "window_ms": round(ms * CALLS, 1),
           "gsymbols_per_s": round(total / (ms * 1e-3) / 1e9, 4),
           "cycles_per_symbol": round(ms * 1e-3 * clk * 1e6 / S, 1),
           "frac_hbm": round(24.0 * total / (PEAK_GBS * 1e9) / (ms * 1e-3), 4),
           "fir_torch": {"ms_per_call": round(fms, 4), "eq_over_fir": round(ms / fms, 2), "max_abs_diff": ferr},
           "block_cma_torch": {"ms_per_call": round(bms, 3), "eq_over_block_cma": round(ms / bms, 3)},
           "rounds_ms": [round(v, 4) for v in t_ms], "gpu": name, "power_limit": power, "max_sm_clock_mhz": clk}
    bank.close()
    fx.close()
    print(json.dumps(rec), flush=True)
    del d_x, d_y, d_e, d_f, out
    torch.cuda.empty_cache()
    return rec


def isi_on_workload(sdr, torch, dev, name, power):
    """residual ISI of the bank and of block CMA on the multipath workload (64 QPSK channels, CMA only)"""
    import eq_ref as R
    from test_eq_host import ESN0, NSYM, NTAPS
    x, h, _ = R.multipath_rows(4, 64, NSYM, ESN0, np.random.default_rng(104))
    eq = sdr.Eq(NTAPS, (4, MU, RADIUS, EMAX, None), n_channels=64)
    eq.process(x)
    isi_eq = np.array([R.isi_db(eq.taps(k), h[k]) for k in range(64)])
    w0 = torch.from_numpy(np.tile(R.centre_spike(NTAPS), (64, 1))).to(dev)
    _, wb = block_cma(torch, torch.from_numpy(x).to(dev), w0)
    wb = wb.cpu().numpy()
    isi_b = np.array([R.isi_db(wb[k], h[k]) if np.isfinite(wb[k]).all() else float("nan") for k in range(64)])
    rec = {"bench": "eq_isi", "M": 4, "channels": 64, "symbols": NSYM, "esn0_db": ESN0, "taps": NTAPS, "mu": MU,
           "block": BLOCK,
           "eq_isi_db_worst_median": [round(float(isi_eq.max()), 1), round(float(np.median(isi_eq)), 1)],
           "block_cma_isi_db_worst_median": [round(float(np.nanmax(isi_b)), 1), round(float(np.nanmedian(isi_b)), 1)],
           "block_cma_diverged": int(np.isnan(isi_b).sum()), "gpu": name, "power_limit": power}
    print(json.dumps(rec), flush=True)
    return rec


def bench_chain(sdr, torch, dev, n, name, power):
    """u8 IQ -> Ddc (C = 8, D = 8, L = 255, tensor path) -> Tsync at 4 frames per symbol (RRC, P = 32) -> Eq (CMA,
    N = 11) -> Csync QPSK designed for the equalizer's radius"""
    import gen
    import tsync_ref as TR
    C_, D, Ld, P = 8, 8, 255, 32
    hd = gen.lowpass_taps(Ld, 0.5 / D, 1.0).astype(np.float32)
    h, _ = TR.rrc_taps(4.0, P, 0.35, 8)
    freqs = np.linspace(-0.4, 0.4, C_)
    st = torch.cuda.current_stream(dev)
    g = torch.Generator(device=dev).manual_seed(7)
    d_in = torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    nf = n // D
    d_y = torch.empty((C_, nf), dtype=torch.complex64, device=dev)
    ana = sdr.Ddc(hd, freqs, 1.0, D, "u8iq", stream=st)
    tloop = sdr.tsync_loop_design(0.01, 0.707, TR.gardner_slope(0.35), 4.0) + (2.0, 0.01)
    ts = sdr.Tsync(h, P, 4 << 64, tloop, n_channels=C_, stream=st)
    eq = sdr.Eq(11, (4, MU, RADIUS, EMAX, None), n_channels=C_, stream=st)
    kp, ki = sdr.tsync_loop_design(0.01, 0.707, math.sqrt(2.0) * RADIUS, 1 / (2 * math.pi))
    cs = sdr.Csync((4, kp, ki, 2.0 * RADIUS, 0.01), n_channels=C_, stream=st)
    cap = int(ts.max_output(nf).max())
    d_s = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    d_q = torch.empty_like(d_s)
    d_z = torch.empty_like(d_s)
    out = {}

    def front():
        ana.reset()
        ts.reset()
        cs.reset()
        ana.process_dev(d_in, n, d_y, nf)
        out["got"] = ts.process_dev(d_y, nf, nf, d_s, cap, cap)

    def without():
        front()
        cs.process_dev(d_s, out["got"], cap, d_z, cap)

    def call():
        front()
        eq.reset()
        eq.process_dev(d_s, out["got"], cap, d_q, cap)
        cs.process_dev(d_q, out["got"], cap, d_z, cap)
    call()
    torch.cuda.synchronize()
    c_ms, w_ms = [], []
    for _ in range(2):
        c_ms.append(events_ms(torch, st, call, 2))
        w_ms.append(events_ms(torch, st, without, 2))
    ms, wms = min(c_ms), min(w_ms)
    rec = {"bench": "ddc_tsync_eq_csync_chain", "fmt": "u8iq", "n_samples": n, "C": C_, "D": D, "taps": Ld,
           "eq_taps": 11, "symbols_per_channel": int(out["got"].min()), "ms_per_call": round(ms, 3),
           "ms_without_eq": round(wms, 3), "eq_share": round((ms - wms) / ms, 4),
           "gsamples_per_s_in": round(n / (ms * 1e-3) / 1e9, 3), "gpu": name, "power_limit": power}
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="fewer symbols per config (a rehearsal, not a measurement)")
    args = ap.parse_args()
    import torch
    import sdr_b200 as sdr
    if not torch.cuda.is_available() or sdr.device_count() < 1:
        raise SystemExit("bench_eq: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    # (C, N, symbols per channel, CMA symbols): C * S * 8 bytes of input exceed the 126 MB L2 from C = 8 on.  The one
    # channel at C = 1 is a 0.5 MB row by choice: a row past L2 would be 2^24 symbols, about 5 s per call at the
    # measured ~590 cycles per symbol, and a chain that reads 8 bytes every ~300 ns is not bound by where they sit
    configs = [(1, 11, 1 << 16, None), (8, 11, 1 << 21, None), (1024, 11, 1 << 15, 1 << 14),
               (1024, 32, 1 << 15, None), (1024, 64, 1 << 15, None), (16384, 7, 1 << 13, None),
               (65536, 4, 1 << 11, None)]
    for C_, N, S, Sc in configs:
        bench_config(sdr, torch, dev, C_, N, S >> (3 if args.quick else 0), Sc, name, power, clk)
    isi_on_workload(sdr, torch, dev, name, power)
    bench_chain(sdr, torch, dev, 1 << (22 if args.quick else 26), name, power)


if __name__ == "__main__":
    main()
