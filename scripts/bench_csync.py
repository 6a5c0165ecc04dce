"""Carrier recovery bank (sdr_csync) throughput on one GPU: one JSON line per config.

For each config (C, M, outputs): check a fresh handle's first call (the first 8192 phases of the first and last channel
against the integer recurrence replayed from the reported errors, and symbols near the start and end of those rows
against x e^{-2 pi i phi / 2^64} in f64 at their exact phases) so that a fast wrong answer cannot be reported; then
alternate, three rounds, 20 back-to-back process_dev calls on device-resident torch.randn rows with, in the same run:
  - "open_loop": x * exp(-2 pi i (phi_0 + s nu_0)) in torch, the HBM-bound price of a derotation without a loop;
  - "vv": the feedforward estimator a user composes in torch, Viterbi & Viterbi: x^M, a moving average of 64 symbols,
    angle / M, unwrapped by a cumulative sum of rounded differences, and the derotation.
Each is timed with CUDA events; the best round counts.  Bytes are algorithmic: 28 per symbol (8 in, 8 out, 8 phase,
4 error), 16 with phase and err not written.  "frac_hbm" is that traffic over the call time against 6552.3 GB/s, the
HBM rate the rest of the project quotes as measured peak; "cycles_per_symbol" is the call time at the card's max SM
clock over the symbols of one channel (channels run side by side, one lane each).  The card's name, power limit and
max SM clock are read in the same run.  Then the EVM of sdr_csync and of Viterbi & Viterbi on the tracking workload of
tests/test_csync_host.py (64 QPSK channels, offsets 0, +-1e-4, +-2e-3 turn per symbol, Es/N0 = 30 dB), and last the
sdr_ddc -> sdr_tsync -> sdr_csync chain on 2^26 u8 IQ samples at C = 8, with the chain without sdr_csync timed beside
it for csync's share.

    python scripts/bench_csync.py [--quick]
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
VV_WINDOW = 64


def loop_for(sdr, M, A=1.0):
    kd = {2: 1.0, 4: math.sqrt(2.0), 8: 1.0 / math.cos(math.pi / 8)}[M] * A
    kp, ki = sdr.tsync_loop_design(0.01, 0.707, kd, 1 / (2 * math.pi))
    return (M, kp, ki, 2.0 * A, 0.01)


def spot_check(d_x, d_z, d_p, d_e, loop, phi0, nu0):
    import csync_ref as R
    worst = 0.0
    C_, S = d_x.shape
    for k in sorted({0, C_ - 1}):
        n8 = min(S, 8192)
        ph = d_p[k, :n8].cpu().numpy().view(np.uint64)
        R.replay(ph[None], d_e[k, :n8].cpu().numpy()[None], [n8], loop, phi0[k], nu0[k])
        for s0 in (0, n8 - 512):
            x = d_x[k, s0:s0 + 512].cpu().numpy()
            want = R.rotate(x, ph[s0:s0 + 512])
            z = d_z[k, s0:s0 + 512].cpu().numpy()
            worst = max(worst, float((np.abs(z - want) / np.abs(x)).max()))
    if not worst <= 1e-6:
        raise SystemExit("spot symbols differ from f64 truth: %.3g of |x| > 1e-6" % worst)
    return worst


def open_loop(torch, x, f0, fr):
    """x e^{-2 pi i (phi_0 + s nu_0)}: phases in turns from the exact integers, f64 then f32"""
    s = torch.arange(x.shape[1], device=x.device, dtype=torch.float64)
    t = torch.frac(f0[:, None] + s[None, :] * fr[:, None]).float()
    return x * torch.polar(torch.ones_like(t), -2 * math.pi * t)


def viterbi_viterbi(torch, x, M, W=VV_WINDOW):
    """feedforward M-th power estimator: moving average of x^M over W symbols, angle / M, unwrapped, derotation"""
    y = x
    for _ in range(M - 1):
        y = y * x
    c = torch.cumsum(torch.nn.functional.pad(y, (1, 0)), dim=1)
    avg = c[:, W:] - c[:, :-W]
    avg = torch.cat([c[:, 1:W], avg], dim=1)
    th = torch.angle(-avg if M > 2 else avg) / M  # x^M = -|x|^M on the points e^{i pi (2k + 1) / M}, M > 2
    step = 2 * math.pi / M
    d = torch.diff(th, dim=1, prepend=th[:, :1])
    th = th - step * torch.cumsum(torch.round(d / step), dim=1)
    return x * torch.polar(torch.ones_like(th), -th)


def bench_config(sdr, torch, dev, C_, M, S, write_all, name, power, clk):
    st = torch.cuda.current_stream(dev)
    loop = loop_for(sdr, M)
    rng = np.random.default_rng(C_ + M)
    phi0 = [int(v) for v in rng.integers(0, 1 << 63, C_, dtype=np.int64)]
    nu0 = [int(v) for v in rng.integers(-(1 << 20), 1 << 20, C_)]
    g = torch.Generator(device=dev).manual_seed(99 + C_ + M)
    d_x = torch.randn((C_, S), dtype=torch.complex64, device=dev, generator=g)
    bank = sdr.Csync(loop, n_channels=C_, phase=phi0, freq=nu0, stream=st)
    d_z = torch.empty_like(d_x)
    d_p = torch.empty((C_, S), dtype=torch.int64, device=dev)
    d_e = torch.empty((C_, S), dtype=torch.float32, device=dev)
    bank.process_dev(d_x, S, S, d_z, S, d_p, d_e)
    torch.cuda.synchronize()
    err = spot_check(d_x, d_z, d_p, d_e, loop, phi0, nu0)
    pa, ea = (d_p, d_e) if write_all else (None, None)

    def call():
        bank.reset()
        bank.process_dev(d_x, S, S, d_z, S, pa, ea)
    f0 = torch.tensor([p * 2.0 ** -64 for p in phi0], dtype=torch.float64, device=dev)
    fr = torch.tensor([v * 2.0 ** -40 for v in nu0], dtype=torch.float64, device=dev)
    out = {}

    def ocall():
        out["o"] = open_loop(torch, d_x, f0, fr)

    def vcall():
        out["v"] = viterbi_viterbi(torch, d_x, M)
    for fn in (call, ocall, vcall):
        fn()
    torch.cuda.synchronize()
    t_ms, o_ms, v_ms = [], [], []
    for _ in range(3):  # alternate in one run
        t_ms.append(events_ms(torch, st, call, CALLS))
        o_ms.append(events_ms(torch, st, ocall, CALLS))
        v_ms.append(events_ms(torch, st, vcall, CALLS))
    ms, oms, vms = min(t_ms), min(o_ms), min(v_ms)
    total = C_ * S
    per_sym = 28.0 if write_all else 16.0
    rec = {"bench": "csync", "C": C_, "M": M, "symbols_per_channel": S, "phase_err_written": write_all,
           "calls": CALLS, "spot_err_rel": err, "ms_per_call": round(ms, 4), "window_ms": round(ms * CALLS, 1),
           "gsymbols_per_s": round(total / (ms * 1e-3) / 1e9, 3),
           "cycles_per_symbol": round(ms * 1e-3 * clk * 1e6 / S, 1),
           "frac_hbm": round(per_sym * total / (PEAK_GBS * 1e9) / (ms * 1e-3), 4),
           "open_loop_torch": {"ms_per_call": round(oms, 4), "csync_over_open_loop": round(ms / oms, 2)},
           "vv_torch": {"ms_per_call": round(vms, 4), "csync_over_vv": round(ms / vms, 2)},
           "rounds_ms": [round(v, 4) for v in t_ms], "gpu": name, "power_limit": power, "max_sm_clock_mhz": clk}
    bank.close()
    print(json.dumps(rec), flush=True)
    del d_x, d_z, d_p, d_e, out
    torch.cuda.empty_cache()
    return rec


def evm_on_tracking_workload(sdr, torch, dev, name, power):
    """EVM after a real gain fit against nearest-point decisions, sdr_csync against Viterbi & Viterbi"""
    import csync_ref as R
    from test_csync_host import ACQ, ESN0, N, OFFSETS
    offs = [OFFSETS[k % 5] for k in range(64)]
    x, theta, _ = R.psk_rows(4, offs, N, ESN0, np.random.default_rng(104))
    z, ph, err = sdr.Csync(loop_for(sdr, 4), n_channels=64).process(x)
    z = np.array(z)
    vv = viterbi_viterbi(torch, torch.from_numpy(x).to(dev), 4).cpu().numpy()

    def evm(y):
        y = y[:, ACQ:].astype(np.complex128)
        pts = R.points(4)
        dec = pts[np.abs(y[:, :, None] / np.abs(y).mean(axis=1)[:, None, None] - pts).argmin(axis=2)]
        g = (np.conj(y) * dec).real.sum(axis=1) / (np.abs(y) ** 2).sum(axis=1)
        return np.sqrt((np.abs(g[:, None] * y - dec) ** 2).mean(axis=1))
    e_c, e_v = evm(z), evm(vv)
    by = {}
    for f in OFFSETS:
        idx = [k for k in range(64) if offs[k] == f]
        by[str(f)] = {"csync": round(float(e_c[idx].max()), 4), "vv": round(float(e_v[idx].max()), 4)}
    rec = {"bench": "csync_evm", "M": 4, "channels": 64, "symbols": N, "skip": ACQ, "esn0_db": ESN0,
           "vv_window": VV_WINDOW, "worst_evm_by_offset": by, "gpu": name, "power_limit": power}
    print(json.dumps(rec), flush=True)
    return rec


def bench_chain(sdr, torch, dev, n, name, power):
    """u8 IQ -> Ddc (C = 8, D = 8, L = 255, tensor path) -> Tsync at 4 frames per symbol (RRC, P = 32) -> Csync QPSK"""
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
    cs = sdr.Csync(loop_for(sdr, 4), n_channels=C_, stream=st)
    cap = int(ts.max_output(nf).max())
    d_s = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    d_z = torch.empty_like(d_s)
    out = {}

    def front():
        ana.reset()
        ts.reset()
        ana.process_dev(d_in, n, d_y, nf)
        out["got"] = ts.process_dev(d_y, nf, nf, d_s, cap, cap)

    def call():
        front()
        cs.reset()
        cs.process_dev(d_s, out["got"], cap, d_z, cap)
    call()
    torch.cuda.synchronize()
    assert np.isfinite(d_z[:, 1000:5096].cpu().numpy()).all()
    c_ms, f_ms = [], []
    for _ in range(2):
        c_ms.append(events_ms(torch, st, call, 2))
        f_ms.append(events_ms(torch, st, front, 2))
    ms, fms = min(c_ms), min(f_ms)
    rec = {"bench": "ddc_tsync_csync_chain", "fmt": "u8iq", "n_samples": n, "C": C_, "D": D, "taps": Ld,
           "symbols_per_channel": int(out["got"].min()), "ms_per_call": round(ms, 3),
           "ms_without_csync": round(fms, 3), "csync_share": round((ms - fms) / ms, 4),
           "gsamples_per_s_in": round(n / (ms * 1e-3) / 1e9, 2), "gpu": name, "power_limit": power}
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="fewer symbols per config (a rehearsal, not a measurement)")
    args = ap.parse_args()
    import torch
    import sdr_b200 as sdr
    if not torch.cuda.is_available() or sdr.device_count() < 1:
        raise SystemExit("bench_csync: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    # (C, M, symbols per channel, phase and err written): C * S * 8 bytes of input exceed the 126 MB L2 from C = 8 on
    configs = [(1, 4, 1 << 17, True), (8, 4, 1 << 22, True), (1024, 4, 1 << 17, True), (1024, 2, 1 << 17, True),
               (1024, 8, 1 << 17, True), (1024, 4, 1 << 17, False), (16384, 4, 1 << 16, True),
               (65536, 4, 1 << 14, True)]
    for C_, M, S, w in configs:
        bench_config(sdr, torch, dev, C_, M, S >> (4 if args.quick else 0), w, name, power, clk)
    evm_on_tracking_workload(sdr, torch, dev, name, power)
    bench_chain(sdr, torch, dev, 1 << (22 if args.quick else 26), name, power)


if __name__ == "__main__":
    main()
