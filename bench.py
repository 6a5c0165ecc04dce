#!/usr/bin/env python
"""bench.py -- headline benchmark of the sample-stream hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--configs all|none]
                    [--dump-outputs DIR]

Headline (`value`, `roofline`, `e2e`, `cpu_baseline`) = BASELINE.json configs[1]: batched 1024-point FFT spectrum of
rtl_tcp-format u8 IQ, 2^28 samples per GPU (fused unpack on load, fftshift + 1/sqrt(N) on store).  A "step" is one
pass of the kernel over the whole 2^28-sample batch (512 MiB in, 2 GiB out: larger than the 126 MB L2, so every step
streams from HBM).  With N > 1 (torchrun) every rank owns its own batch: no data-path collective, scaling = weak,
value = all ranks' samples / max-over-ranks device time.

The same JSON line carries `configs`: the other four BASELINE configs measured the same way (CUDA events on the
launching stream, barrier on both sides, max over ranks), each with its own roofline fraction -- C1 (64-tap FIR, real
and complex taps) and C3's FIR stage as ONE contiguous 2^26*N-sample stream cut across the ranks with tap-length halos
(`shard.sample_range`), C4 as 1024 channels / N (`shard.unit_range`), C5 (N = 256 ... 65536, 1 GiB of c64 per GPU) and
C3's whole device-resident chain as independent batches.  For N > 1 the halo- and channel-split outputs are gathered
(off the timed path) and compared bit for bit with rank 0's single-GPU run of the whole stream / all channels
(`parity`).

Prints ONE JSON line on rank 0.

--dump-outputs DIR writes what the headline workload's last timed step computed (rank 0's outputs) as DIR/<name>.npy,
so that two builds run with the same arguments can be compared output for output: the inputs come from fixed seeds,
and a stateful workload (FIR history, PLL, resampler) is reset before the timed steps, so its last step depends on
--steps alone.  See dump_outputs for the format and the sampling of large outputs.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "unnamed-rust-sdr_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the `ncu --set full` captures
# summarised under profiles/ (same command line as the bench, one launch).  null = not captured for that workload.
NCU_TRAFFIC = {
    "c2_fft1024_u8iq_2p28": (2.6255e9, "profiles/r01f_ncu_fft1024_u8.txt"),
    "fir64_d1_u8iq_2p26": (6.124e8, "profiles/r01_prof_fir_umma_c1_v2.txt"),
    "fir255_d1_u8iq_2p26": (6.122e8, "profiles/r01_prof_fir_umma_k255_v2.txt"),
    "c5_fft65536_c64_2p27": (2.102e9, "profiles/r01_prof_fft_l2_64k_v1.txt"),
    "fir255_d10_u8iq_2p26": (1.624e8, "profiles/r01_prof_fir_umma_c3_v1.txt"),
}
try:  # later rounds add their captures without touching this file
    NCU_TRAFFIC.update({k: tuple(v) for k, v in json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).items()})
except Exception:
    pass

SEED = 0x5D12B200
FIR_C64 = {"fir255_c64": (255, 0), "fir64_c64": (64, 0), "fir255_c64_split2": (255, 16), "fir64_c64_split2": (64, 16),
           "fir255_c64_cuda": (255, 2), "fir64_c64_cuda": (64, 2)}
DUMP_BYTES = 60 << 20  # all --dump-outputs files together, .npy headers included, stay under 64 MB
DUMP_ROW = 4096        # a 1-D output stream is sampled in blocks of this many samples


def sample_rows(n_rows, k):
    """the fixed, seeded choice of k of n_rows rows that --dump-outputs writes, in row order"""
    return np.sort(np.random.default_rng(SEED).choice(n_rows, k, replace=False))


def dump_outputs(torch, outputs, directory):
    """Writes every {name: tensor} of `outputs` as directory/<name>.npy in float32: complex values get a trailing
    (re, im) axis, integer flags become 0.0 / 1.0.  An output larger than its share of DUMP_BYTES is cut into rows (its
    first axis; a 1-D stream into blocks of DUMP_ROW samples, dropping the tail that fills no block) and only the rows
    chosen by sample_rows are written."""
    os.makedirs(directory, exist_ok=True)
    share = DUMP_BYTES // len(outputs)
    for name, t in outputs.items():
        elem_bytes = 8 if t.is_complex() else 4
        if t.numel() * elem_bytes > share:
            if t.dim() == 1:
                t = t[:t.numel() // DUMP_ROW * DUMP_ROW].view(-1, DUMP_ROW)
            rows = sample_rows(t.shape[0], max(1, share // (t[0].numel() * elem_bytes)))
            t = t.index_select(0, torch.from_numpy(rows).to(t.device))
        t = torch.view_as_real(t.contiguous()) if t.is_complex() else t.float()
        np.save(os.path.join(directory, name + ".npy"), t.cpu().numpy())


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons while the timed region runs"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.stop = threading.Event()
        self.th = None

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [c.strip() for c in out.strip().split(",")]
                if len(f) >= 7:
                    self.rows.append(f)
            except Exception:
                pass
            self.stop.wait(0.1)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"], "samples": 0}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]),
                "power_w_max": max(float(r[2]) for r in self.rows), "reasons": reasons, "samples": len(self.rows)}


# ---------------------------------------------------------------------------------------------------
# workload descriptions shared by both arms (`config` must be identical in the repo arm and the reference arm)
# ---------------------------------------------------------------------------------------------------
def c2_name(log2_samples=28):
    return "c2_fft1024_u8iq_2p%d" % log2_samples


def config_dict(name):
    """the `config` object of the JSON line: a function of the workload name only, so that `--impl reference`
    prints the identical object"""
    table = {
        "c2": (c2_name(28), "batched 1024-pt FFT of u8 IQ, fused unpack + fftshift + 1/sqrt(N), 262144 transforms", 1 << 28),
        "c2_small": (c2_name(24), "batched 1024-pt FFT of u8 IQ, fused unpack + fftshift + 1/sqrt(N), 16384 transforms", 1 << 24),
        "c1": ("fir64_d1_u8iq_2p26", "fused u8-IQ unpack + 64-tap real FIR, decimation 1", 1 << 26),
        "c1c": ("fir64c_d1_u8iq_2p26", "fused u8-IQ unpack + 64-tap complex FIR, decimation 1", 1 << 26),
        "c3": ("fir255_d10_u8iq_2p26", "fused u8-IQ unpack + 255-tap real FIR, decimation 10", 1 << 26),
        "fir255_u8": ("fir255_d1_u8iq_2p26", "fused u8-IQ unpack + 255-tap real FIR, decimation 1", 1 << 26),
        "c3_2p28": ("fir255_d10_u8iq_2p28", "fused u8-IQ unpack + 255-tap real FIR, decimation 10", 1 << 28),
        "c3chain": ("c3_chain_fir255_d10_sincbest_2p26", "u8 IQ -> 255-tap FIR /10 -> SampleRate x0.2 (sincbest), device resident", 1 << 26),
        "c4": ("c4_channelizer_128ch_2p16", "128 channels x (255-tap FIR + PLL)", 128 << 16),
        "c4_1024": ("c4_channelizer_1024ch_2p16", "1024 channels x (255-tap FIR + PLL), channels split over the GPUs", 1024 << 16),
    }
    alias = {"default": "c2", "fft1024_u8": "c2", "fir64_u8": "c1", "fir255_d10_u8": "c3"}
    key = alias.get(name, name)
    if key in FIR_C64:
        K, flags = FIR_C64[key]
        how = {0: "tcgen05, 3 bf16 terms", 16: "tcgen05, 2 bf16 terms", 2: "CUDA cores"}[flags]
        table[key] = ("%s_1024ch_2p16" % key, "1024 c64 channel streams x %d real taps (%s)" % (K, how), 1024 << 16)
    if key.startswith("c5_"):
        n = 1 << int(key[3:])
        wname, desc, units = "c5_fft%d_c64_2p27" % n, "batched %d-pt c64 FFT, %d transforms" % (n, (1 << 27) // n), 1 << 27
    elif key in table:
        wname, desc, units = table[key]
    else:
        wname, desc, units = key, key, None
    return {"workload": wname, "desc": desc, "samples_per_gpu_per_step": units,
            "l2": "inputs+outputs per step exceed the 126 MB L2 (streamed from HBM every step)",
            "parallelism": "independent shards per GPU, no data-path collective"}


# ---------------------------------------------------------------------------------------------------
# CPU legs: the oracle port of the reference path on the host cores (bench.py's `cpu_baseline` / `--impl reference`
# are the only places outside tests/ that may execute oracle/).  Each returns seconds for `units` samples.
# ---------------------------------------------------------------------------------------------------
_CPU_INPUT = {}


def _cpu_u8(units, seed=5):
    key = ("u8", units)
    if key not in _CPU_INPUT:  # generated once, outside the timed region
        _CPU_INPUT.clear()
        _CPU_INPUT[key] = np.random.default_rng(seed).integers(0, 256, 2 * units, dtype=np.uint8)
    return _CPU_INPUT[key]


def _cpu_fft_u8(units, threads):
    import oracle_lib as O
    iq = _cpu_u8(units)
    t0 = time.perf_counter()
    O.fft_batch_u8(iq, 1024, threads)
    return time.perf_counter() - t0


def _taps(K, complex_taps=False):
    import gen
    fs = 2.048e6 if K == 64 else 2.4e6
    if complex_taps:
        return gen.complex_bandpass_taps(K, 200e3, 100e3, fs)
    return gen.lowpass_taps(K, 200e3 if K == 64 else 100e3, fs)


def _cpu_fir_u8(K, D, complex_taps):
    def run(units, threads):
        import oracle_lib as O
        iq = _cpu_u8(units)
        taps = _taps(K, complex_taps)
        t0 = time.perf_counter()
        O.fir_u8_mt(iq, taps, D, threads)
        return time.perf_counter() - t0
    return run


def _cpu_fft_c64(n):
    def run(units, threads):
        import oracle_lib as O
        import gen
        xs = gen.complex_noise(units, 3)
        t0 = time.perf_counter()
        O.fft_batch_c64(xs, n, False, threads)
        return time.perf_counter() - t0
    return run


def _cpu_channelizer(units, threads):
    import oracle_lib as O
    import gen
    c = max(1, threads)
    m = max(1024, units // c)
    xs = gen.complex_noise(c * m, 3).reshape(c, m)
    od = O.pll_design(0.0, 0.035, (O.BQ_LOWPASS, 80000.0, 0.7), (O.BQ_LOWPASS, 20000.0, 0.7), (O.BQ_LOWPASS, 20000.0, 0.7))
    taps = gen.lowpass_taps(255, 100e3, 1.8e6)
    t0 = time.perf_counter()
    O.channelizer_mt(xs, taps, od, 1.8e6, threads)
    return time.perf_counter() - t0


def _cpu_fm(units, threads):
    import oracle_lib as O
    import gen
    x = gen.complex_noise(max(4096, units), 3)
    p = O.Pll(O.pll_design(0.0, 0.035, (O.BQ_LOWPASS, 80000.0, 0.7), (O.BQ_IDENTITY, 0.0, 0.0),
                           (O.BQ_LOWPASS, 20000.0, 0.7)), 1.8e6)
    t0 = time.perf_counter()
    p.apply(x)  # the demodulator PLL alone: > 90 % of the chain's CPU time, one thread (the loop is sequential)
    return time.perf_counter() - t0


def cpu_leg(name):
    """(function(units, threads) -> seconds, bounded sample size in samples) for a workload name"""
    alias = {"default": "c2", "fft1024_u8": "c2", "fir64_u8": "c1", "fir255_d10_u8": "c3"}
    key = alias.get(name, name)
    if key in ("c2", "c2_small"):
        return _cpu_fft_u8, 1 << 28
    if key == "c1":
        return _cpu_fir_u8(64, 1, False), 1 << 24
    if key == "c1c":
        return _cpu_fir_u8(64, 1, True), 1 << 24
    if key in ("c3", "c3_2p28", "c3chain", "c3chain_linear", "c3chain_fastest"):
        return _cpu_fir_u8(255, 10, False), 1 << 24
    if key == "fir255_u8":
        return _cpu_fir_u8(255, 1, False), 1 << 24
    if key.startswith("c5_"):
        return _cpu_fft_c64(1 << int(key[3:])), 1 << 26
    if key.startswith("c4") or key in FIR_C64:
        return _cpu_channelizer, 1 << 19
    if key.startswith("fm"):
        return _cpu_fm, 1 << 19
    raise SystemExit("unknown workload " + name)


def numpy_fft_line(threads):
    """SURVEY 8(d): an honest optimised CPU line beside the port -- pocketfft (numpy, one thread; scipy, all threads)
    on the same workload: unpack (b - 128) / 128 and 1024-point transforms of c64 blocks, fftshift, 1/sqrt(N)."""
    units = 1 << 24
    iq = _cpu_u8(1 << 28)[:2 * units]

    def run(fft):
        t0 = time.perf_counter()
        x = ((iq.astype(np.float32) - np.float32(128.0)) / np.float32(128.0)).view(np.complex64).reshape(-1, 1024)
        X = fft(x)
        np.fft.fftshift(X, axes=1) * np.float32(1.0 / 32.0)
        return time.perf_counter() - t0
    out = {"sample": "%d samples of the same workload" % units}
    try:
        run(lambda x: np.fft.fft(x, axis=1)[:16])
        out["numpy_fft_1thread"] = units / run(lambda x: np.fft.fft(x, axis=1)) / 1e9
    except Exception as e:  # pragma: no cover
        out["numpy_fft_1thread"] = None
        out["error"] = repr(e)
    try:
        import scipy.fft as sf
        out["scipy_fft_all_threads"] = units / run(lambda x: sf.fft(x, axis=1, workers=threads)) / 1e9
        out["threads"] = threads
    except Exception:
        out["scipy_fft_all_threads"] = None
    out["unit"] = "Gsamples/s"
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path, all host threads.  The Rust crate
    cannot be built in this image (no cargo/rustc), so this is the oracle port: the f32-faithful C++ restatement
    of the reference's per-sample structure, re-planning the FFT on every call as src/fft.rs:10-11 does."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_lib as O
    threads = O.hardware_threads()
    fn, units = cpu_leg(args.workload)
    cfg = config_dict(args.workload)
    for _ in range(args.warmup):
        fn(max(units // 8, 1 << 16), threads)
    t = 0.0
    for _ in range(args.steps):
        t += fn(units, threads)
    value = units * args.steps / t / 1e9
    line = {
        "impl": "reference", "metric": "FIR/FFT Gsamples/s", "value": value, "unit": "Gsamples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": "Gsamples/s", "cores": threads, "kind": "port",
                         "sample": "%d samples of the same workload per step; CPU oracle port of the reference path "
                                   "(per-sample structure and f32 operation order of the Rust source, FFT re-planned per "
                                   "call as fft.rs:10-11 does), std::thread over independent blocks / ranges" % units},
        "e2e": {"value": value, "unit": "Gsamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# GPU side
# ---------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, torch, sdr, dev, dist, rank, world, stream):
        self.torch, self.sdr, self.dev, self.dist, self.rank, self.world, self.stream = torch, sdr, dev, dist, rank, world, stream

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, v):
        if self.dist is None:
            return float(v)
        t = self.torch.tensor([float(v)], device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t)

    def time_steps(self, step, steps, warmup):
        """W untimed steps, then K steps between CUDA events on the launching stream, barrier + synchronize on
        both sides, MAX over ranks.  Returns (ms per step, launches of this library's kernels in the timed region)."""
        torch = self.torch
        for _ in range(warmup):
            step()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        l0 = self.sdr.kernel_launch_count()
        ev0.record()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        self.host_ms_per_step = (time.perf_counter() - t0) * 1e3 / steps  # enqueue time only (nothing synchronises in a step)
        ev1.record()
        self.barrier()
        launches = self.sdr.kernel_launch_count() - l0
        return self.max_over_ranks(ev0.elapsed_time(ev1)) / steps, int(launches)

    def randint_u8(self, n_bytes, seed):
        g = self.torch.Generator(device=self.dev).manual_seed(seed)
        return self.torch.randint(0, 256, (n_bytes,), dtype=self.torch.uint8, device=self.dev, generator=g)

    def gather_rows(self, t):
        """every rank's 1-D tensor (lengths may differ) -> list of per-rank tensors on every rank (off the timed path)"""
        torch, dist = self.torch, self.dist
        n = torch.tensor([t.numel()], device=self.dev, dtype=torch.int64)
        lens = [torch.zeros_like(n) for _ in range(self.world)]
        dist.all_gather(lens, n)
        lens = [int(v) for v in lens]
        m = max(lens)
        pad = torch.zeros(m, dtype=t.dtype, device=self.dev)
        pad[:t.numel()] = t
        out = torch.empty(self.world * m, dtype=t.dtype, device=self.dev)
        dist.all_gather_into_tensor(out, pad)
        return [out[r * m:r * m + lens[r]] for r in range(self.world)]


def wl_fft1024_u8(cx, log2_samples=28):
    torch, sdr, dev = cx.torch, cx.sdr, cx.dev
    n = 1024
    samples = 1 << log2_samples
    batches = samples // n
    raw = cx.randint_u8(2 * samples, SEED + 2)
    out = torch.empty((batches, n), dtype=torch.complex64, device=dev)
    plan = sdr.FftPlan(n, "u8iq", shift=True, norm=True, device=dev.index, stream=cx.stream)

    def step():
        plan.exec_dev(raw, batches, out)

    host = {}

    def e2e_setup():
        host["in"] = torch.empty(2 * samples, dtype=torch.uint8).pin_memory()
        host["in"].copy_(raw)
        host["out"] = torch.empty((batches, n), dtype=torch.complex64).pin_memory()
        host["plan"] = sdr.FftPlan(n, "u8iq", shift=True, norm=True, device=dev.index)

    def e2e_step():
        sdr.lib().sdr_fft_exec(host["plan"].h, host["in"].data_ptr(), batches, host["out"].data_ptr())
        return float(host["out"][batches - 1, 0].real)

    return dict(key="c2" if log2_samples == 28 else "c2_small", units=samples, bytes_per_unit=10.0, step=step,
                e2e_setup=e2e_setup, e2e_step=e2e_step, host=host, h2d=2 * samples, d2h=8 * samples,
                dtype="f32", kernel="fft1024_warp_kernel<u8iq>", outputs=lambda: {"spectrum": out})


def wl_fir_u8(cx, key, K=64, D=1, log2_samples=26, complex_taps=False):
    """One contiguous stream of world * 2^log2_samples samples cut across the ranks on multiples of D with a tap-length
    halo (SURVEY 8e row 1/2); at world == 1 this is the plain single-stream run."""
    torch, sdr, dev = cx.torch, cx.sdr, cx.dev
    per_gpu = 1 << log2_samples
    total = per_gpu * cx.world
    taps = _taps(K, complex_taps)
    raw = cx.randint_u8(2 * total, SEED + 1)           # the same stream on every rank (same seed, same generator)
    halo = -(-(K - 1) // D) * D                        # K-1 rounded up to a multiple of D: the phase stays 0 at `lo`
    lo, hi, hlo = sdr.shard.sample_range(total, cx.world, cx.rank, halo, D)
    mine = raw[2 * lo:2 * hi]
    n = hi - lo
    n_out = n // D + 1  # the decimation phase carries over between steps
    out = torch.empty(n_out, dtype=torch.complex64, device=dev)
    fir = sdr.Fir(taps, "u8iq", decimation=D, device=dev.index, stream=cx.stream)
    last = {}

    def step():
        last["n"] = fir.process_dev(mine, n, out, n_out)

    def parity():
        if cx.world == 1:
            return None
        fir.reset()
        if lo > hlo:
            fir.process_dev(raw[2 * hlo:2 * lo], lo - hlo, out, n_out)   # prime the history with the halo
        got = fir.process_dev(mine, n, out, n_out)
        parts = cx.gather_rows(torch.view_as_real(out[:got]).reshape(-1).view(torch.int32))
        ok = True
        if cx.rank == 0:
            whole = torch.empty(total // D + 1, dtype=torch.complex64, device=dev)
            f0 = sdr.Fir(taps, "u8iq", decimation=D, device=dev.index, stream=cx.stream)
            g0 = f0.process_dev(raw, total, whole, whole.numel())
            cat = torch.cat(parts)
            ref = torch.view_as_real(whole[:g0]).reshape(-1).view(torch.int32)
            ok = bool(cat.numel() == ref.numel() and torch.equal(cat, ref))
            f0.close()
        return ok

    host = {}

    def e2e_setup():
        host["in"] = torch.empty(2 * n, dtype=torch.uint8).pin_memory()
        host["in"].copy_(mine)
        host["out"] = torch.empty(n_out, dtype=torch.complex64).pin_memory()
        host["fir"] = sdr.Fir(taps, "u8iq", decimation=D, device=dev.index)

    def e2e_step():
        import ctypes as C
        a, b = C.c_size_t(0), C.c_size_t(0)
        sdr.lib().sdr_fir_process(host["fir"].h, host["in"].data_ptr(), n, n, host["out"].data_ptr(),
                                  n_out, n_out, C.byref(a), C.byref(b))
        return float(host["out"][max(b.value, 1) - 1].real)

    return dict(key=key, units=n, bytes_per_unit=2.0 + 8.0 / D, step=step, e2e_setup=e2e_setup, e2e_step=e2e_step,
                host=host, h2d=2 * n, d2h=8 * n_out, dtype="u8 x s8 -> s32 (tcgen05 kind::i8), f32 out",
                kernel="fir_umma_kernel (tcgen05/TMEM)", parity=parity,
                sharding="one %d-sample stream, contiguous ranges with a %d-sample halo" % (total, halo),
                outputs=lambda: {"filtered": out[:last["n"]]}, reset=fir.reset)


def wl_c3_chain(cx, key="c3chain", log2_samples=26, converter=0):
    """C3 end to end on the device: u8 IQ -> 255-tap FIR, Decimate 10 (2.4 MS/s -> 240 kS/s) -> SampleRate x0.2
    (-> 48 kS/s, converter 0 = SincBestQuality, the reference's default) with every intermediate left in HBM."""
    torch, sdr, dev = cx.torch, cx.sdr, cx.dev
    samples = 1 << log2_samples
    D = 10
    taps = _taps(255)
    raw = cx.randint_u8(2 * samples, SEED + 3 + cx.rank)
    n_mid = samples // D + 1
    mid = torch.empty(n_mid, dtype=torch.complex64, device=dev)
    n_fin = n_mid // 5 + 16
    fin = torch.empty(n_fin, dtype=torch.complex64, device=dev)
    fir = sdr.Fir(taps, "u8iq", decimation=D, device=dev.index, stream=cx.stream)
    src = sdr.SampleRate(converter, 2, device=dev.index, stream=cx.stream)
    last = {}

    def step():
        got = fir.process_dev(raw, samples, mid, n_mid)
        last["n"] = src.process_dev(0.2, mid, got, fin, n_fin)[1]

    def reset():
        fir.reset()
        src.reset()

    return dict(key=key, units=samples, bytes_per_unit=2.0 + 8.0 / 50, step=step, e2e_setup=None, e2e_step=None,
                h2d=2 * samples, d2h=8 * n_fin, dtype="u8 x s8 -> s32 (tcgen05), sinc accumulation per DESIGN.md",
                kernel="fir_umma_poly_kernel + src_sinc kernels", sharding="independent captures per GPU",
                outputs=lambda: {"resampled": fin[:last["n"]]}, reset=reset)


def wl_fft_c64(cx, logn=12, log2_samples=27):
    torch, sdr, dev = cx.torch, cx.sdr, cx.dev
    n = 1 << logn
    samples = 1 << log2_samples
    batches = samples // n
    x = torch.empty((batches, n), dtype=torch.complex64, device=dev)
    g = torch.Generator(device=dev).manual_seed(SEED + 5 + cx.rank)
    torch.view_as_real(x).uniform_(-1, 1, generator=g)
    out = torch.empty_like(x)
    plan = sdr.FftPlan(n, "c64", device=dev.index, stream=cx.stream)

    def step():
        plan.exec_dev(x, batches, out)

    return dict(key="c5_%d" % logn, units=samples, bytes_per_unit=16.0, step=step, e2e_setup=None, e2e_step=None,
                h2d=8 * samples, d2h=8 * samples, dtype="f32", kernel="fft", sharding="independent batches per GPU",
                outputs=lambda: {"spectrum": out})


def wl_fir_c64(cx, key, K=255, total_ch=1024, log2_n=16, flags=0):
    """the FIR half of C4 alone: total_ch c64 channel streams x K real taps (Fir<f32, Complex<f32>>), channels split
    over the ranks; flags: 0 = default (tcgen05, three bf16 terms), 16 = SDR_FIR_SPLIT2, 2 = SDR_FIR_NO_TENSOR (CUDA cores)"""
    torch, sdr, dev = cx.torch, cx.sdr, cx.dev
    import gen
    n = 1 << log2_n
    taps = gen.lowpass_taps(K, 100e3, 1.8e6)
    clo, chi = sdr.shard.unit_range(total_ch, cx.world, cx.rank)
    n_ch = chi - clo
    g = torch.Generator(device=dev).manual_seed(SEED + 6 + cx.rank)
    x = torch.view_as_complex(torch.rand((n_ch, n, 2), dtype=torch.float32, device=dev, generator=g) * 2 - 1)
    out = torch.empty((n_ch, n), dtype=torch.complex64, device=dev)
    fir = sdr.Fir(taps, "c64", n_channels=n_ch, flags=flags, device=dev.index, stream=cx.stream)

    def step():
        fir.process_dev(x, n, out, n, n, n)

    kern = {0: "fir_umma_c64_kernel<3> (tcgen05, bf16 x 3)", 16: "fir_umma_c64_kernel<2> (tcgen05, bf16 x 2)",
            2: "fir_rb_kernel (CUDA cores)"}.get(flags, "fir")
    return dict(key=key, units=n_ch * n, bytes_per_unit=16.0, step=step, e2e_setup=None, e2e_step=None,
                h2d=8 * n_ch * n, d2h=8 * n_ch * n, dtype="bf16 x bf16 -> f32 (tcgen05 kind::f16)" if flags != 2 else "f32",
                kernel=kern, sharding="%d channels, %d per GPU (shard.unit_range)" % (total_ch, n_ch),
                outputs=lambda: {"filtered": out}, reset=fir.reset)


def wl_channelizer(cx, key="c4", total_ch=128, log2_n=16, fast=True):
    """C4: total_ch channels split over the ranks (shard.unit_range), each channel = 255-tap FIR + PLL"""
    torch, sdr, dev = cx.torch, cx.sdr, cx.dev
    import gen
    n = 1 << log2_n
    taps = gen.lowpass_taps(255, 100e3, 1.8e6)
    B = sdr.BiquadD
    design = sdr.PllDesign(0.0, 0.035, B.LowPass(80000.0, 0.7), B.LowPass(20000.0, 0.7), B.LowPass(20000.0, 0.7))
    clo, chi = sdr.shard.unit_range(total_ch, cx.world, cx.rank)
    n_ch = chi - clo
    g = torch.Generator(device=dev).manual_seed(SEED + 4)
    x_all = torch.rand((total_ch, n, 2), dtype=torch.float32, device=dev, generator=g) * 2 - 1   # same on every rank
    x = torch.view_as_complex(x_all[clo:chi].contiguous())
    out = torch.empty((n_ch, n), dtype=torch.float32, device=dev)
    lk = torch.empty((n_ch, n), dtype=torch.uint8, device=dev)
    ch = sdr.Channelizer(taps, design, n_ch, 1.8e6, fast_math=fast, device=dev.index, stream=cx.stream)

    def step():
        ch.process_dev(x, n, out, lk, n, n)

    def parity():
        if cx.world == 1:
            return None
        ch.reset()
        ch.process_dev(x, n, out, lk, n, n)
        po = cx.gather_rows(out.reshape(-1).view(torch.int32))
        pl = cx.gather_rows(lk.reshape(-1))
        ok = True
        if cx.rank == 0:
            xa = torch.view_as_complex(x_all)
            o0 = torch.empty((total_ch, n), dtype=torch.float32, device=dev)
            l0 = torch.empty((total_ch, n), dtype=torch.uint8, device=dev)
            c0 = sdr.Channelizer(taps, design, total_ch, 1.8e6, fast_math=fast, device=dev.index, stream=cx.stream)
            c0.process_dev(xa, n, o0, l0, n, n)
            ok = bool(torch.equal(torch.cat(po), o0.reshape(-1).view(torch.int32)) and torch.equal(torch.cat(pl), l0.reshape(-1)))
            c0.close()
        return ok

    return dict(key=key, units=n_ch * n, bytes_per_unit=12.125, step=step, e2e_setup=None, e2e_step=None,
                h2d=8 * n_ch * n, d2h=5 * n_ch * n, dtype="f32", kernel="multi-channel FIR + pll_kernel",
                parity=parity, bound="latency (PLL dependent chain)",
                sharding="%d channels, %d per GPU (shard.unit_range)" % (total_ch, n_ch),
                outputs=lambda: {"pll_out": out, "locked": lk}, reset=ch.reset)


def wl_fm(cx, n_st=128, log2_n=18, fast=True):
    """SURVEY 8(f) row 3: the FM stereo receiver of src/main.rs:32-81 for a batch of stations, device resident."""
    torch, sdr, dev = cx.torch, cx.sdr, cx.dev
    n = 1 << log2_n
    row = 2 * n
    raw = cx.randint_u8(n_st * row, SEED + 9).reshape(n_st, row)
    fm = sdr.FmStereo(n_st, 1.8e6, fast_math=fast, device=dev.index, stream=cx.stream)
    cap = fm.max_output(n)
    out = torch.empty((n_st, cap, 2), dtype=torch.float32, device=dev)
    last = {}

    def step():
        last["n"] = fm.process_dev(raw, n, row, out, cap, cap, end_of_input=False)

    return dict(key="fm", units=n_st * n, bytes_per_unit=2.0 + 8.0 / 37.5, step=step, e2e_setup=None, e2e_step=None,
                h2d=2 * n_st * n, d2h=8 * n_st * cap, dtype="f32 (f64 atan2/sincos in the PLLs)",
                kernel="pll_kernel + src_sinc + pll_stereo_kernel + biquad_kernel", bound="latency (PLL dependent chain)",
                outputs=lambda: {"audio": out[:, :last["n"]]}, reset=fm.reset)


def make_workload(name, cx):
    if name == "fm":
        return wl_fm(cx)
    if name == "fmf64":
        return wl_fm(cx, fast=False)
    if name == "fm1024":
        return wl_fm(cx, n_st=1024, log2_n=16)
    if name in ("c2", "fft1024_u8", "default"):
        return wl_fft1024_u8(cx)
    if name == "c2_small":
        return wl_fft1024_u8(cx, 24)
    if name in ("c1", "fir64_u8"):
        return wl_fir_u8(cx, "c1", 64, 1)
    if name == "c1c":
        return wl_fir_u8(cx, "c1c", 64, 1, complex_taps=True)
    if name in ("c3", "fir255_d10_u8"):
        return wl_fir_u8(cx, "c3", 255, 10)
    if name == "c3_2p28":
        return wl_fir_u8(cx, "c3_2p28", 255, 10, log2_samples=28)
    if name == "c3chain":
        return wl_c3_chain(cx)
    if name == "c3chain_linear":
        return wl_c3_chain(cx, "c3chain_linear", converter=4)
    if name == "c3chain_fastest":
        return wl_c3_chain(cx, "c3chain_fastest", converter=2)
    if name == "fir255_u8":
        return wl_fir_u8(cx, "fir255_u8", 255, 1)
    if name == "c4":
        return wl_channelizer(cx, "c4", 128 * cx.world, 16)
    if name == "c4f64":
        return wl_channelizer(cx, "c4", 128 * cx.world, 16, fast=False)
    if name == "c4_1024":
        return wl_channelizer(cx, "c4_1024", 1024, 16)
    if name.startswith("c5_"):
        return wl_fft_c64(cx, int(name[3:]))
    if name in FIR_C64:
        K, flags = FIR_C64[name]
        return wl_fir_c64(cx, name, K, 1024, 16, flags)
    raise SystemExit("unknown workload " + name)


SECONDARY = ["c1", "c1c", "c3", "c3chain", "c4_1024", "fir255_c64", "fir64_c64"] + ["c5_%d" % l for l in range(8, 17)]


def measure_config(cx, name, steps, warmup, peak):
    """one entry of the `configs` array"""
    torch = cx.torch
    t0 = time.perf_counter()
    wl = make_workload(name, cx)
    ms, launches = cx.time_steps(wl["step"], steps, warmup)
    units_all = cx.max_over_ranks(wl["units"]) if cx.world == 1 else None
    if cx.dist is not None:   # ranks may own different unit counts (range / channel split): sum them
        t = torch.tensor([float(wl["units"])], device=cx.dev)
        cx.dist.all_reduce(t, op=cx.dist.ReduceOp.SUM)
        units_all = float(t)
    parity = wl["parity"]() if wl.get("parity") else None
    if parity is not None:
        parity = bool(cx.max_over_ranks(0.0 if parity else 1.0) == 0.0)
    cfg = config_dict(wl["key"])
    achieved = wl["units"] * wl["bytes_per_unit"] / (ms * 1e-3) / 1e9   # this rank's GPU (rank 0 reports)
    entry = {"workload": cfg["workload"], "desc": cfg["desc"], "value": units_all / (ms * 1e-3) / 1e9,
             "unit": "Gsamples/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
             "samples_per_step_all_gpus": units_all, "sharding": wl.get("sharding"), "parity_bit_exact": parity,
             "gpu_launches": launches, "host_enqueue_ms_per_step": round(cx.host_ms_per_step, 4),
             "dtype": wl["dtype"], "kernel": wl["kernel"],
             "roofline": {"bound": wl.get("bound", "hbm"), "achieved": achieved, "peak": peak, "unit": "GB/s",
                          "frac": achieved / peak, "algorithmic_bytes_per_sample": wl["bytes_per_unit"],
                          "traffic": NCU_TRAFFIC.get(cfg["workload"], (None, None))[0]},
             "setup_s": None}
    del wl
    torch.cuda.synchronize(cx.dev)
    torch.cuda.empty_cache()
    entry["setup_s"] = round(time.perf_counter() - t0, 2)
    return entry


def pcie_ceiling(cx, h2d_bytes, d2h_bytes, reps=3):
    """what this box can do for the e2e step with NOTHING but the copies: every rank at once moves h2d_bytes up and
    d2h_bytes down between pinned host memory and its GPU (one cudaMemcpyAsync each, two streams, full duplex)."""
    torch = cx.torch
    hin = torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory()
    hout = torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory()
    din = torch.empty(h2d_bytes, dtype=torch.uint8, device=cx.dev)
    dout = torch.empty(d2h_bytes, dtype=torch.uint8, device=cx.dev)
    s_up, s_dn = torch.cuda.Stream(cx.dev), torch.cuda.Stream(cx.dev)

    def once():
        with torch.cuda.stream(s_up):
            din.copy_(hin, non_blocking=True)
        with torch.cuda.stream(s_dn):
            hout.copy_(dout, non_blocking=True)
        s_up.synchronize()
        s_dn.synchronize()
    once()
    cx.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    cx.barrier()
    dt = cx.max_over_ranks((time.perf_counter() - t0) / reps)
    return dt


def bind_to_gpu_cores(local, world_local):
    """Give each rank its own slice of the host cores (the box exposes one NUMA node, so this only stops the ranks'
    copy-submission threads from migrating over each other); pinned buffers are allocated after this."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = max(1, len(cores) // max(world_local, 1))
        mine = cores[local * per:(local + 1) * per] or cores
        os.sched_setaffinity(0, mine)
        return len(mine)
    except Exception:
        return None


def main():
    sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--configs", default="all", help="all | none | comma list of secondary workloads for the `configs` array")
    ap.add_argument("--config-steps", type=int, default=10)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of the headline workload as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; --impl reference has none")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import sdr_b200 as sdr

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or sdr.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device (libsdr_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    # CPU leg first, on rank 0, BEFORE the process group exists: the other ranks then wait in the rendezvous (a blocking
    # socket read), not in a spinning NCCL barrier that would take host cores away from the baseline
    cpu = None
    if rank == 0 and not args.no_cpu:
        import oracle_lib as O
        threads = O.hardware_threads()
        fn, units = cpu_leg(args.workload)
        fn(units // 16, threads)
        secs = fn(units, threads)
        u1 = max(units // max(threads, 1), 1 << 16)
        secs1 = fn(u1, 1)
        cpu = {"value": units / secs / 1e9, "unit": "Gsamples/s", "cores": threads, "kind": "port",
               "sample": "%d samples of the same workload" % units, "single_thread_value": u1 / secs1 / 1e9}
        if args.workload in ("c2", "default", "fft1024_u8"):
            cpu["optimised_cpu"] = numpy_fft_line(threads)
        _CPU_INPUT.clear()

    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    # everything runs on one explicit stream: the library launches on it and the CUDA events are recorded on it
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    cx = Ctx(torch, sdr, dev, dist, rank, world, stream)
    wl = make_workload(args.workload, cx)
    peak, peak_src = measured_peaks()

    with ClockSampler(local) as clk:
        # the sampler runs from the first warm-up step to the end of the timed region; a short untimed pre-roll
        # keeps the GPU under the same load long enough for nvidia-smi to see it (a step is ~0.5 ms)
        for _ in range(args.warmup):
            wl["step"]()
        t_pre = time.perf_counter()
        while time.perf_counter() - t_pre < 0.4:
            wl["step"]()
            torch.cuda.synchronize(dev)
        if wl.get("reset"):  # the pre-roll's step count varies with the clock; the timed steps start from a fresh stream
            wl["reset"]()
        per_step_ms, launches = cx.time_steps(wl["step"], args.steps, 0)
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, wl["outputs"](), args.dump_outputs)
    value = world * wl["units"] / (per_step_ms * 1e-3) / 1e9
    achieved = wl["units"] * wl["bytes_per_unit"] / (per_step_ms * 1e-3) / 1e9  # GB/s on this rank's GPU

    e2e = None
    if not args.no_e2e and wl["e2e_step"] is not None:
        cores = bind_to_gpu_cores(local, world)
        wl["e2e_setup"]()
        wl["e2e_step"]()
        cx.barrier()
        t0 = time.perf_counter()
        chk = 0.0
        for _ in range(args.e2e_steps):
            chk += wl["e2e_step"]()
        cx.barrier()
        dt = cx.max_over_ranks((time.perf_counter() - t0) / args.e2e_steps)
        wl["host"].clear()
        ceil_dt = pcie_ceiling(cx, wl["h2d"], wl["d2h"])
        e2e = {"value": world * wl["units"] / dt / 1e9, "unit": "Gsamples/s", "h2d_bytes_per_step": wl["h2d"],
               "d2h_bytes_per_step": wl["d2h"], "ms_per_step": dt * 1e3, "steps": args.e2e_steps,
               "api": "host-buffer C ABI call (pinned host memory), H2D + kernel + D2H inside the timed region",
               "ceiling": {"value": world * wl["units"] / ceil_dt / 1e9, "unit": "Gsamples/s", "ms_per_step": ceil_dt * 1e3,
                           "h2d_gbs_per_gpu": wl["h2d"] / ceil_dt / 1e9, "d2h_gbs_per_gpu": wl["d2h"] / ceil_dt / 1e9,
                           "what": "the same bytes moved by bare concurrent pinned cudaMemcpyAsync on every rank at once, no kernel"},
               "frac_of_ceiling": ceil_dt / dt, "host_cores_per_rank": cores}

    configs = []
    if args.configs != "none":
        names = SECONDARY if args.configs == "all" else [c for c in args.configs.split(",") if c]
        names = [c for c in names if c != args.workload]
        for k in ("step", "e2e_step", "e2e_setup", "outputs", "reset"):  # free the headline's device buffers
            wl.pop(k, None)
        torch.cuda.synchronize(dev)
        torch.cuda.empty_cache()
        for name in names:
            try:
                configs.append(measure_config(cx, name, args.config_steps, 3, peak))
            except Exception as e:  # one failing secondary config must not take the headline line with it
                configs.append({"workload": config_dict(name)["workload"], "error": repr(e)[:300]})
                torch.cuda.empty_cache()

    if rank == 0:
        cfg = config_dict(args.workload)
        line = {
            "metric": "FIR/FFT Gsamples/s", "value": value, "unit": "Gsamples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": per_step_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": wl["dtype"], "data": "synthetic",
            "config": cfg,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": NCU_TRAFFIC.get(cfg["workload"], (None, None))[0],
                         "traffic_source": NCU_TRAFFIC.get(cfg["workload"], (None, None))[1],
                         "algorithmic_bytes": wl["units"] * wl["bytes_per_unit"],
                         "peak_source": peak_src, "kernel": wl["kernel"],
                         "algorithmic_bytes_per_sample": wl["bytes_per_unit"]},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
            "host_enqueue_ms_per_step": round(cx.host_ms_per_step, 4), "clocks": clk.summary(),
            "configs": configs,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
