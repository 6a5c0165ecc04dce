"""GPU: every kernel path of the power-of-two FFT (csrc/fft.cu) against f64 truth, at the sizes, formats, flags, batch
counts and addresses that select it, and the exact relations that hold between paths.

Dispatch (launch_fmt; n = 16 ... 65536, one launch per call, except f32 rfft at 2^15 / 2^16, which the plan runs as
convert + plain c64 transform + finish).  "Unaligned" means element-aligned but not 16-byte aligned.

  n              format, flags               address                    kernel                                 loop
  16 ... 128     any                         any                        fft_cta_kernel<log n>                  SEQ = 4096/n per CTA
  256, 512       any                         any                        fft_reg2_kernel<log n>                 persistent, SEQ 16, 8
  1024           u8, shift                   input 16-byte aligned      fft1024_warp_kernel<U8, 1, TMA>        persistent warps
  1024           u8, no shift                input 16-byte aligned      fft1024_warp_kernel<U8, 0, TMA>        persistent warps
  1024           c64                         input 16-byte aligned      fft1024_warp_kernel<C64, 2>            persistent warps
  1024           f32, plain or rfft          any                        fft_cta_kernel<10>                     SEQ = 4
  1024           u8, c64                     input unaligned            fft_cta_kernel<10>                     SEQ = 4
  2048, 4096     c64                         any                        fft_reg2_kernel<log n, REGPF>          persistent, SEQ 2, 1
  2048, 4096     u8, f32 (plain or rfft)     any                        fft_reg2_kernel<log n>                 persistent, SEQ 2, 1
  8192           c64                         any                        fft_reg2_kernel<13, REGPF>             persistent
  8192           u8, f32 (plain or rfft)     input 16-byte aligned      fft_reg2_kernel<13> + cp.async prefetch persistent
  8192           u8, f32 (plain or rfft)     input unaligned            fft_cta_kernel<13>                     1 per CTA
  16384          f32 rfft                    any                        fft_cta_kernel<14>                     1 per CTA
  2^14 ... 2^16  no rfft                     in and out 16-byte aligned fft_l2t_kernel<log n - 8>              persistent items
  2^14 ... 2^16  no rfft                     in or out unaligned        fft_l2_kernel<log n - 8>               persistent tickets
  2^15, 2^16     f32 rfft                    any                        convert + fft_l2t_kernel<C64> + finish persistent items
  2^14           SDR_FFT_NO_L2=1             any                        fft_cta_kernel<14>                     1 per CTA
  2^15, 2^16     SDR_FFT_NO_L2=1             any                        fft_cols_kernel, two launches          not persistent

The output feeds fft_l2t_kernel's scratch tensor map, which cuTensorMapEncodeTiled refuses for an address that is not
16-byte aligned: that is why an unaligned output also selects fft_l2_kernel.

Reference: X64 = torch.fft.fft in complex128 on the device, from the exactly unpacked input (u8: (b - 128)/128; f32:
real + 0j); three rows per case are pinned to numpy.fft.fft on the host.  Shift, norm (the plan's f32 1/sqrt(N)) and
the rfft slice (bins 0 ... n - n/2 - 1) are applied in f64 as include/sdr_b200.h defines them.

Bars, per transform:  rms_rel = |X - X64|_2 / |X64|_2 <= 5e-8 log2 N  and  max_k |X - X64| / rms(X64) <= 4e-7 log2 N.
An f32 FFT of u8 noise (scipy, complex64) has rms_rel 4.9e-8 (N = 16) ... 1.4e-7 (N = 65536) and max_rel 3.8e-7 ...
6.4e-7: the bars are 3 to 10 times that.

Batch counts: 1; a count that is not a multiple of the transforms per CTA; and 3 SMs max(1, 65536/n) + 7, which makes
every persistent kernel go round its loop at least three times with a ragged last round (launch_w1k keeps 2 SMs x 8
warps resident, launch_reg2 SMs x occupancy x SEQ transforms, the four-step kernels SMs x occupancy items of n/4096
columns).  Every output buffer carries a 64-element guard filled with a sentinel that must survive the call; a
sentinel left inside the output fails the f64 bars (it is a NaN).
"""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DEV = "cuda"
LOGNS = list(range(4, 17))
RMS_BAR, MAX_BAR = 5e-8, 4e-7
GUARD = 64
SENTINEL = 0x7FBADBAD  # a NaN: an output element the kernel never wrote fails the bars
ES = {"u8iq": 2, "c64": 8, "f32": 4}
# name: (input format, shift, norm, rfft)
VARIANTS = {
    "u8": ("u8iq", False, False, False), "u8-shift": ("u8iq", True, False, False),
    "u8-norm": ("u8iq", False, True, False), "u8-shift-norm": ("u8iq", True, True, False),
    "c64": ("c64", False, False, False), "c64-shift": ("c64", True, False, False),
    "c64-norm": ("c64", False, True, False), "c64-shift-norm": ("c64", True, True, False),
    "f32": ("f32", False, False, False), "f32-rfft": ("f32", False, False, True), "f32-rfft-norm": ("f32", False, True, True),
}
COUNTS = ["1", "ragged", "wrap"]
WORST = {}  # (kernel, format) -> [rms_rel / log2 N, max_rel / log2 N, n of each]


def _torch():
    import torch
    return torch


def sync():
    if DEV == "cuda":
        _torch().cuda.synchronize()


def sm_count():
    return _torch().cuda.get_device_properties(0).multi_processor_count


def batch_count(n, count):
    if count == "1":
        return 1
    if count == "ragged":
        return 2 * max(8, 4096 // n) + 3  # not a multiple of SEQ (4096/n), of 8 warps, or of 2
    return 3 * sm_count() * max(1, 65536 // n) + 7


def kernel_of(n, fmt, shift=False, rfft=False, in16=True, out16=True, no_l2=False):
    """the kernel launch_fmt runs (the table above)"""
    logn = n.bit_length() - 1
    if logn <= 7:
        return "fft_cta_kernel<%d>" % logn
    if logn in (8, 9):
        return "fft_reg2_kernel<%d>" % logn
    if logn == 10:
        if fmt == "u8iq" and in16 and not rfft:
            return "fft1024_warp_kernel<U8, %d, TMA>" % int(shift)
        if fmt == "c64" and in16:
            return "fft1024_warp_kernel<C64, 2>"
        return "fft_cta_kernel<10>"
    if logn in (11, 12):
        return "fft_reg2_kernel<%d%s>" % (logn, ", REGPF" if fmt == "c64" else "")
    if logn == 13:
        if fmt == "c64":
            return "fft_reg2_kernel<13, REGPF>"
        return "fft_reg2_kernel<13> + cp.async prefetch" if in16 else "fft_cta_kernel<13>"
    if rfft:
        return "fft_cta_kernel<14>" if logn == 14 else "convert + fft_l2t_kernel<C64> + finish"
    if no_l2:
        return "fft_cta_kernel<14>" if logn == 14 else "fft_cols_kernel x2"
    return "fft_l2t_kernel" if in16 and out16 else "fft_l2_kernel"


def bars(n):
    logn = n.bit_length() - 1
    return RMS_BAR * logn, MAX_BAR * logn


def plan_norm(n):
    return float(np.float32(1.0) / np.sqrt(np.float32(n)))


def plan(sdr, n, fmt, shift=False, norm=False, rfft=False):
    torch = _torch()
    stream = torch.cuda.current_stream() if DEV == "cuda" else None
    return sdr.FftPlan(n, fmt, shift=shift, norm=norm, rfft=rfft, stream=stream)


def bits(t):
    return _torch().view_as_real(t).view(_torch().int32)


def same_bits(a, b):
    return a.shape == b.shape and bool(_torch().equal(bits(a), bits(b)))


def raw_bytes(raw):
    torch = _torch()
    if raw.dtype == torch.complex64:
        raw = torch.view_as_real(raw)
    return raw.reshape(-1).view(torch.uint8)


# ---- inputs and the f64 reference, one case (n, format, count) cached at a time -----------------------------------
_CASE = {}


def _unpack64(raw, fmt):
    torch = _torch()
    if fmt == "u8iq":
        r = raw.to(torch.float64)
        return torch.complex((r[:, 0::2] - 128.0) / 128.0, (r[:, 1::2] - 128.0) / 128.0)
    return raw.to(torch.complex128)


def _unpack64_host(raw, fmt):
    if fmt == "u8iq":
        r = raw.astype(np.float64)
        return (r[0::2] - 128.0) / 128.0 + 1j * ((r[1::2] - 128.0) / 128.0)
    return raw.astype(np.complex128)


def case(n, fmt, count):
    """{"raw": device input (batches, n) in the plan's format, "X64": plain f64 spectra, "batches"}"""
    key = (n, fmt, count)
    if key in _CASE:
        return _CASE[key]
    _CASE.clear()
    torch = _torch()
    batches = batch_count(n, count)
    seed = 1000 * n + 10 * list(ES).index(fmt) + COUNTS.index(count)
    g = torch.Generator(device=DEV).manual_seed(seed)
    if fmt == "u8iq":
        raw = torch.randint(0, 256, (batches, 2 * n), dtype=torch.uint8, device=DEV, generator=g)
    elif fmt == "c64":
        raw = torch.empty((batches, n), dtype=torch.complex64, device=DEV)
        torch.view_as_real(raw).uniform_(-1.0, 1.0, generator=g)
    else:
        raw = torch.empty((batches, n), dtype=torch.float32, device=DEV).uniform_(-1.0, 1.0, generator=g)
    X64 = torch.fft.fft(_unpack64(raw, fmt), dim=1)
    for r in sorted({0, batches // 2, batches - 1}):  # the device reference pinned to numpy on the host
        ref = np.fft.fft(_unpack64_host(raw[r].cpu().numpy(), fmt))
        dev = X64[r].cpu().numpy()
        assert np.abs(dev - ref).max() <= 1e-12 * np.sqrt(np.mean(np.abs(ref) ** 2)), (n, fmt, r)
    _CASE[key] = {"raw": raw, "X64": X64, "batches": batches}
    return _CASE[key]


def expected(X64, n, shift=False, norm=False, rfft=False):
    torch = _torch()
    X = X64
    if rfft:
        X = X[:, :n - n // 2]
    elif shift:
        X = torch.roll(X, n // 2, dims=1)
    if norm:
        X = X * plan_norm(n)
    return X


def run_dev(p, inp, batches, out_offset=0):
    """exec_dev into a fresh output of batches * out_len + GUARD c64 at `out_offset` bytes past a 256-byte boundary,
    filled with SENTINEL; asserts the guard survived; returns the (batches, out_len) complex64 output"""
    torch = _torch()
    used = batches * p.out_len
    buf = torch.full((2 * (used + GUARD) + 2,), SENTINEL, dtype=torch.int32, device=DEV)
    out = buf[out_offset // 4:out_offset // 4 + 2 * (used + GUARD)].view(torch.complex64)
    p.exec_dev(inp, batches, out)
    sync()
    assert bool((bits(out[used:]) == SENTINEL).all()), "write past the output"
    return out[:used].view(batches, p.out_len)


def errors(got, want):
    """worst (rms_rel, max_rel) over the transforms (rows), and the row of each"""
    torch = _torch()
    d = got.to(torch.complex128) - want
    e2 = d.real ** 2 + d.imag ** 2
    del d
    p2 = want.real ** 2 + want.imag ** 2
    rms = torch.sqrt(e2.sum(dim=1) / p2.sum(dim=1))
    mx = torch.sqrt(e2.max(dim=1).values / p2.mean(dim=1))
    # NaN (an unwritten sentinel, a poisoned row) must fail: nan_to_num maps it above every bar
    rms, mx = torch.nan_to_num(rms, nan=1.0), torch.nan_to_num(mx, nan=1.0)
    return float(rms.max()), float(mx.max()), int(rms.argmax()), int(mx.argmax())


def check_errors(kernel, fmt, n, rms, mx, where=""):
    """records the path's worst errors for the report, then holds them to the bars"""
    logn = n.bit_length() - 1
    w = WORST.setdefault((kernel, fmt), [0.0, 0.0, 0, 0])
    if rms / logn > w[0]:
        w[0], w[2] = rms / logn, n
    if mx / logn > w[1]:
        w[1], w[3] = mx / logn, n
    b_rms, b_max = bars(n)
    assert rms <= b_rms, "%s %s n=%d: rms_rel %.3g > %.3g %s" % (kernel, fmt, n, rms, b_rms, where)
    assert mx <= b_max, "%s %s n=%d: max_rel %.3g > %.3g %s" % (kernel, fmt, n, mx, b_max, where)


def check_bars(kernel, fmt, n, got, want):
    rms, mx, r_rms, r_mx = errors(got, want)
    check_errors(kernel, fmt, n, rms, mx, "(rows %d, %d)" % (r_rms, r_mx))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    _CASE.clear()
    if WORST:
        print("\nworst error per path, divided by log2 N (bars: rms %.1e, max %.1e):" % (RMS_BAR, MAX_BAR))
        for (k, f), (r, m, nr, nm) in sorted(WORST.items()):
            print("  %-42s %-5s rms_rel %.3e (n=%d)  max_rel %.3e (n=%d)" % (k, f, r, nr, m, nm))


def _plain(sdr, n, fmt, count):
    c = case(n, fmt, count)
    if "plain" not in c:
        c["plain"] = run_dev(plan(sdr, n, fmt), c["raw"], c["batches"])
    return c["plain"]


# ---- every (n, format, flags, count) against f64, and exactly against the plain transform -------------------------
@pytest.mark.parametrize("count", COUNTS)
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("logn", LOGNS)
def test_path_against_f64_and_plain(sdr, logn, variant, count):
    """f64 bars on every transform; shift = roll(plain, n/2) and norm = f32(plain) * f32(1/sqrt n) bit for bit (the
    header's definitions); rfft = the first n - n/2 bins of the plain f32 transform (times the norm) bit for bit where
    both run the same kernel arithmetic; host exec = exec_dev bit for bit"""
    torch = _torch()
    n = 1 << logn
    fmt, shift, norm, rfft = VARIANTS[variant]
    c = case(n, fmt, count)
    p = plan(sdr, n, fmt, shift, norm, rfft)
    got = run_dev(p, c["raw"], c["batches"])
    kernel = kernel_of(n, fmt, shift, rfft)
    check_bars(kernel, fmt, n, got, expected(c["X64"], n, shift, norm, rfft))

    plain = _plain(sdr, n, fmt, count)
    if rfft and n == 16384:
        pass  # fft_cta_kernel<14> (rfft) against fft_l2t_kernel (plain): different radix splits; the bars hold
    elif shift or norm or rfft:
        # 2^15, 2^16: rfft runs the c64 instance of fft_l2t_kernel on (x, 0), plain f32 the f32 instance on x: the same
        # operations (test_input_formats_agree_with_c64)
        want = plain[:, :n - n // 2] if rfft else torch.roll(plain, n // 2, dims=1) if shift else plain
        if norm:
            want = torch.view_as_complex(torch.view_as_real(want) * torch.tensor(plan_norm(n), dtype=torch.float32,
                                                                                   device=DEV))
        assert same_bits(got, want.contiguous())
    if rfft:  # rfft implies shift (header): the flag changes nothing
        p2 = plan(sdr, n, fmt, True, norm, True)
        assert same_bits(run_dev(p2, c["raw"], c["batches"]), got)
    if count != "wrap":
        host = p.exec(c["raw"].cpu().numpy())
        assert np.array_equal(host.view(np.uint32), got.cpu().numpy().view(np.uint32))


# ---- u8 and f32 input against c64 input of the same samples -------------------------------------------------------
def _differs_from_c64(n, fmt):
    """where the u8 or f32 instance of a kernel does not perform the c64 instance's operations:
    - 1024: the u8 warp kernel uses packed complex adds (dft32<true>: no multiply-add contraction across them) and the
      c64 one does not; f32 runs fft_cta_kernel<10> (radix 16, 16, 4 instead of 32 x 32);
    - 8192, f32: fft_reg2_kernel<13> (cp.async prefetch) unpacks the raw copy into registers as (x, 0), so the compiler
      knows the imaginary parts of pass 0 are zero; with the unpacked adds of this size (Reg2Plan::PACKED is false
      at 8192 only) it drops the zero terms and contracts a product into the following add (the f32 instance has
      38 FADD and 3 FMUL fewer, 1 FFMA more), which rounds once where the c64 instance rounds twice.  At the other
      reg2 sizes the adds are packed (inline PTX), which the compiler neither folds nor contracts."""
    return n == 1024 or (n == 8192 and fmt == "f32")


@pytest.mark.parametrize("fmt", ["u8iq", "f32"])
@pytest.mark.parametrize("logn", LOGNS)
def test_input_formats_agree_with_c64(sdr, logn, fmt):
    """u8 = c64 of the unpacked samples, f32 = c64 with zero imaginary part, bit for bit wherever both formats run the
    same kernel arithmetic; where they do not (_differs_from_c64) both meet the f64 bars"""
    torch = _torch()
    n = 1 << logn
    c = case(n, fmt, "wrap")
    got = run_dev(plan(sdr, n, fmt), c["raw"], c["batches"])
    x = _unpack64(c["raw"], fmt).to(torch.complex64)  # exact: u8 samples are multiples of 1/128
    two = run_dev(plan(sdr, n, "c64"), x, c["batches"])
    del x
    if _differs_from_c64(n, fmt):
        check_bars(kernel_of(n, fmt), fmt, n, got, c["X64"])
        check_bars(kernel_of(n, "c64"), "c64", n, two, c["X64"])
    else:
        assert same_bits(got, two)


# ---- a transform's place in the persistent loop does not change its bits -----------------------------------------
def _per_cta(n):
    """transforms per resident CTA (four-step kernels: one CTA takes one item of n/4096 columns per round)"""
    if n == 1024:
        return 16  # launch_w1k: 2 CTAs of 8 warps per SM, exactly
    if n >= 16384:
        return 4096 / (2 * n)  # 2 n/4096 items per transform
    return max(1, 4096 // n)


ROW_CASES = [(logn, v) for logn in LOGNS for v in ("u8", "c64", "f32")] + [(10, "u8-shift"), (13, "f32-rfft")]


@pytest.mark.parametrize("logn,variant", ROW_CASES)
def test_rows_equal_one_transform_calls(sdr, logn, variant):
    """rows at the start, at every place a round of the persistent loop could end (resident CTAs = SMs x 1 ... 8 per
    SM: the occupancy the launcher queries lies in that range) and in the ragged tail of a wrapping run are bit-identical
    to a 1-transform call on the same input"""
    n = 1 << logn
    fmt, shift, norm, rfft = VARIANTS[variant]
    c = case(n, fmt, "wrap")
    B = c["batches"]
    p = plan(sdr, n, fmt, shift, norm, rfft)
    got = run_dev(p, c["raw"], B)
    sms, per = sm_count(), _per_cta(n)
    rows = {0, 1, B - 2, B - 1}
    for k in range(1, 9):
        r = int(np.ceil(sms * k * per))
        rows |= {r - 1, r}
    for r in sorted(x for x in rows if 0 <= x < B):
        one = run_dev(p, c["raw"][r:r + 1], 1)
        assert same_bits(one, got[r:r + 1]), (n, variant, r)


# ---- one poisoned transform stays in its row ---------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["u8iq", "c64", "f32"])
@pytest.mark.parametrize("logn", LOGNS)
def test_poisoned_transform_stays_in_its_row(sdr, logn, fmt):
    """a NaN in transform r (c64, f32) makes every bin of row r NaN; a changed byte (u8) changes row r; every other row
    is bit-identical to the clean run.  r lies in a late round and in the ragged last round, so a leak through an
    exchange buffer, a prefetch buffer or the in-flight scratch of the four-step kernels shows"""
    torch = _torch()
    n = 1 << logn
    c = case(n, fmt, "wrap")
    B = c["batches"]
    plain = _plain(sdr, n, fmt, "wrap")
    rows = sorted({B // 2 + 1, B - 3})
    raw = c["raw"].clone()
    j = n // 3
    for r in rows:
        if fmt == "u8iq":
            raw[r, 2 * j] ^= 0x55
        elif fmt == "c64":
            raw[r, j] = complex(float("nan"), float("nan"))
        else:
            raw[r, j] = float("nan")
    got = run_dev(plan(sdr, n, fmt), raw, B)
    keep = torch.ones(B, dtype=torch.bool, device=DEV)
    keep[rows] = False
    assert same_bits(got[keep], plain[keep])
    for r in rows:
        if fmt == "u8iq":
            assert not same_bits(got[r], plain[r])
        else:
            assert bool((torch.isnan(got[r].real) | torch.isnan(got[r].imag)).all()), (n, fmt, r)


# ---- the host pipeline over several chunks ----------------------------------------------------------------------
@pytest.mark.parametrize("n,fmt,batches", [(1024, "u8iq", 2 * 16384 + 5), (8192, "c64", 1300)])
def test_host_exec_over_several_chunks_equals_exec_dev(sdr, n, fmt, batches):
    """exec stages 32 MiB of input per chunk, double-buffered: three chunks here, the last one short"""
    torch = _torch()
    g = torch.Generator(device=DEV).manual_seed(n + batches)
    if fmt == "u8iq":
        raw = torch.randint(0, 256, (batches, 2 * n), dtype=torch.uint8, device=DEV, generator=g)
    else:
        raw = torch.empty((batches, n), dtype=torch.complex64, device=DEV)
        torch.view_as_real(raw).uniform_(-1.0, 1.0, generator=g)
    assert batches * n * ES[fmt] > 2 * (32 << 20)
    p = plan(sdr, n, fmt, shift=True, norm=True)
    dev = run_dev(p, raw, batches)
    host = p.exec(raw.cpu().numpy())
    assert np.array_equal(host.view(np.uint32), dev.cpu().numpy().view(np.uint32))


# ---- addresses ---------------------------------------------------------------------------------------------------
def _unaligned_arith_differs(n, fmt):
    """1024, u8 / c64: the aligned call runs the warp kernel (32 x 32), the unaligned one fft_cta_kernel<10> (16, 16,
    4).  Everywhere else the two kernels perform the same operations in the same order (f32 at 8192 aside, see
    test_unaligned_input): fft_cta_kernel<13> and fft_reg2_kernel<13> both run the Stockham passes 16, 16, 16, 2 with the
    same table twiddles and unpacked butterflies; fft_l2_kernel and fft_l2t_kernel read the same tile elements into the
    same registers and share every arithmetic line (the product-tree twiddles included) -- they differ only in how the
    tile reaches the registers (ticket order and global loads against static items and TMA copies)."""
    return n == 1024 and fmt != "f32"


@pytest.mark.parametrize("fmt", ["u8iq", "c64", "f32"])
@pytest.mark.parametrize("logn", LOGNS)
def test_unaligned_input(sdr, logn, fmt):
    """exec_dev with the input one element past a 16-byte boundary: the fallback kernels at 1024, 8192 and 2^14 ...
    2^16; f64 bars, and bit-identical to the aligned call where the arithmetic is the same"""
    torch = _torch()
    n = 1 << logn
    c = case(n, fmt, "wrap")
    B = c["batches"]
    src = raw_bytes(c["raw"])
    es = ES[fmt]
    buf = torch.empty(src.numel() + 16, dtype=torch.uint8, device=DEV)
    buf[es:es + src.numel()].copy_(src)
    got = run_dev(plan(sdr, n, fmt), buf.data_ptr() + es, B)
    check_bars(kernel_of(n, fmt, in16=False), fmt, n, got, c["X64"])
    if n == 8192 and fmt == "f32":
        # fft_cta_kernel<13> stages the input through shared memory and computes what the c64 instances compute; the
        # aligned call's prefetching instance does not (_differs_from_c64)
        x = c["raw"].to(torch.complex64)
        assert same_bits(got, run_dev(plan(sdr, n, "c64"), x, B))
    elif not _unaligned_arith_differs(n, fmt):
        assert same_bits(got, _plain(sdr, n, fmt, "wrap"))


@pytest.mark.parametrize("fmt", ["u8iq", "c64", "f32"])
@pytest.mark.parametrize("logn", LOGNS)
def test_output_at_8_not_16_byte_alignment(sdr, logn, fmt):
    """an output 8 bytes past a 16-byte boundary (fft_l2_kernel at 2^14 ... 2^16): bit-identical to the aligned call"""
    n = 1 << logn
    c = case(n, fmt, "wrap")
    got = run_dev(plan(sdr, n, fmt), c["raw"], c["batches"], out_offset=8)
    assert same_bits(got, _plain(sdr, n, fmt, "wrap"))
    check_bars(kernel_of(n, fmt, out16=False), fmt, n, got, c["X64"])


@pytest.mark.parametrize("n", [1024, 16384])
@pytest.mark.parametrize("fmt,in_off,out_off", [("u8iq", 1, 0), ("c64", 4, 0), ("f32", 2, 0), ("c64", 0, 4),
                                                ("u8iq", 0, 4)])
def test_exec_dev_refuses_misaligned_pointers(sdr, n, fmt, in_off, out_off):
    """an input that is not a multiple of its element size, or an output that is not 8-byte aligned, is refused
    with SDR_ERR_MISALIGNED (105) before anything runs: the output is untouched"""
    torch = _torch()
    batches = 3
    inp = torch.zeros(batches * n * ES[fmt] + 16, dtype=torch.uint8, device=DEV)
    out = torch.full((2 * batches * n + 8,), SENTINEL, dtype=torch.int32, device=DEV)
    p = plan(sdr, n, fmt)
    with pytest.raises(sdr.SdrError) as e:
        p.exec_dev(inp.data_ptr() + in_off, batches, out.data_ptr() + out_off)
    assert e.value.code == 105
    sync()
    assert bool((out == SENTINEL).all())


@pytest.mark.parametrize("fmt", ["u8iq", "c64", "f32"])
def test_host_exec_takes_input_at_any_offset(sdr, fmt):
    """exec copies host input into its own device buffers: a host view at an odd byte offset is fine"""
    n, batches = 1024, 5
    c = case(n, fmt, "ragged")
    host = c["raw"][:batches].cpu().numpy()
    nb = host.nbytes
    buf = np.zeros(nb + 16, np.uint8)
    off = 1 if fmt == "u8iq" else 4 if fmt == "c64" else 2
    view = np.frombuffer(buf.data, host.dtype, count=host.size, offset=off).reshape(host.shape)
    view[...] = host
    p = plan(sdr, n, fmt)
    got = p.exec(view)
    want = p.exec(np.ascontiguousarray(host))
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


# ---- SDR_FFT_NO_L2=1: the operational fallback for MPS / partitioned GPUs ------------------------------------------
NO_L2_CASES = [(logn, v) for logn in (14, 15, 16) for v in ("u8", "c64", "u8-shift-norm", "c64-shift-norm")]


def no_l2_child(path):
    """run in a process with SDR_FFT_NO_L2=1: the f64 errors of NO_L2_CASES at a wrapping count, as JSON"""
    import sdr_b200 as sdr
    res = []
    for logn, variant in NO_L2_CASES:
        n = 1 << logn
        fmt, shift, norm, rfft = VARIANTS[variant]
        c = case(n, fmt, "wrap")
        got = run_dev(plan(sdr, n, fmt, shift, norm), c["raw"], c["batches"])
        rms, mx, _, _ = errors(got, expected(c["X64"], n, shift, norm))
        res.append({"n": n, "variant": variant, "rms": rms, "max": mx})
    with open(path, "w") as f:
        json.dump(res, f)


def test_no_l2_fallback(sdr):
    """SDR_FFT_NO_L2=1 (read once per process) selects fft_cta_kernel<14> and the two-launch four-step"""
    here = os.path.dirname(os.path.abspath(__file__))
    pkg = os.path.join(os.path.dirname(here), "unnamed-rust-sdr_b200")
    code = "import sys; sys.path[:0] = [%r, %r]; import test_gpu_fft_paths as T; T.no_l2_child(sys.argv[1])" % (pkg, here)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "no_l2.json")
        subprocess.check_call([sys.executable, "-c", code, path], env=dict(os.environ, SDR_FFT_NO_L2="1"))
        with open(path) as f:
            res = json.load(f)
    assert len(res) == len(NO_L2_CASES)
    for r in res:
        n, fmt = r["n"], VARIANTS[r["variant"]][0]
        check_errors(kernel_of(n, fmt, no_l2=True), fmt, n, r["rms"], r["max"], r["variant"])
