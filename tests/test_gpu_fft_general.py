"""GPU: every FftPlan length that is not a single-launch power of two -- the direct DFT, Bluestein and the four-step
path -- and the sliding-window spectra of WindowFft, against f64 truth (the bars of fft_bars.py), at the lengths that
reach each inner kernel, the formats, flags and batch counts that cross a slab, and the addresses the caller picks.

Dispatch (fft_plan_init / fft_run_dev in csrc/api.cu; kernels in csrc/fft.cu):

  n                                   path             kernels                                         slab (transforms)
  1 ... 63, not a power of two >= 16  direct DFT       fft_naive_kernel, one thread per output bin     none
  2^4 ... 2^16                        (test_gpu_fft_paths.py)
  every other n <= 2^26               Bluestein        bluestein_pre, 2 x length-m c64 transform,      2^23 / m
    m = pow2 >= 2n - 1, >= 16                          bluestein_mul, bluestein_post
  2^17 ... 2^27; f32 rfft of 2^15, 2^16  four-step     fft_convert, fft_huge_launch (transpose, N2 x     2^25 / n
                                                       2^(l/2), transpose with f64 twiddle, N1 x 2^ceil(l/2),
                                                       transpose), fft_finish; rfft 2^15 / 2^16 run one
                                                       c64 fft_l2t_kernel instead of fft_huge_launch

  inner c64 transform of length 2^l    kernel (launch_fmt, with the plan's 16-byte aligned scratch)
  l = 8, 9                             fft_reg2_kernel<l>
  l = 10                               fft1024_warp_kernel<C64, 2>
  l = 11 ... 13                        fft_reg2_kernel<l, REGPF>
  l = 14 ... 16                        fft_l2t_kernel<l - 8> (with the plan's work array)
  l = 17 ... 27                        fft_huge_launch: 2^(l/2) and 2^ceil(l/2) inside, so l = 20 runs the warp
                                       kernel, l = 26, 27 fft_reg2_kernel<13, REGPF>, l = 27 fft_l2t_kernel<6> (2^14)

Only the first kernel (format, caller's input address) and the last (shift, norm, rfft, caller's output address) of
these paths differ between variants, so the relations between variants hold bit for bit: shift = roll(plain, n/2),
norm = f32(plain) * f32(1/sqrt n), rfft = the first n - n/2 bins of the plain f32 transform, u8 = c64 of the exactly
unpacked samples, f32 = c64 with a zero imaginary part, and an unaligned input or output = the aligned call.  The last
two hold in fft_naive_kernel too: its f32 instance keeps the products with the known zero (SASS: FMUL RZ, -R.. then
FFMA, the c64 instance's sequence), so nothing is folded or contracted differently.

Reference: X64 = torch.fft.fft in complex128 on the device, from the exactly unpacked input; rows of cases up to 2^20
points are pinned to numpy.fft.fft on the host.  Every transform meets the bars of fft_bars.py (rms_rel, and max_rel
with Bluestein's term for a towering bin: the DC bin of u8 noise is 55 times rms(X64) at n = 2^26).  Every output
carries a guard of sentinels (NaN) that must survive.
Counts: 1; a ragged count (7, or 4099 for the direct DFT); "slabs" = 2 slabs + 3 transforms (3 slabs, the last one
short), or 2 transforms where that would exceed 2^27 points; "many" = 70001 direct-DFT transforms.
"""
import numpy as np
import pytest

import fft_bars as B
from test_gpu_fft_paths import (ES, GUARD, SENTINEL, VARIANTS, _torch, _unpack64_host, bits, plan, plan_norm,
                                raw_bytes, same_bits, sync)

pytestmark = pytest.mark.gpu

DEV = "cuda"
CHUNK = 1 << 24  # elements per step of the error reduction: bounds its temporaries at the longest lengths
WORST = {}  # (path, format) -> {"rms": (rms / bar, rms, bar, n), "max": (...)}

DIRECT_N = [1, 2, 3, 4, 5, 7, 8, 12, 15, 31, 33, 60, 63]
# near both ends of each m up to 2^19, one n per m above (2^k + 2^(k-5) and 2^(k+1) - 2^(k-5) factor into 2, 3, 11
# and 2, 3, 7, which keeps the complex128 reference off cuFFT's own Bluestein at 2^21 ... 2^26 points)
BLUESTEIN_N = [65, 127, 129, 255, 257, 511, 513, 1000, 1023, 1025, 2047, 2049, 4095, 4097, 8191, 8193, 14400, 16383,
               16385, 30000, 32767, 32769, 40000, 65535, 65537, 100000, 131071, 131073, 180000, 262143, 262145,
               524289, (1 << 20) + 1, (1 << 21) + (1 << 16), (1 << 22) + (1 << 17), (1 << 23) + (1 << 18),
               (1 << 24) + (1 << 19), (1 << 26) - (1 << 20)]
FOURSTEP_N = [1 << l for l in range(17, 28)]
RFFT_MODE3_N = [1 << 15, 1 << 16]
SMALL = 1 << 17   # every variant at every count up to here
HUGE = 1 << 24    # above: two variants
SOME_VARIANTS = ["u8", "u8-shift-norm", "c64", "c64-shift-norm", "f32", "f32-rfft", "f32-rfft-norm"]
HUGE_VARIANTS = ["u8", "u8-shift-norm"]


def _pow2_inner(l):
    if l in (8, 9):
        return "fft_reg2_kernel<%d>" % l
    if l == 10:
        return "fft1024_warp_kernel<C64, 2>"
    if l <= 13:
        return "fft_reg2_kernel<%d, REGPF>" % l
    if l <= 16:
        return "fft_l2t_kernel<%d>" % (l - 8)
    return "four-step 2^%d x 2^%d" % (l // 2, l - l // 2)


def kernel_of(n, rfft=False):
    p = B.path(n, rfft)
    if p == "direct":
        return "direct: fft_naive_kernel"
    if p == "bluestein":
        lm = B.ilog2(B.bluestein_m(n))
        return "bluestein m=2^%d: %s" % (lm, _pow2_inner(lm))
    return "four-step: convert, %s, finish" % _pow2_inner(B.ilog2(n))


def slab_of(n, rfft=False):
    p = B.path(n, rfft)
    if p == "bluestein":
        return max(1, (64 << 20) // (8 * B.bluestein_m(n)))
    if p == "fourstep":
        return max(1, (256 << 20) // (8 * n))
    return None


def batch_count(n, count, rfft=False):
    if count == "1":
        return 1
    if count == "many":
        return 70001
    if count == "ragged":
        return 4099 if B.path(n, rfft) == "direct" else 7
    s = slab_of(n, rfft)
    return 2 * s + 3 if (2 * s + 3) * n <= 1 << 27 else 2


# ---- inputs and the f64 reference, one case (n, format, count) cached at a time -----------------------------------
_CASE = {}


def _free_case():
    big = any(c["raw"].numel() > CHUNK for c in _CASE.values())
    _CASE.clear()
    if big:
        _torch().cuda.empty_cache()  # the machine is shared: give the longest cases' memory back


def make_input(n, fmt, rows, seed):
    torch = _torch()
    g = torch.Generator(device=DEV).manual_seed(seed)
    if fmt == "u8iq":
        return torch.randint(0, 256, (rows, 2 * n), dtype=torch.uint8, device=DEV, generator=g)
    if fmt == "c64":
        raw = torch.empty((rows, n), dtype=torch.complex64, device=DEV)
        torch.view_as_real(raw).uniform_(-1.0, 1.0, generator=g)
        return raw
    return torch.empty((rows, n), dtype=torch.float32, device=DEV).uniform_(-1.0, 1.0, generator=g)


def exact(raw, fmt, dtype):
    """the samples of raw as complex `dtype` (exact: u8 samples are multiples of 1/128), one temporary at most"""
    torch = _torch()
    if fmt != "u8iq":
        return raw.to(dtype)
    r = raw.view(raw.shape[0], -1, 2).to(torch.float64 if dtype == torch.complex128 else torch.float32)
    return torch.view_as_complex(r.sub_(128.0).div_(128.0))


def reference(raw, fmt, n):
    """f64 spectra of the rows of raw; rows of up to 2^20 points pinned to numpy on the host"""
    torch = _torch()
    rows = raw.shape[0]
    X64 = torch.fft.fft(exact(raw, fmt, torch.complex128), dim=1)
    if n <= 1 << 20:
        for r in sorted({0, rows // 2, rows - 1}):
            ref = np.fft.fft(_unpack64_host(raw[r].cpu().numpy(), fmt))
            dev = X64[r].cpu().numpy()
            assert np.abs(dev - ref).max() <= 1e-12 * max(1e-300, np.sqrt(np.mean(np.abs(ref) ** 2))), (n, fmt, r)
    return X64


def case(n, fmt, count):
    """{"raw": device input (rows, n) in the plan's format, "rows", "plain": the plain transform once run,
    "X64": its f64 spectra once x64() has made them}"""
    key = (n, fmt, count)
    if key in _CASE:
        return _CASE[key]
    _free_case()
    rows = batch_count(n, count, fmt == "f32")
    seed = (1000003 * n + 10 * list(ES).index(fmt) + ["1", "ragged", "slabs", "many"].index(count)) % (1 << 62)
    raw = make_input(n, fmt, rows, seed)
    _CASE[key] = {"raw": raw, "rows": rows, "plain": None, "X64": None, "n": n, "fmt": fmt}
    return _CASE[key]


def x64(c):
    if c["X64"] is None:
        c["X64"] = reference(c["raw"], c["fmt"], c["n"])
    return c["X64"]


def run_dev(p, inp, rows, out_offset=0):
    """exec_dev into a fresh output of rows * out_len + GUARD c64 at `out_offset` bytes past a 256-byte boundary,
    filled with SENTINEL; asserts the guard survived; returns the (rows, out_len) complex64 output"""
    torch = _torch()
    used = rows * p.out_len
    buf = torch.full((2 * (used + GUARD) + 2,), SENTINEL, dtype=torch.int32, device=DEV)
    out = buf[out_offset // 4:out_offset // 4 + 2 * (used + GUARD)].view(torch.complex64)
    p.exec_dev(inp, rows, out)
    sync()
    assert bool((bits(out[used:]) == SENTINEL).all()), "write past the output"
    return out[:used].view(rows, p.out_len)


def errors(got, X64, n, shift=False, norm=False, rfft=False):
    """rms_rel, max_rel and peak of each row of got (fft_bars.py) against X64 with the flags applied in f64 (shift:
    out[j] = X[(j - n/2) mod n]; rfft: bins 0 ... n - n/2 - 1; norm: times the plan's f32 1/sqrt n), rms(X64) over all n
    bins.  A NaN fails every bar; a row of X64 that is all zero (u8 samples that are all 128) must be matched exactly."""
    torch = _torch()
    rows, out_len = got.shape
    e2s = torch.zeros(rows, dtype=torch.float64, device=DEV)
    e2m, p2m, p2s = torch.zeros_like(e2s), torch.zeros_like(e2s), torch.zeros_like(e2s)
    step = max(1, CHUNK // rows)
    for c0 in range(0, n, step):
        x = X64[:, c0:c0 + step]
        p2s += (x.real ** 2 + x.imag ** 2).sum(dim=1)
    for c0 in range(0, out_len, step):
        k = torch.arange(c0, min(out_len, c0 + step), device=DEV)
        if shift and not rfft:
            k = (k - n // 2) % n
        want = X64.index_select(1, k)
        d = got[:, c0:c0 + k.numel()].to(torch.complex128) - (want * plan_norm(n) if norm else want)
        e2 = d.real ** 2 + d.imag ** 2
        del d
        e2s += e2.sum(dim=1)
        e2m = torch.maximum(e2m, e2.max(dim=1).values)
        p2m = torch.maximum(p2m, (want.real ** 2 + want.imag ** 2).max(dim=1).values)
        del e2, want
    mean = p2s / n
    ms = mean * plan_norm(n) ** 2 if norm else mean  # rms(X64)^2 of the flagged spectrum

    def rel(e):
        r = torch.where(ms > 0, torch.sqrt(e / ms), torch.where(e == 0, torch.zeros_like(e), torch.ones_like(e)))
        return torch.nan_to_num(r, nan=1.0)

    return rel(e2s / out_len), rel(e2m), torch.where(mean > 0, torch.sqrt(p2m / mean), torch.zeros_like(mean))


def check_bars(fmt, n, got, X64, shift=False, norm=False, rfft=False, what=""):
    """holds every row to the path's f64 bars, and records the path's worst errors for the report"""
    rms, mx, peak = errors(got, X64, n, shift, norm, rfft)
    b_rms, b_max, b_peak = B.bars(n, rfft)
    allowed = b_max + b_peak * peak
    r_rms, r_mx = int(rms.argmax()), int((mx / allowed).argmax())
    rms, mx, allowed, pk = float(rms[r_rms]), float(mx[r_mx]), float(allowed[r_mx]), float(peak[r_mx])
    w = WORST.setdefault((B.path(n, rfft), fmt), {"rms": (0.0,), "max": (0.0,)})
    if rms / b_rms > w["rms"][0]:
        w["rms"] = (rms / b_rms, rms, b_rms, n)
    if mx / allowed > w["max"][0]:
        w["max"] = (mx / allowed, mx, allowed, n)
    where = "%s %s n=%d %s (rows %d, %d)" % (kernel_of(n, rfft), fmt, n, what, r_rms, r_mx)
    assert rms <= b_rms, "%s: rms_rel %.3g > %.3g" % (where, rms, b_rms)
    assert mx <= allowed, "%s: max_rel %.3g > %.3g (peak %.1f)" % (where, mx, allowed, pk)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    _free_case()
    if WORST:
        print("\nworst f64 error per path and input format, next to its bar (fft_bars.py; max: with the peak term):")
        for (p, f), w in sorted(WORST.items()):
            (_, r, rb, rn), (_, m, mb, mn) = w["rms"], w["max"]
            print("  %-9s %-5s rms_rel %.3e (bar %.3e, n=%d)  max_rel %.3e (bar %.3e, n=%d)" % (p, f, r, rb, rn, m, mb,
                                                                                              mn))


def _plain(sdr, n, fmt, count):
    c = case(n, fmt, count)
    if c["plain"] is None:
        c["plain"] = run_dev(plan(sdr, n, fmt), c["raw"], c["rows"])
    return c["plain"]


def scaled(x, n):
    torch = _torch()
    return torch.view_as_complex(torch.view_as_real(x) * torch.tensor(plan_norm(n), dtype=torch.float32, device=DEV))


# ---- every length, format, flag and count against f64, and exactly against the plain transform ---------------------
def _variants(n, count):
    if n <= SMALL:
        return list(VARIANTS)
    if n <= HUGE:
        return SOME_VARIANTS if count == "1" else ["u8", "c64-shift-norm", "f32-rfft-norm"]
    return HUGE_VARIANTS if count == "1" else ["u8"]


def _cases():
    out = []
    for n in DIRECT_N:
        for count in ("1", "ragged", "many"):
            out += [(n, v, count) for v in VARIANTS]
    for n in BLUESTEIN_N + FOURSTEP_N:
        for count in ("1", "ragged", "slabs") if n <= SMALL else ("1", "slabs"):
            if batch_count(n, count) * n <= 1 << 27:
                out += [(n, v, count) for v in _variants(n, count)]
    for n in RFFT_MODE3_N:
        out += [(n, v, count) for count in ("1", "slabs") for v in ("f32-rfft", "f32-rfft-norm")]
    return out


@pytest.mark.parametrize("n,variant,count", _cases())
def test_path_against_f64_and_plain(sdr, n, variant, count):
    """f64 bars on every transform; shift = roll(plain, n/2), norm = f32(plain) * f32(1/sqrt n) and rfft = the first
    n - n/2 bins of the plain f32 transform, bit for bit; the rfft flag makes shift a no-op; host exec = exec_dev"""
    torch = _torch()
    fmt, shift, norm, rfft = VARIANTS[variant]
    c = case(n, fmt, count)
    X64 = x64(c)
    if n > HUGE:
        torch.cuda.empty_cache()  # the plan's scratch is 4 GiB at 2^27: leave no cached blocks beside it
    p = plan(sdr, n, fmt, shift, norm, rfft)
    got = run_dev(p, c["raw"], c["rows"])
    if n > HUGE:
        p.close()
    check_bars(fmt, n, got, X64, shift, norm, rfft, variant)
    del X64
    if shift or norm or rfft:
        plain = _plain(sdr, n, fmt, count)
        want = plain[:, :n - n // 2] if rfft else torch.roll(plain, n // 2, dims=1) if shift else plain
        if norm:
            want = scaled(want, n)
        assert same_bits(got, want.contiguous()), (n, variant, count)
        del want
    if rfft:
        assert same_bits(run_dev(plan(sdr, n, fmt, True, norm, True), c["raw"], c["rows"]), got)
    if count != "slabs" and c["rows"] * n <= 1 << 22:
        host = p.exec(c["raw"].cpu().numpy())
        assert np.array_equal(host.view(np.uint32), got.cpu().numpy().view(np.uint32))


# ---- the exact relations at one length per inner kernel, across slabs ---------------------------------------------
# direct DFT; Bluestein at m = 2^8 ... 2^20 and 2^27; four-step at 2^17, 2^20, 2^22, 2^26 (2 transforms: 2 slabs)
REL_N = [3, 8, 60, 127, 257, 1000, 1025, 4095, 8193, 16385, 40000, 100000, 180000, 262145, (1 << 26) - (1 << 20),
         1 << 17, 1 << 20, 1 << 22, 1 << 26]


def _rel_count(n):
    return "many" if B.path(n) == "direct" else "slabs"


def _rel_fmts(n, fmts):
    return fmts if n <= HUGE else fmts[:1]


@pytest.mark.parametrize("n,fmt", [(n, f) for n in REL_N for f in _rel_fmts(n, ["u8iq", "f32"])])
def test_input_formats_agree_with_c64(sdr, n, fmt):
    """u8 = c64 of the exactly unpacked samples, f32 = c64 with zero imaginary part, bit for bit: only the first kernel
    (fft_naive_kernel's load, bluestein_pre, fft_convert) sees the format"""
    torch = _torch()
    c = case(n, fmt, _rel_count(n))
    got = _plain(sdr, n, fmt, _rel_count(n))
    x = exact(c["raw"], fmt, torch.complex64)
    two = run_dev(plan(sdr, n, "c64"), x, c["rows"])
    del x
    assert same_bits(got, two), (n, fmt)


@pytest.mark.parametrize("n,fmt", [(n, f) for n in REL_N for f in _rel_fmts(n, ["u8iq", "c64", "f32"])])
def test_unaligned_input_and_output(sdr, n, fmt):
    """the input one element past a 16-byte boundary and the output 8 bytes past one: bit-identical to the aligned call
    (the slab loop's input and output offsets are computed from these addresses)"""
    torch = _torch()
    c = case(n, fmt, _rel_count(n))
    src = raw_bytes(c["raw"])
    es = ES[fmt]
    buf = torch.empty(src.numel() + 16, dtype=torch.uint8, device=DEV)
    buf[es:es + src.numel()].copy_(src)
    del src
    got = run_dev(plan(sdr, n, fmt), buf.data_ptr() + es, c["rows"], out_offset=8)
    del buf
    assert same_bits(got, _plain(sdr, n, fmt, _rel_count(n))), (n, fmt)


@pytest.mark.parametrize("n,fmt", [(n, f) for n in REL_N for f in _rel_fmts(n, ["u8iq", "c64", "f32"])])
def test_rows_equal_one_transform_calls(sdr, n, fmt):
    """rows at the start, on both sides of every slab boundary and at the end are bit-identical to a 1-transform
    call on the same plan (which also reuses the scratch the long call left behind)"""
    c = case(n, fmt, _rel_count(n))
    R = c["rows"]
    s = slab_of(n) or 4096
    got = _plain(sdr, n, fmt, _rel_count(n))
    p = plan(sdr, n, fmt)
    rows = {0, 1, R - 2, R - 1} | {r for k in (1, 2) for r in (k * s - 1, k * s)}
    for r in sorted(x for x in rows if 0 <= x < R):
        assert same_bits(run_dev(p, c["raw"][r:r + 1], 1), got[r:r + 1]), (n, fmt, r)


@pytest.mark.parametrize("n,fmt", [(n, f) for n in REL_N for f in _rel_fmts(n, ["u8iq", "c64"])])
def test_second_call_equals_a_fresh_plan(sdr, n, fmt):
    """a call on a plan whose scratch holds another signal's slabs equals a call on a fresh plan: nothing of the
    Bluestein padding, the four-step scratch or the direct DFT's table is left stale"""
    c = case(n, fmt, _rel_count(n))
    R = c["rows"]
    p = plan(sdr, n, fmt)
    other = make_input(n, fmt, R, 99991 + n)
    if fmt == "c64":
        other = other * 100.0  # a different scale: a stale slab shows far outside the bars
    run_dev(p, other, R)
    del other
    assert same_bits(run_dev(p, c["raw"], R), _plain(sdr, n, fmt, _rel_count(n))), (n, fmt)
    # and a short call after the long one
    r = min(R - 1, slab_of(n) or 1)
    assert same_bits(run_dev(p, c["raw"][r:r + 1], 1), _plain(sdr, n, fmt, _rel_count(n))[r:r + 1])


@pytest.mark.parametrize("n,fmt", [(n, f) for n in REL_N if n <= HUGE for f in ["u8iq", "c64", "f32"]])
def test_poisoned_transform_stays_in_its_row(sdr, n, fmt):
    """a NaN in transform r (c64, f32) makes every bin of row r NaN; a changed byte (u8) changes row r; every other row
    is bit-identical to the clean run.  r lies in a later slab and in the last one"""
    torch = _torch()
    c = case(n, fmt, _rel_count(n))
    R = c["rows"]
    plain = _plain(sdr, n, fmt, _rel_count(n))
    s = slab_of(n) or R // 2
    rows = sorted({min(R - 1, s + 1), R - 2})
    raw = c["raw"].clone()
    j = n // 3
    for r in rows:
        if fmt == "u8iq":
            raw[r, 2 * j] ^= 0x55
        elif fmt == "c64":
            raw[r, j] = complex(float("nan"), float("nan"))
        else:
            raw[r, j] = float("nan")
    got = run_dev(plan(sdr, n, fmt), raw, R)
    del raw
    keep = torch.ones(R, dtype=torch.bool, device=DEV)
    keep[rows] = False
    assert same_bits(got[keep], plain[keep])
    for r in rows:
        if fmt == "u8iq":
            assert not same_bits(got[r], plain[r])
        else:
            assert bool((torch.isnan(got[r].real) | torch.isnan(got[r].imag)).all()), (n, fmt, r)


# ---- the host pipeline where a 32 MiB chunk holds one transform ----------------------------------------------------
@pytest.mark.parametrize("n,fmt", [(1 << 23, "c64"), (1 << 24, "u8iq"), ((1 << 22) + (1 << 17), "c64")])
def test_host_exec_one_transform_per_chunk(sdr, n, fmt):
    """exec stages 32 MiB of input per chunk and alternates two buffers; with one transform per chunk each chunk is
    a whole call of the four-step or Bluestein path over the plan's one set of scratch"""
    assert (32 << 20) // (n * ES[fmt]) <= 1
    _free_case()
    raw = make_input(n, fmt, 3, n + 7)
    p = plan(sdr, n, fmt, shift=True, norm=True)
    dev = run_dev(p, raw, 3)
    host = p.exec(raw.cpu().numpy())
    assert np.array_equal(host.view(np.uint32), dev.cpu().numpy().view(np.uint32))
    check_bars(fmt, n, dev, reference(raw, fmt, n), shift=True, norm=True, what="host exec")


# ---- lengths and flags the plan refuses ----------------------------------------------------------------------------
def test_limits(sdr):
    with pytest.raises(sdr.SdrError) as e:
        sdr.FftPlan((1 << 26) + 1, "c64")  # Bluestein would need m = 2^28
    assert e.value.code == 101  # SDR_ERR_UNSUPPORTED
    for fmt in ("u8iq", "c64"):
        for n in (1000, 1 << 17, 7):
            with pytest.raises(sdr.SdrError) as e:
                sdr.FftPlan(n, fmt, rfft=True)
            assert e.value.code == 100  # SDR_ERR_INVALID_ARG


# ---- WindowFft: the gather in front of every path ------------------------------------------------------------------
def frames(x, N, D):
    """the kept windows of the whole stream x (device complex64): window j ends at sample (j + 1) D - 1 and starts
    with the deque's zeros before the stream's first sample"""
    torch = _torch()
    W = x.numel() // D
    padded = torch.cat([torch.zeros(N, dtype=torch.complex64, device=DEV), x])
    return padded.as_strided((W, N), (D, 1), D).contiguous()


def unpacked(raw, fmt):
    torch = _torch()
    return exact(raw.view(1, -1), fmt, torch.complex64).view(-1)


def window_truth(sdr, x, N, D, fmt):
    """(spectra of every window by a c64 FftPlan(N, shift, norm) on windows framed here, f64 spectra of the windows)"""
    torch = _torch()
    f = frames(x, N, D)
    W = f.shape[0]
    want = run_dev(plan(sdr, N, "c64", shift=True, norm=True), f, W) if W else f
    X64 = torch.fft.fft(f.to(torch.complex128), dim=1)
    return want, X64


def stream_input(fmt, n, seed):
    raw = make_input(n, fmt, 1, seed)
    return raw.view(-1)


def feed(wf, raw, fmt, blocks):
    """host process() over consecutive blocks of raw (sample counts), concatenated"""
    per = 2 if fmt == "u8iq" else 1
    host = raw.cpu().numpy()
    out, pos = [], 0
    for b in blocks:
        out.append(wf.process(host[per * pos:per * (pos + b)]))
        pos += b
    assert pos * per == host.size
    return np.concatenate(out)


WINDOW_CASES = [(60, 7), (60, 60), (60, 97), (1024, 256), (1024, 1024), (1024, 1500), (16384, 4096), (16384, 16384),
                (16384, 20000), (1000, 333), (1000, 1000), (1000, 2500), (40000, 10000), (40000, 40000),
                (40000, 50001), (1 << 17, 30000), (1 << 17, 1 << 17), (1 << 17, 150000)]


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("N,D", WINDOW_CASES)
def test_window_every_window(sdr, N, D, fmt):
    """every window of a stream fed in calls of 0 samples, calls that complete no window and calls that complete
    several equals FftPlan(N, "c64", shift, norm) on numpy-style framed windows bit for bit, and meets the f64 bars"""
    torch = _torch()
    _free_case()
    n = 20 * D + D // 3 + 5
    raw = stream_input(fmt, n, N + D)
    x = unpacked(raw, fmt)
    want, X64 = window_truth(sdr, x, N, D, fmt)
    first = D // 2  # completes no window
    blocks = [0, first, 0, 3 * D + 1, 1, 0, n - first - 3 * D - 2]
    wf = sdr.WindowFft(N, D, fmt)
    got = feed(wf, raw, fmt, blocks)
    assert got.shape == (n // D, N)
    assert np.array_equal(got.view(np.uint32), want.cpu().numpy().view(np.uint32))
    check_bars("c64" if fmt == "c64" else "u8iq", N, torch.from_numpy(got).to(DEV), X64, shift=True, norm=True,
               what="window D=%d" % D)


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("N", [16, 1])
def test_window_call_of_more_than_65535_windows(sdr, N, fmt):
    """one call that completes 70000 windows gathers them in two launches (65535 windows each at most): the second
    chunk's windows follow the first's"""
    torch = _torch()
    _free_case()
    n, D = 70000, 1
    raw = stream_input(fmt, n, 70000 + N)
    x = unpacked(raw, fmt)
    want, X64 = window_truth(sdr, x, N, D, fmt)
    wf = sdr.WindowFft(N, D, fmt)
    got = feed(wf, raw, fmt, [n])
    assert got.shape == (n, N)
    assert np.array_equal(got.view(np.uint32), want.cpu().numpy().view(np.uint32))
    if N > 1:
        check_bars(fmt, N, torch.from_numpy(got).to(DEV), X64, shift=True, norm=True, what="window D=1")
    else:
        assert np.array_equal(got[:, 0], x.cpu().numpy())  # a 1-point transform is the sample itself


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("N,D", [(1000, 333), (1 << 17, 40000), (60, 60)])
def test_window_process_dev_unaligned_input_and_refused_call(sdr, N, D, fmt):
    """process_dev with the input one element past a 16-byte boundary equals host process() of a fresh handle; a call
    refused with SDR_ERR_OUTPUT_TOO_SMALL changes nothing, so the stream goes on as if it had not been made"""
    torch = _torch()
    _free_case()
    n = 9 * D + 17
    raw = stream_input(fmt, n, 3 * N + D)
    want = feed(sdr.WindowFft(N, D, fmt), raw, fmt, [n])
    es = ES[fmt]
    src = raw_bytes(raw)
    buf = torch.empty(src.numel() + 16, dtype=torch.uint8, device=DEV)
    buf[es:es + src.numel()].copy_(src)
    base = buf.data_ptr() + es
    wf = sdr.WindowFft(N, D, fmt)
    out = torch.full((2 * (n // D + 1) * N,), SENTINEL, dtype=torch.int32, device=DEV)
    sync()  # the handle runs on a stream of its own
    pos, done = 0, 0
    for b in (D + 3, 4 * D, n - 5 * D - 3):
        nw = wf.output_count(b)
        assert nw > 0
        with pytest.raises(sdr.SdrError) as e:
            wf.process_dev(base + es * pos, b, out.data_ptr(), nw - 1)
        assert e.value.code == 104  # SDR_ERR_OUTPUT_TOO_SMALL
        assert wf.output_count(b) == nw
        dst = out.view(torch.complex64)[done * N:]
        assert wf.process_dev(base + es * pos, b, dst, nw) == nw
        pos += b
        done += nw
    sync()
    got = out.view(torch.complex64)[:done * N].cpu().numpy().reshape(done, N)
    assert bool((out[2 * done * N:] == SENTINEL).all())
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("N,D", [(1000, 333), (40000, 50001), (60, 7)])
def test_window_reset_mid_stream_equals_a_fresh_handle(sdr, N, D, fmt):
    _free_case()
    n = 6 * D + 11
    a = stream_input(fmt, n, 5 * N + D)
    b = stream_input(fmt, n, 7 * N + D)
    wf = sdr.WindowFft(N, D, fmt)
    per = 2 if fmt == "u8iq" else 1
    feed(wf, a[:per * (n // 2 + 1)], fmt, [n // 2 + 1])  # stops mid-window, with history
    wf.reset()
    got = feed(wf, b, fmt, [D - 1, n - D + 1])
    want = feed(sdr.WindowFft(N, D, fmt), b, fmt, [n])
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
