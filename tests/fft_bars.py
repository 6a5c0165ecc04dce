"""f64 error bars of the FFT paths, as functions of the length.  test_fft_bars_host.py shows where they come from
(f32 models of each algorithm sit at least 3 times inside them); the GPU tests hold the kernels to them.

Per transform (row), against X64, the f64 transform of the same exactly represented input, with rms(X64) taken over
all n bins (also for rfft, which keeps n - n/2 of them: the kept half of a short real transform can be nearly empty):
    rms_rel = rms_k |X - X64| / rms(X64)      max_rel = max_k |X - X64| / rms(X64)      peak = max_k |X64| / rms(X64)
    rms_rel <= rms bar        max_rel <= max bar + peak coefficient * peak

  path (FftPlan mode, csrc/api.cu)   lengths                                        rms bar              max bar              peak
  power-of-two kernels (0)           2^4 ... 2^16                                   5e-8 log2 n          4e-7 log2 n          0
  four-step (3)                      2^17 ... 2^27; f32 rfft of 2^15, 2^16          5e-8 log2 n          4e-7 log2 n          0
  direct DFT (1)                     n <= 64 and not a power of two >= 16           1e-7 (3 + log2 n)    5e-7 (3 + log2 n)    0
  Bluestein (2)                      every other n up to 2^26, m = 2^ceil(log2(2n - 1)), at least 16
                                                                                    1.2e-7 log2 m        5e-7 log2 m          1e-6

The power-of-two bars are test_gpu_fft_paths.py's.  The direct DFT is a sequential f32 sum of n products, so its error
grows with n from a floor of a few roundings (the f32 twiddle, the product, the norm) at n = 2 or 3; Bluestein runs
three length-m transforms and two chirp products, so its error follows log2 m, not log2 n.  Bluestein also errs in
proportion to each bin itself (about 1.5e-7 of it in the f32 model), which shows where one bin towers over the rest:
u8 samples have a mean of -1/256 (1 + i), so the DC bin of u8 noise is 0.0068 sqrt(n) times rms(X64) -- 55 times at
n = 2^26 -- and the peak term carries it.
"""
import math

POW2_RMS, POW2_MAX = 5e-8, 4e-7          # per log2 n
DIRECT_RMS, DIRECT_MAX = 1e-7, 5e-7      # per (3 + log2 n)
BLUESTEIN_RMS, BLUESTEIN_MAX = 1.2e-7, 5e-7  # per log2 m
BLUESTEIN_PEAK = 1e-6  # times max_k |X64| / rms(X64), added to the max bar
MAX_LOG = 27  # the longest plain transform; Bluestein's m may not exceed it either


def ilog2(n):
    """log2 n for a power of two, else -1"""
    return n.bit_length() - 1 if n > 0 and n & (n - 1) == 0 else -1


def bluestein_m(n):
    m = 16
    while m < 2 * n - 1:
        m <<= 1
    return m


def path(n, rfft=False):
    """the plan mode fft_plan_init picks: "pow2", "fourstep", "direct" or "bluestein" (None: refused)"""
    l = ilog2(n)
    if 4 <= l <= 16 and not (rfft and l >= 15):
        return "pow2"
    if l >= 15:
        return "fourstep" if l <= MAX_LOG else None
    if n <= 64:
        return "direct"
    return "bluestein" if bluestein_m(n) <= 1 << MAX_LOG else None


def bars(n, rfft=False):
    """(rms bar, max bar, peak coefficient) of a length-n transform"""
    p = path(n, rfft)
    if p == "direct":
        s = 3.0 + math.log2(n)
        return DIRECT_RMS * s, DIRECT_MAX * s, 0.0
    if p == "bluestein":
        lm = ilog2(bluestein_m(n))
        return BLUESTEIN_RMS * lm, BLUESTEIN_MAX * lm, BLUESTEIN_PEAK
    if p is None:
        raise ValueError("no FFT plan of length %d" % n)
    return POW2_RMS * ilog2(n), POW2_MAX * ilog2(n), 0.0
