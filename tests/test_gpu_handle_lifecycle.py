"""GPU: a clone carries its source's whole stream state and owns its own resources.  For every cloneable handle, on
its own stream and on a torch stream the caller owns: process a first block, clone, close the source, finish the input
on the clone.  The clone's outputs equal, bit for bit, those of a fresh handle fed the same two blocks, and a
caller-owned stream still takes work after the source and the clone are gone."""
import numpy as np
import pytest

import gen

pytestmark = pytest.mark.gpu

TAPS = gen.lowpass_taps(32, 0.1, 1.0)


def _noise(n, seed):
    return gen.complex_noise(n, seed).astype(np.complex64)


def _rows(c, n, seed):
    return _noise(c * n, seed).reshape(c, n)


def _pll_design(sdr):
    return sdr.PllDesign(0.0, 0.035, sdr.BiquadD.LowPass(80000.0, 0.7), sdr.Identity(),
                         sdr.BiquadD.LowPass(20000.0, 0.7))


def _src_blocks():
    x = _noise(6000, 12).view(np.float32).reshape(-1, 2)
    return [x[:2500], x[2500:], x[:0]]  # the empty block flushes the converter


# name -> (make(sdr, stream), the blocks of input, run(handle, block) -> list of output arrays)
CASES = {
    "fir": (lambda sdr, st: sdr.Fir(TAPS, "c64", stream=st),
            lambda: np.split(_noise(20000, 1), [8192]),  # a split on the 4096-output tile grid
            lambda h, b: [h.process(b)]),
    "pll": (lambda sdr, st: sdr.PllBatch([_pll_design(sdr)], 2, 1.8e6, stream=st),
            lambda: np.split(_rows(2, 6000, 2), [2345], axis=1),
            lambda h, b: list(h.process(np.ascontiguousarray(b)))),
    "biquad": (lambda sdr, st: sdr.Biquad(sdr.BiquadD.LowPass(1000.0, 0.7), 48000.0, n_streams=2,
                                          complex_samples=True, stream=st),
               lambda: np.split(_rows(2, 6000, 3), [2345], axis=1),
               lambda h, b: [h.process(np.ascontiguousarray(b))]),
    "src": (lambda sdr, st: sdr.SampleRate(sdr.ConverterType.SincFastest, 2, stream=st),
            _src_blocks,
            lambda h, b: list(h.process(0.5, b, 8192))),
    "pfb": (lambda sdr, st: sdr.Pfb(TAPS, 8, 8, stream=st),
            lambda: np.split(_noise(8000, 4), [2349]),
            lambda h, b: [h.process(b)]),
    "pfs": (lambda sdr, st: sdr.Pfs(TAPS, 8, 8, stream=st),
            lambda: np.split(_rows(900, 8, 5), [301]),
            lambda h, b: [h.process(b)]),
    "ddc": (lambda sdr, st: sdr.Ddc(TAPS, [0.1, -0.2], 1.0, 4, input_format="c64", stream=st),
            lambda: np.split(_noise(8000, 6), [2349]),
            lambda h, b: [h.process(b)]),
    "duc": (lambda sdr, st: sdr.Duc(TAPS, [0.1, -0.2], 1.0, 4, stream=st),
            lambda: np.split(_rows(2, 3000, 7), [1003], axis=1),
            lambda h, b: [h.process(np.ascontiguousarray(b))]),
    "psd": (lambda sdr, st: sdr.Psd(256, 128, 4, fmt="c64", stream=st),
            lambda: np.split(_noise(20000, 8), [5000]),  # mid-group: the clone carries the open accumulator
            lambda h, b: [h.process(b)]),
    "fcfb": (lambda sdr, st: sdr.Fcfb(TAPS, [0.1, -0.2], 1.0, [4, 8], input_format="c64", stream=st),
             lambda: np.split(_noise(20000, 9), [7001]),
             lambda h, b: h.process(b)),
    "fcsb": (lambda sdr, st: sdr.Fcsb(TAPS, [0.1, -0.2], 1.0, [4, 8], stream=st),
             lambda: [[_noise(1000, 10), _noise(500, 11)], [_noise(1500, 12), _noise(750, 13)]],
             lambda h, b: [h.process(b)]),
    "rrb": (lambda sdr, st: sdr.Rrb(TAPS, [3, 2], [2, 5], stream=st),
            lambda: [[_noise(1001, 14), _noise(999, 15)], [_noise(3000, 16), _noise(2500, 17)]],
            lambda h, b: h.process(b)),
}


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8) if a.dtype == np.uint8 else a.view(np.uint32)


@pytest.mark.parametrize("caller_stream", [False, True], ids=["own_stream", "caller_stream"])
@pytest.mark.parametrize("name", list(CASES))
def test_clone_outlives_its_source(sdr, name, caller_stream):
    import torch
    make, blocks, run = CASES[name]
    st = torch.cuda.Stream() if caller_stream else None
    bs = blocks()

    fresh = make(sdr, st)
    run(fresh, bs[0])
    want = [o for b in bs[1:] for o in run(fresh, b)]
    fresh.close()

    src = make(sdr, st)
    run(src, bs[0])
    clone = src.try_clone() if name == "src" else src.clone()
    src.close()
    got = [o for b in bs[1:] for o in run(clone, b)]
    clone.close()

    assert len(got) == len(want)
    for g, w in zip(got, want):
        if np.isscalar(w):
            assert g == w
        else:
            assert np.asarray(g).shape == np.asarray(w).shape
            assert np.array_equal(_bits(g), _bits(w))
    if caller_stream:
        with torch.cuda.stream(st):
            t = torch.arange(4096, device="cuda", dtype=torch.float32) * 2.0
        st.synchronize()
        assert t.sum().item() == 4095.0 * 4096.0
