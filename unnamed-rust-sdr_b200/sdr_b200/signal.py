"""Host-side mirror of the reference's stream abstraction (src/signal/mod.rs:13-123) with the
GPU operators behind the adaptors.  The reference pulls one sample at a time (`next()`); a GPU
needs blocks, so every Signal here exposes `next_block(n)` (at most n samples, empty = end of
stream) and the adaptors batch exactly where the reference's own chunked adaptor does
(src/signal/adapters/resample.rs:38-82).  Sample-for-sample the streams are the same.

    signal::from_iter            -> from_array(rate, samples)
    rtltcp::RtlTcpSignal         -> from_u8iq(rate, bytes)       (unpack fused into the consumer)
    Signal::filter(taps)         -> Filter   (GPU Fir; PllDesign -> (value, locked) pairs)
    Signal::decimate(rate)       -> Decimate (fused into a preceding FIR: only kept outputs computed)
    Signal::resample[_with]      -> Resample (SampleRate on the GPU, 4096-frame chunks)
    Signal::take / skip / block / map / iter

Two ways to pull a chain.  `next_block(n)` / `collect()` return numpy arrays: every adaptor hops
through host memory, like the reference's per-sample chain.  `next_block_dev(n, ctx)` /
`collect_dev()` keep every intermediate in HBM (SURVEY 8(f) row 1): blocks travel between the
adaptors as CUDA tensors on one stream (`DeviceCtx`), the operators run through their `*_dev`
entry points, and only the sink decides when (if ever) samples come back to the host.  Both ways
run the same kernels on the same blocks, so they return the same samples bit for bit.
"""
import collections

import numpy as np

from . import ops
from ._ffi import FMT_C64, FMT_F32, FMT_U8IQ

DEFAULT_BLOCK = 1 << 20


class DeviceCtx:
    """Where a device-resident chain lives: one CUDA device and one stream.  torch is used for nothing but
    device memory and the stream handle (the arithmetic is libsdr_b200's)."""

    def __init__(self, device=0, stream=None):
        import torch
        self.torch = torch
        self.index = int(device)
        self.device = torch.device("cuda", self.index)
        self.stream = stream if stream is not None else torch.cuda.current_stream(self.device)

    def upload(self, a):
        a = np.ascontiguousarray(a)
        with self.torch.cuda.stream(self.stream):
            return self.torch.from_numpy(a).to(self.device)

    def empty(self, shape, dtype):
        t = self.torch
        td = {np.dtype(np.complex64): t.complex64, np.dtype(np.float32): t.float32, np.dtype(np.uint8): t.uint8}[np.dtype(dtype)]
        with t.cuda.stream(self.stream):
            return t.empty(shape, dtype=td, device=self.device)

    def cat(self, parts):
        with self.torch.cuda.stream(self.stream):
            return self.torch.cat(parts)

    def download(self, d):
        self.stream.synchronize()
        return d.cpu().numpy()


class Signal:
    def rate(self):
        raise NotImplementedError

    def next_block(self, n):
        raise NotImplementedError

    def next_block_dev(self, n, ctx):
        """at most n samples as a CUDA tensor on ctx.stream.  Default: an adaptor without a device form (e.g. a
        numpy Map) hops through the host once; every adaptor below overrides it."""
        return ctx.upload(self.next_block(n))

    def collect_dev(self, block=DEFAULT_BLOCK, ctx=None, device=0):
        """drain the chain without leaving HBM; returns one CUDA tensor (asynchronous on ctx.stream)"""
        ctx = ctx or DeviceCtx(device)
        parts = []
        while True:
            b = self.next_block_dev(block, ctx)
            if b.shape[0] == 0:
                break
            parts.append(b)
        if not parts:
            return ctx.empty((0,), getattr(self, "dtype", None) or np.complex64)
        return parts[0] if len(parts) == 1 else ctx.cat(parts)

    # ---- combinators (src/signal/mod.rs:18-122) ----
    def block(self, size, dedup=False):
        return Block(self, size, dedup=dedup)

    def decimate(self, rate):
        return Decimate(self, rate)

    def filter(self, design):
        return Filter(self, design)

    def map(self, f):
        return Map(self, f)

    def resample(self, rate):
        return self.resample_with(ops.ConverterType.SincBestQuality, rate)  # mod.rs:83

    def resample_with(self, typ, rate):
        return Resample(self, typ, rate)

    def skip(self, duration):
        return Skip(self, duration)

    def take(self, duration):
        return Take(self, duration)

    def iter(self):
        while True:
            b = self.next_block(DEFAULT_BLOCK)
            if len(b) == 0:
                return
            yield from b

    def collect(self, block=DEFAULT_BLOCK):
        parts = []
        while True:
            b = self.next_block(block)
            if len(b) == 0:
                break
            parts.append(b)
        if not parts:
            return np.empty(0, getattr(self, "dtype", np.complex64))
        return np.concatenate(parts)


class FromArray(Signal):
    """signal::from_iter (src/signal/sources.rs:31-36) over an in-memory array."""

    def __init__(self, rate, samples):
        self._rate = np.float32(rate)
        self.data = np.asarray(samples)
        self.dtype = self.data.dtype
        self.pos = 0

    def rate(self):
        return self._rate

    def next_block(self, n):
        b = self.data[self.pos:self.pos + n]
        self.pos += len(b)
        return b

    def next_block_dev(self, n, ctx):
        return ctx.upload(self.next_block(n))


class FromDevice(Signal):
    """a capture that already sits in HBM (a CUDA tensor of complex64 / float32 samples, or of raw rtl_tcp bytes
    with raw_u8iq=True): the source of a chain that never touches host memory."""

    def __init__(self, rate, tensor, raw_u8iq=False):
        self._rate = np.float32(rate)
        self.t = tensor
        self.is_raw = bool(raw_u8iq)
        self.dtype = np.complex64 if raw_u8iq else {"torch.complex64": np.complex64, "torch.float32": np.float32}[str(tensor.dtype)]
        self.pos = 0  # in samples

    def rate(self):
        return self._rate

    def next_raw_dev(self, n, ctx):
        assert self.is_raw
        b = self.t[2 * self.pos:2 * (self.pos + n)]
        b = b[:b.shape[0] // 2 * 2]
        self.pos += b.shape[0] // 2
        return b

    def next_block_dev(self, n, ctx):
        if self.is_raw:
            raw = self.next_raw_dev(n, ctx)
            out = ctx.empty((raw.shape[0] // 2,), np.complex64)
            if out.shape[0]:
                ops.unpack_u8iq_dev(raw, out.shape[0], out, ctx.index, ctx.stream)
            return out
        b = self.t[self.pos:self.pos + n]
        self.pos += b.shape[0]
        return b

    def next_block(self, n):
        ctx = DeviceCtx(self.t.device.index)
        return ctx.download(self.next_block_dev(n, ctx))

    def next_raw(self, n):
        ctx = DeviceCtx(self.t.device.index)
        return ctx.download(self.next_raw_dev(n, ctx))


class FromU8IQ(Signal):
    """rtl_tcp byte stream (src/rtltcp.rs:151-168).  Consumers that understand u8 IQ (Filter, fft)
    take the raw bytes and unpack on the GPU; anything else gets unpacked complex64."""

    def __init__(self, rate, iq_bytes):
        self._rate = np.float32(rate)
        self.raw = np.ascontiguousarray(iq_bytes, np.uint8)
        self.dtype = np.complex64
        self.pos = 0  # in samples

    def rate(self):
        return self._rate

    def next_raw(self, n):
        b = self.raw[2 * self.pos:2 * (self.pos + n)]
        b = b[:len(b) // 2 * 2]
        self.pos += len(b) // 2
        return b

    def next_block(self, n):
        raw = self.next_raw(n)
        if len(raw) == 0:
            return np.empty(0, np.complex64)
        return ops.unpack_u8iq(raw)

    def next_raw_dev(self, n, ctx):
        return ctx.upload(self.next_raw(n))

    def next_block_dev(self, n, ctx):
        raw = self.next_raw_dev(n, ctx)
        out = ctx.empty((raw.shape[0] // 2,), np.complex64)
        if out.shape[0]:
            ops.unpack_u8iq_dev(raw, out.shape[0], out, ctx.index, ctx.stream)
        return out


def _has_raw(sig):
    """does this upstream hand out raw rtl_tcp bytes (so the consumer can unpack on load)?"""
    return bool(getattr(sig, "is_raw", False)) or isinstance(sig, FromU8IQ) or \
        (isinstance(sig, (Block, Take, Skip)) and _has_raw(sig.signal))


def from_array(rate, samples):
    return FromArray(rate, samples)


def from_u8iq(rate, iq_bytes):
    return FromU8IQ(rate, iq_bytes)


def from_device(rate, tensor, raw_u8iq=False):
    return FromDevice(rate, tensor, raw_u8iq)


class Filter(Signal):
    """signal::Filter (src/signal/adapters/mod.rs:67-100): design_for(&signal) then apply per sample.
    design: taps array (FilterDesign for Vec<C>, fir.rs:44-50) or a PllDesign."""

    def __init__(self, signal, design, decimation=1):
        self.signal = signal
        self.design = design
        self.decimation = decimation
        self.op = None
        if isinstance(design, ops.PllDesign):
            self.kind = "pll"
            self.dtype = np.float32
        else:
            self.kind = "fir"
            taps = np.asarray(design)
            sample_real = np.dtype(getattr(signal, "dtype", np.complex64)).kind == "f"
            self.dtype = np.float32 if sample_real else np.complex64
            self._fmt = "u8iq" if _has_raw(signal) else ("f32" if sample_real else "c64")
            self._taps = taps
        self.locked = None

    def rate(self):
        return self.signal.rate()

    def _ensure(self, ctx=None):
        if self.op is None:
            kw = {} if ctx is None else {"device": ctx.index, "stream": ctx.stream}
            if self.kind == "fir":
                self.op = ops.Fir(self._taps, self._fmt, decimation=self.decimation, **kw)
            else:
                self.op = self.design.design(float(self.signal.rate()), **kw)

    def next_block(self, n):
        self._ensure()
        want = n * self.decimation
        while True:
            if self.kind == "fir" and self._fmt == "u8iq":
                x = self.signal.next_raw(want)
                cnt = len(x) // 2
            else:
                x = self.signal.next_block(want)
                cnt = len(x)
            if cnt == 0:
                return np.empty(0, self.dtype)
            if self.kind == "fir":
                y = self.op.process(x)
                if len(y) == 0:
                    continue  # a short block that produced no kept output: pull again
                return y
            out, locked = self.op.process(x)
            self.locked = locked
            return out

    def next_block_dev(self, n, ctx):
        """the same blocks through sdr_fir_process_dev / sdr_pll_process_dev: input and output stay in HBM"""
        self._ensure(ctx)
        want = n * self.decimation
        while True:
            if self.kind == "fir" and self._fmt == "u8iq":
                x = self.signal.next_raw_dev(want, ctx)
                cnt = x.shape[0] // 2
            else:
                x = self.signal.next_block_dev(want, ctx)
                cnt = x.shape[0]
            if cnt == 0:
                return ctx.empty((0,), self.dtype)
            x = x.contiguous()
            if self.kind == "fir":
                n_out = self.op.output_count(cnt)
                y = ctx.empty((n_out,), self.dtype)
                got = self.op.process_dev(x, cnt, y, max(n_out, 1))
                assert got == n_out
                if n_out == 0:
                    continue
                return y
            out = ctx.empty((cnt,), np.float32)
            locked = ctx.empty((cnt,), np.uint8)
            self.op.process_dev(x, cnt, out, locked)
            self.locked = locked
            return out


class Decimate(Signal):
    """signal::Decimate (src/signal/adapters/mod.rs:14-41).  wait = (rate_in/rate).round() as usize;
    keeps the last sample of every group; rate() still reports the upstream rate (:38-40)."""

    def __init__(self, signal, rate):
        self.wait = ops.decimate_wait(float(signal.rate()), float(rate))
        if self.wait == 0:
            raise ValueError("Decimate: wait == 0 (the reference underflows at adapters/mod.rs:31)")
        self.dtype = getattr(signal, "dtype", np.complex64)
        if isinstance(signal, Filter) and signal.kind == "fir" and signal.op is None and signal.decimation == 1:
            # fuse: the FIR computes only the kept outputs
            self.signal = Filter(signal.signal, signal.design, decimation=self.wait)
            self.fused = True
        else:
            self.signal = signal
            self.fused = False
        self.phase = 0

    def rate(self):
        return self.signal.rate()

    def next_block(self, n):
        if self.fused:
            return self.signal.next_block(n)
        while True:
            x = self.signal.next_block(n * self.wait)
            if len(x) == 0:
                return x
            first = self.wait - 1 - self.phase
            y = x[first::self.wait]
            self.phase = (self.phase + len(x)) % self.wait
            if len(y):
                return y

    def next_block_dev(self, n, ctx):
        if self.fused:
            return self.signal.next_block_dev(n, ctx)
        while True:
            x = self.signal.next_block_dev(n * self.wait, ctx)
            if x.shape[0] == 0:
                return x
            first = self.wait - 1 - self.phase
            with ctx.torch.cuda.stream(ctx.stream):
                y = x[first::self.wait].contiguous()  # a strided device copy: indexing only, no arithmetic
            self.phase = (self.phase + x.shape[0]) % self.wait
            if y.shape[0]:
                return y


class Resample(Signal):
    """signal::Resample (src/signal/adapters/resample.rs:5-86).  buffer_size is the reference's 4096 frames (:21);
    a larger value batches more per SampleRate::process call (identical samples whenever 1/ratio is exactly
    representable -- the positions P + m*step do not depend on where the stream is cut)."""

    def __init__(self, signal, typ, rate, buffer_size=4096):
        self.signal = signal
        self._rate = np.float32(rate)
        self.dtype = getattr(signal, "dtype", np.complex64)
        self.channels = 2 if np.dtype(self.dtype).kind == "c" else 1
        self.typ = typ
        self.sr = None
        self.ratio = float(np.float64(np.float32(rate)) / np.float64(np.float32(signal.rate())))  # :25
        self.buffer_size = int(buffer_size)
        self.buffer = None
        self.done = False
        self.pending = None

    def rate(self):
        return self._rate

    def _chunk(self):
        """one turn of the `while buffer_next >= buffer_resampled.len()` loop (:44-77)"""
        if self.sr is None:
            self.sr = ops.SampleRate(self.typ, self.channels)
            self.buffer = np.empty((0, self.channels), np.float32)
        while True:
            need = self.buffer_size - len(self.buffer)
            if need > 0:
                x = self.signal.next_block(need)
                if len(x):
                    xf = np.ascontiguousarray(x, self.dtype).view(np.float32).reshape(-1, self.channels)
                    self.buffer = np.concatenate([self.buffer, xf])
            used, out = self.sr.process(self.ratio, self.buffer, self.buffer_size)
            if len(self.buffer) == 0 and len(out) == 0:
                self.done = True
                return np.empty(0, self.dtype)
            self.buffer = self.buffer[used:]
            if len(out) == 0:
                continue
            return out.reshape(-1).view(self.dtype) if self.channels == 2 else out.reshape(-1)

    def next_block(self, n):
        if self.pending is None:
            self.pending = np.empty(0, self.dtype)
        if self.done and len(self.pending) == 0:
            return np.empty(0, self.dtype)
        while len(self.pending) == 0 and not self.done:
            self.pending = self._chunk()
        b = self.pending[:n]
        self.pending = self.pending[n:]
        return b

    def _chunk_dev(self, ctx):
        """the same loop with the 4096-frame buffer and the resampled chunk in HBM (sdr_src_process_dev); only the
        two frame counts of SRC_DATA come back to the host, as they do from libsamplerate"""
        t = ctx.torch
        if self.sr is None:
            self.sr = ops.SampleRate(self.typ, self.channels, device=ctx.index, stream=ctx.stream)
            self.buffer = ctx.empty((0, self.channels), np.float32)
        while True:
            need = self.buffer_size - self.buffer.shape[0]
            if need > 0:
                x = self.signal.next_block_dev(need, ctx)
                if x.shape[0]:
                    with t.cuda.stream(ctx.stream):
                        xf = (t.view_as_real(x) if self.channels == 2 else x.reshape(-1, 1)).reshape(-1, self.channels)
                        self.buffer = t.cat([self.buffer, xf]) if self.buffer.shape[0] else xf.contiguous()
            n_in = self.buffer.shape[0]
            out = ctx.empty((self.buffer_size, self.channels), np.float32)
            used, got = self.sr.process_dev(self.ratio, self.buffer if n_in else None, n_in, out, self.buffer_size)
            if n_in == 0 and got == 0:
                self.done = True
                return ctx.empty((0,), self.dtype)
            self.buffer = self.buffer[used:]
            if got == 0:
                continue
            with t.cuda.stream(ctx.stream):
                o = out[:got]
                return t.view_as_complex(o) if self.channels == 2 else o.reshape(-1)

    def next_block_dev(self, n, ctx):
        if self.pending is None:
            self.pending = ctx.empty((0,), self.dtype)
        if self.done and self.pending.shape[0] == 0:
            return ctx.empty((0,), self.dtype)
        while self.pending.shape[0] == 0 and not self.done:
            self.pending = self._chunk_dev(ctx)
        b = self.pending[:n]
        self.pending = self.pending[n:]
        return b


class Take(Signal):
    """signal::Take (adapters/mod.rs:241-268): (rate * duration).round() samples."""

    def __init__(self, signal, duration):
        self.signal = signal
        self.left = ops.duration_samples(float(signal.rate()), float(duration))
        self.dtype = getattr(signal, "dtype", np.complex64)

    def rate(self):
        return self.signal.rate()

    def next_block(self, n):
        n = min(n, self.left)
        if n == 0:
            return np.empty(0, self.dtype)
        b = self.signal.next_block(n)
        self.left -= len(b)
        return b

    def next_raw(self, n):
        n = min(n, self.left)
        if n == 0:
            return np.empty(0, np.uint8)
        b = self.signal.next_raw(n)
        self.left -= len(b) // 2
        return b

    def next_block_dev(self, n, ctx):
        n = min(n, self.left)
        if n == 0:
            return ctx.empty((0,), self.dtype)
        b = self.signal.next_block_dev(n, ctx)
        self.left -= b.shape[0]
        return b

    def next_raw_dev(self, n, ctx):
        n = min(n, self.left)
        if n == 0:
            return ctx.empty((0,), np.uint8)
        b = self.signal.next_raw_dev(n, ctx)
        self.left -= b.shape[0] // 2
        return b


class Skip(Signal):
    """signal::Skip (adapters/mod.rs:166-194)."""

    def __init__(self, signal, duration):
        self.signal = signal
        self.left = ops.duration_samples(float(signal.rate()), float(duration))
        self.dtype = getattr(signal, "dtype", np.complex64)

    def rate(self):
        return self.signal.rate()

    def _drop(self, pull, per):
        while self.left > 0:
            b = pull(min(self.left, DEFAULT_BLOCK))
            if b.shape[0] == 0:
                return False
            self.left -= b.shape[0] // per
        return True

    def next_block(self, n):
        if not self._drop(self.signal.next_block, 1):
            return np.empty(0, self.dtype)
        return self.signal.next_block(n)

    def next_raw(self, n):
        if not self._drop(self.signal.next_raw, 2):
            return np.empty(0, np.uint8)
        return self.signal.next_raw(n)

    def next_block_dev(self, n, ctx):
        if not self._drop(lambda k: self.signal.next_block_dev(k, ctx), 1):
            return ctx.empty((0,), self.dtype)
        return self.signal.next_block_dev(n, ctx)

    def next_raw_dev(self, n, ctx):
        if not self._drop(lambda k: self.signal.next_raw_dev(k, ctx), 2):
            return ctx.empty((0,), np.uint8)
        return self.signal.next_raw_dev(n, ctx)


class _TeeDeque:
    """TeeDeque of adapters/block.rs:7-103: one deque of blocks (newest at the front), one `available` counter per
    reader.  push (:76-89) recycles the oldest block once no reader still needs it; a reader created by clone
    (:92-103) starts with available = data.len(), i.e. it ALSO sees the blocks still held in the deque."""

    def __init__(self):
        self.data = collections.deque()
        self.available = [0]

    def push(self, blk):
        if max(self.available) < len(self.data):
            self.data.pop()  # the reference re-uses this Vec's storage; the contents are overwritten
        self.data.appendleft(blk)
        self.available = [a + 1 for a in self.available]

    def try_pop(self, rid):
        """(:46-58) -> (block or None, blocks still available to this reader after the pop)"""
        if self.available[rid] > 0:
            self.available[rid] -= 1
            i = self.available[rid]
            return self.data[i], i
        return None, 0

    def new_reader(self):
        self.available.append(len(self.data))
        return len(self.available) - 1


class Block(Signal):
    """signal::Block (adapters/block.rs:106-207): the upstream is pulled in blocks of ceil(size * rate) samples
    (:117), one block AHEAD of the reader (target = 1, :171-189) -- the reference fills it on a rayon task, here
    "ahead" means the upstream's kernels for block k+1 are already queued on the stream while block k is served --
    and `clone()` is a tee: readers share one upstream, and each sees every block pushed after it was created plus
    the blocks the deque still held (:92-103, :129-140).

    Faithful to a reference quirk: when a reader moves to a new block, `next` returns `current[0]` WITHOUT advancing
    `i` (:197-199), so the first sample of every block is delivered twice (n+1 samples per n-sample block).
    `dedup=True` delivers each sample once instead (a deliberate divergence; clones inherit it)."""

    def __init__(self, signal, size, dedup=False, _share=None):
        if _share is not None:
            self.__dict__.update(_share)
            self.rid = self.tee.new_reader()
        else:
            self.signal = signal
            self._rate = signal.rate()
            self.block_size = ops.block_samples(float(size), float(signal.rate()))
            self.dtype = getattr(signal, "dtype", np.complex64)
            self.is_raw = _has_raw(signal)
            self.dedup = bool(dedup)
            self.tee = _TeeDeque()
            self.rid = 0
        self.current = None
        self.i = 0

    def clone(self):
        share = {k: getattr(self, k) for k in ("signal", "_rate", "block_size", "dtype", "is_raw", "dedup", "tee")}
        return Block(None, 0.0, _share=share)

    def rate(self):
        return self._rate

    def _fetch(self, pull, length):
        """the else-branch of Block::next (:156-200): try_pop, top the deque up to one block ahead, pop"""
        blk, avail = self.tee.try_pop(self.rid)
        needs_extra = blk is None
        if avail < 1:
            jobs = (1 - avail) + (1 if needs_extra else 0)
            for _ in range(jobs):
                self.tee.push(pull(self.block_size))  # a short or empty block at the end of the stream (:181-185)
            if needs_extra:
                blk, _ = self.tee.try_pop(self.rid)
        self.current, self.i = blk, 0
        return length(blk)

    def _serve(self, n, pull, length, take, cat, empty):
        if self.current is None or self.i >= length(self.current):
            if self._fetch(pull, length) == 0:
                return empty()
            if not self.dedup:
                # (:197-199) current[0] is returned and i stays 0: the next call returns it again
                first = take(self.current, 0, 1)
                rest = take(self.current, 0, min(n - 1, length(self.current)))
                self.i = length(rest)
                return cat([first, rest]) if length(rest) else first
        b = take(self.current, self.i, self.i + n)
        self.i += length(b)
        return b

    def next_block(self, n):
        return self._serve(n, self.signal.next_block, len, lambda b, a, z: b[a:z], np.concatenate,
                           lambda: np.empty(0, self.dtype))

    def next_raw(self, n):
        return self._serve(n, self.signal.next_raw, lambda b: len(b) // 2, lambda b, a, z: b[2 * a:2 * z],
                           np.concatenate, lambda: np.empty(0, np.uint8))

    def next_block_dev(self, n, ctx):
        return self._serve(n, lambda k: self.signal.next_block_dev(k, ctx), lambda b: b.shape[0],
                           lambda b, a, z: b[a:z], ctx.cat, lambda: ctx.empty((0,), self.dtype))

    def next_raw_dev(self, n, ctx):
        return self._serve(n, lambda k: self.signal.next_raw_dev(k, ctx), lambda b: b.shape[0] // 2,
                           lambda b, a, z: b[2 * a:2 * z], ctx.cat, lambda: ctx.empty((0,), np.uint8))


class Map(Signal):
    """signal::Map (adapters/mod.rs:139-163); f is applied to whole blocks (vectorised: numpy arrays on the host
    path, CUDA tensors on the device path)."""

    def __init__(self, signal, f):
        self.signal, self.f = signal, f
        self.dtype = None

    def rate(self):
        return self.signal.rate()

    def next_block(self, n):
        b = self.signal.next_block(n)
        if len(b) == 0:
            return b
        out = self.f(b)
        self.dtype = out.dtype
        return out

    def next_block_dev(self, n, ctx):
        b = self.signal.next_block_dev(n, ctx)
        if b.shape[0] == 0:
            return b
        with ctx.torch.cuda.stream(ctx.stream):
            return self.f(b)


def fft(signal):
    """fft::fft(signal) (src/fft.rs:3-28): drains the signal, one N-point transform."""
    if isinstance(signal, FromU8IQ):
        raw = signal.next_raw(1 << 62)
        n = len(raw) // 2
        if n == 0:
            return np.empty(0, np.float32), np.empty(0, np.complex64)
        plan = ops.FftPlan(n, "u8iq", shift=True, norm=True)
        vals = plan.exec(raw)[0]
        plan.close()
        return ops.fft_labels(n, float(signal.rate())), vals
    x = signal.collect()
    return ops.fft(x, float(signal.rate()))


def rfft(signal):
    """fft::rfft(signal) (src/fft.rs:30-37)."""
    return ops.rfft(signal.collect(), float(signal.rate()))


def fft_dev(signal, ctx=None, device=0):
    """fft::fft(signal) with the drained signal and the spectrum left in HBM: (labels on the host -- they are a
    function of N and the rate only, fft.rs:14-24 -- , CUDA tensor of N shifted, 1/sqrt(N)-scaled bins)."""
    ctx = ctx or DeviceCtx(device)
    x = signal.collect_dev(ctx=ctx).contiguous()
    n = int(x.shape[0])
    if n == 0:
        return np.empty(0, np.float32), ctx.empty((0,), np.complex64)
    plan = ops.FftPlan(n, "c64", shift=True, norm=True, device=ctx.index, stream=ctx.stream)
    out = ctx.empty((n,), np.complex64)
    plan.exec_dev(x, 1, out)
    ctx.stream.synchronize()  # the plan owns scratch that must outlive the launch
    plan.close()
    return ops.fft_labels(n, float(signal.rate())), out


def window_spectra(signal, duration, fps, block=DEFAULT_BLOCK):
    """signal.window(duration).decimate(fps).map(|w| fft::fft(w)) of examples/live.rs:30-39 as a generator of
    (labels, spectra[n_windows, window]) per input block.  window = round(duration * rate) (adapters/mod.rs:279),
    hop = Decimate's wait (mod.rs:22).  Raw u8 IQ sources are unpacked on the device."""
    rate = float(signal.rate())
    window = ops.duration_samples(rate, duration)
    hop = ops.decimate_wait(rate, fps)
    raw = _has_raw(signal)
    wf = ops.WindowFft(window, hop, "u8iq" if raw else "c64")
    labels = ops.fft_labels(window, rate)
    try:
        while True:
            b = signal.next_raw(block) if raw else signal.next_block(block)
            if len(b) == 0:
                return
            s = wf.process(b)
            if len(s):
                yield labels, s
    finally:
        wf.close()


def power_spectra(signal, duration, fps, average, window=None, block=DEFAULT_BLOCK):
    """The power counterpart of window_spectra: signal.window(duration).decimate(fps).map(fft::fft), |.|^2 and the
    mean of `average` consecutive spectra, as a generator of (labels, power[n_spectra, window]) per input block.
    window = round(duration * rate), hop = Decimate's wait, as window_spectra; `window` (the taper) is that many real
    values or None (rectangular).  Raw u8 IQ sources are fed as bytes and unpacked on the device."""
    rate = float(signal.rate())
    n = ops.duration_samples(rate, duration)
    hop = ops.decimate_wait(rate, fps)
    raw = _has_raw(signal)
    psd = ops.Psd(n, hop, average, window, "u8iq" if raw else "c64")
    labels = ops.fft_labels(n, rate)
    try:
        while True:
            b = signal.next_raw(block) if raw else signal.next_block(block)
            if len(b) == 0:
                return
            p = psd.process(b)
            if len(p):
                yield labels, p
    finally:
        psd.close()
