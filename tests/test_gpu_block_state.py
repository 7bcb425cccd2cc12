"""Reset returns every block, fused stage, graph and DAG to the state of a fresh stream.

Each case feeds a seeded stream of amplitude ~10 in ragged chunks, resets, feeds the same chunks again and requires the
second output to equal the first.  A carried buffer that reset misses (FIR history, IIR state, the discriminator's
previous sample, a delay line, the PLL's loop state) or an index it does not rewind (decimation phase, rotator phase)
changes the start of the second stream by far more than the tolerance.  The tolerance is not zero because the
single-pole scan's decoupled look-back may group its partial sums differently from run to run.

Tolerance: |y2 - y1| <= 1e-6 * max(1, ||y1||_inf)."""
import ctypes
import math

import numpy as np
import pytest

from luaradio_b200 import _lib
from oracle import lr_oracle as O

pytestmark = pytest.mark.gpu

N = 250000
CHUNKS = (7, 4099, 100003)          # then the rest of the stream
HOST, DEV = _lib.LRB200_HOST, _lib.LRB200_DEVICE
C64, F32 = np.complex64, np.float32


def chunk_bounds(n):
    cuts = [0]
    for c in CHUNKS:
        cuts.append(min(n, cuts[-1] + c))
    cuts.append(n)
    return list(zip(cuts[:-1], cuts[1:]))


def stream(dtype, seed, n=N):
    rng = np.random.default_rng(seed)
    x = rng.uniform(-10, 10, n)
    if dtype == C64:
        x = x + 1j * rng.uniform(-10, 10, n)
    return x.astype(dtype)


def same_after_reset(feed, reset, x):
    """feed(x) returns one output array, or a tuple of them for several output ports."""
    y1 = feed(x)
    _lib.check(reset(), "reset")
    y2 = feed(x)
    for a, b in zip(y1 if isinstance(y1, tuple) else (y1,), y2 if isinstance(y2, tuple) else (y2,)):
        assert len(a) > 0 and np.all(np.isfinite(a)) and float(np.max(np.abs(a))) > 0
        assert len(b) == len(a)
        tol = 1e-6 * max(1.0, float(np.max(np.abs(a))))
        err = float(np.max(np.abs(a.astype(np.complex128) - b.astype(np.complex128))))
        assert err <= tol, "after reset: max abs err %.3g > %.3g" % (err, tol)


def f32(a):
    return np.ascontiguousarray(a, F32)


def lowpass(m, cutoff):
    return f32(O.firwin_lowpass(m, cutoff))


# ---- single handles in host mode, reset through lrb200_block_reset ---------------------------------------------------
def _fir(kind, m, d):
    def make(lib):
        taps = np.ascontiguousarray(O.firwin_complex_bandpass(m, [0.05, 0.3]), C64) if kind == "cccf" else lowpass(m, 0.8 / d)
        return getattr(lib, "lrb200_fir_create_" + kind)(taps.ctypes.data, m, d, HOST)
    return make


def _iir(kind, b, a):
    def make(lib):
        bb, aa = f32(b), f32(a)
        return getattr(lib, "lrb200_iir_create_" + kind)(bb.ctypes.data, len(bb), aa.ctypes.data, len(aa), HOST)
    return make


def _hilbert(lib):
    taps = lowpass(129, 0.5)
    return lib.lrb200_hilbert_create(taps.ctypes.data, 129, HOST)


SP_B, SP_A = O.singlepole_lowpass_taps(2e3, 48000.0)

SINGLE = {
    "fir_crcf_16": (_fir("crcf", 16, 1), C64, C64),
    "fir_crcf_128_d5": (_fir("crcf", 128, 5), C64, C64),
    "fir_cccf_129": (_fir("cccf", 129, 1), C64, C64),
    "fir_rrrf_133_d5": (_fir("rrrf", 133, 5), F32, F32),
    "fir_crcf_4097": (_fir("crcf", 4097, 1), C64, C64),
    "hilbert_129": (_hilbert, F32, C64),
    "rotator": (lambda lib: lib.lrb200_rotator_create(0.1234567, HOST), C64, C64),
    "discriminator": (lambda lib: lib.lrb200_discrim_create(1.25, HOST), C64, F32),
    "downsampler": (lambda lib: lib.lrb200_downsample_create(5, 8, HOST), C64, C64),
    "iir_single_pole_real": (_iir("rrrf", SP_B, SP_A), F32, F32),
    "iir_single_pole_complex": (_iir("crcf", SP_B, SP_A), C64, C64),
    "iir_general_na3": (_iir("rrrf", [0.2, 0.3, 0.1], [1.0, -1.2, 0.5]), F32, F32),
    "delay_129": (lambda lib: lib.lrb200_delay_create(129, 8, HOST), C64, C64),
}


@pytest.mark.parametrize("case", sorted(SINGLE))
def test_block_reset_restarts_the_stream(case):
    make, in_t, out_t = SINGLE[case]
    lib = _lib.require_device()
    h = _lib.check_handle(make(lib), case)

    def feed(x):
        outs = []
        for a, b in chunk_bounds(len(x)):
            seg = np.ascontiguousarray(x[a:b])
            y = np.zeros(max(1, lib.lrb200_block_max_output(h, b - a)), out_t)
            no = ctypes.c_size_t()
            _lib.check(lib.lrb200_block_execute(h, seg.ctypes.data, b - a, y.ctypes.data, ctypes.byref(no)), case)
            outs.append(y[:no.value].copy())
        return np.concatenate(outs)

    try:
        same_after_reset(feed, lambda: lib.lrb200_block_reset(h), stream(in_t, 1))
    finally:
        lib.lrb200_block_destroy(h)


def test_pll_reset_restarts_the_stream():
    """The PLL's reset state is its start frequency, not zero: two outputs through lrb200_block_execute_multi."""
    lib = _lib.require_device()
    h = _lib.check_handle(lib.lrb200_pll_create(500.0, -2000.0, 2000.0, 1.0, 48000.0, HOST), "pll")

    def feed(x):
        outs, errs = [], []
        for a, b in chunk_bounds(len(x)):
            seg = np.ascontiguousarray(x[a:b])
            y, e = np.zeros(b - a, C64), np.zeros(b - a, F32)
            ins, ys = (ctypes.c_void_p * 1)(seg.ctypes.data), (ctypes.c_void_p * 2)(y.ctypes.data, e.ctypes.data)
            no = ctypes.c_size_t()
            _lib.check(lib.lrb200_block_execute_multi(h, ins, 1, b - a, ys, 2, ctypes.byref(no)), "pll")
            outs.append(y[:no.value].copy())
            errs.append(e[:no.value].copy())
        return np.concatenate(outs), np.concatenate(errs)

    try:
        same_after_reset(feed, lambda: lib.lrb200_block_reset(h), stream(C64, 2))
    finally:
        lib.lrb200_block_destroy(h)


# ---- graphs, reset through lrb200_graph_reset ------------------------------------------------------------------------
def _wbfm_chain(lib):
    import bench
    t1, t2, b, a = bench.chain_taps()
    return [lib.lrb200_rotator_create(bench.TUNE_OFFSET / bench.RATE, DEV),
            lib.lrb200_fir_create_crcf(t1.ctypes.data, 128, 1, DEV),
            lib.lrb200_downsample_create(5, 8, DEV),
            lib.lrb200_discrim_create(2 * math.pi * 1.25, DEV),
            lib.lrb200_fir_create_rrrf(t2.ctypes.data, 128, 1, DEV),
            lib.lrb200_iir_create_rrrf(b.ctypes.data, 2, a.ctypes.data, 2, DEV),
            lib.lrb200_downsample_create(5, 4, DEV)]


def _audio_tail(m, cutoff, b, a, d):
    def make(lib):
        taps, bb, aa = lowpass(m, cutoff), f32(b), f32(a)
        return [lib.lrb200_fir_create_rrrf(taps.ctypes.data, m, 1, DEV),
                lib.lrb200_iir_create_rrrf(bb.ctypes.data, 2, aa.ctypes.data, 2, DEV),
                lib.lrb200_downsample_create(d, 4, DEV)]
    return make


def _rot_cccf_down(lib):
    taps = np.ascontiguousarray(O.firwin_complex_bandpass(128, [0.05, 0.3]), C64)
    return [lib.lrb200_rotator_create(-0.155, DEV), lib.lrb200_fir_create_cccf(taps.ctypes.data, 128, 1, DEV),
            lib.lrb200_downsample_create(5, 8, DEV)]


def _iir_down(lib):
    b, a = f32(SP_B), f32(SP_A)
    return [lib.lrb200_iir_create_crcf(b.ctypes.data, 2, a.ctypes.data, 2, DEV), lib.lrb200_downsample_create(5, 8, DEV)]


def _resampler(up, down, scale):
    def make(lib):
        m = 24 * max(up, down)
        taps = lowpass(m, 1.0 / max(up, down))
        blocks = [lib.lrb200_mulconst_create(float(up), 0.0, 1, 0, DEV)] if scale else []
        blocks += [lib.lrb200_upsample_create(up, 8, DEV), lib.lrb200_fir_create_crcf(taps.ctypes.data, m, 1, DEV)]
        return blocks + ([lib.lrb200_downsample_create(down, 8, DEV)] if down > 1 else [])
    return make


DEEMPH_750US = O.fm_deemphasis_taps(750e-6, 220500.0)
GRAPHS = {
    # name: (blocks, input type, output type, what the fused graph must look like)
    "wbfm_chain": (_wbfm_chain, C64, F32, lambda d: d.startswith("tuner+discrim(128,/5)") and "+pole" in d),
    "audio_tail_slow_pole": (_audio_tail(128, 15e3 / 110250.0, *DEEMPH_750US, 5), F32, F32,
                             lambda d: d == "fir*iir1_rrrf(133,/5)[fused x3] | pole_rrrf"),
    "audio_tail_64_d4": (_audio_tail(64, 5e3 / 24e3, SP_B, SP_A, 4), F32, F32,
                         lambda d: d.count("|") == 1 and d.endswith("[fused x2]") and "pole" not in d),
    "rotator_cccf_d5": (_rot_cccf_down, C64, C64, lambda d: d == "rot+fir_cccf[fused x3]"),
    "iir_d5": (_iir_down, C64, C64, lambda d: d == "iir_crcf[fused x2]"),
    "interpolator_x2": (_resampler(2, 1, True), C64, C64, lambda d: "|" not in d and "x2" in d),
    "rational_3_2": (_resampler(3, 2, False), C64, C64, lambda d: "|" not in d and "x3/2" in d),
    "rational_4_25": (_resampler(4, 25, False), C64, C64, lambda d: "|" not in d and "x4/25" in d),
}


def make_graph(lib, handles, fuse):
    g = _lib.check_handle(lib.lrb200_graph_create(), "graph")
    for h in handles:
        _lib.check(lib.lrb200_graph_append(g, _lib.check_handle(h, "block")), "graph_append")
    _lib.check(lib.lrb200_graph_commit(g, fuse), "graph_commit")
    return g


@pytest.mark.parametrize("fuse", [1, 0])
@pytest.mark.parametrize("case", sorted(GRAPHS))
def test_graph_reset_restarts_the_stream(case, fuse):
    make, in_t, out_t, fused_ok = GRAPHS[case]
    lib = _lib.require_device()
    g = make_graph(lib, make(lib), fuse)
    desc = lib.lrb200_graph_describe(g).decode()
    if fuse:
        assert fused_ok(desc), desc

    def feed(x):
        outs = []
        for a, b in chunk_bounds(len(x)):
            seg = np.ascontiguousarray(x[a:b])
            y = np.zeros(max(1, lib.lrb200_graph_max_output(g, b - a)), out_t)
            no = ctypes.c_size_t()
            _lib.check(lib.lrb200_graph_execute(g, seg.ctypes.data, b - a, y.ctypes.data, ctypes.byref(no)), case)
            outs.append(y[:no.value].copy())
        return np.concatenate(outs)

    try:
        same_after_reset(feed, lambda: lib.lrb200_graph_reset(g), stream(in_t, 3))
    finally:
        lib.lrb200_graph_destroy(g)


# ---- a device DAG, reset through lrb200_dag_reset --------------------------------------------------------------------
def test_dag_reset_restarts_the_stream():
    """input -> [FIR(64) -> /2, fused graph] -> Delay(129) and PLL -> MultiplyConjugate(delayed, PLL output)."""
    lib = _lib.require_device()
    taps = lowpass(64, 0.4)
    d = _lib.check_handle(lib.lrb200_dag_create(), "dag")
    g = make_graph(lib, [lib.lrb200_fir_create_crcf(taps.ctypes.data, 64, 1, DEV), lib.lrb200_downsample_create(2, 8, DEV)], 1)
    assert "[fused x2]" in lib.lrb200_graph_describe(g).decode()

    def add(h, *refs):
        ins = (ctypes.c_int * len(refs))(*refs)
        node = lib.lrb200_dag_add_block(d, _lib.check_handle(h, "block"), ins, len(refs))
        assert node >= 0, _lib.last_error()
        return node

    try:
        src = lib.lrb200_dag_add_graph(d, g, -1)
        assert src >= 0, _lib.last_error()
        dly = add(lib.lrb200_delay_create(129, 8, DEV), src * 4)
        pll = add(lib.lrb200_pll_create(500.0, -2000.0, 2000.0, 1.0, 48000.0, DEV), src * 4)
        mix = add(lib.lrb200_binary_create(b"multiplyconjugate", 1, DEV), dly * 4, pll * 4)
        outs = [mix * 4, pll * 4 + 1]
        _lib.check(lib.lrb200_dag_set_outputs(d, (ctypes.c_int * 2)(*outs), 2), "dag_set_outputs")

        def feed(x):
            got = ([], [])
            for a, b in chunk_bounds(len(x)):
                seg = np.ascontiguousarray(x[a:b])
                ys = [np.zeros(max(1, lib.lrb200_dag_max_output(d, k, b - a)), t) for k, t in enumerate((C64, F32))]
                no = (ctypes.c_size_t * 2)()
                _lib.check(lib.lrb200_dag_execute(d, seg.ctypes.data, b - a, (ctypes.c_void_p * 2)(*[y.ctypes.data for y in ys]),
                                                  no), "dag_execute")
                for k in range(2):
                    got[k].append(ys[k][:no[k]].copy())
            return tuple(np.concatenate(v) for v in got)

        same_after_reset(feed, lambda: lib.lrb200_dag_reset(d), stream(C64, 4))
    finally:
        lib.lrb200_dag_destroy(d)
