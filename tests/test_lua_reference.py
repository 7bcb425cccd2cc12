"""The glue in lua/radio_b200/ run against the REFERENCE'S OWN Lua code: radio/core/{class,util,block,composite}.lua and the
real block / composite files of the hot path are loaded from the reference tree into the test interpreter
(tests/lua_reference_env.py; mocks only for ffi, pipes, platform, types), the glue is installed the way INTEGRATION.md says
(`require('radio_b200.blocks_patch')(radio)`), the flow graph of examples/rtlsdr_wbfm_mono.lua is built with the reference's
CompositeBlock:connect, and CompositeBlock:_prepare_to_run() runs for real: differentiate, crawl, pipes, rate validation,
initialize, evaluation order.  The mock library logs what the glue asked of libluaradio_b200.

This is the closest a machine without LuaJIT gets to running the glue; those tests need the LuaRadio tree
(tests/lua_reference_env.py: $LUARADIO_REFERENCE) and skip where it is absent.  The oracle pins at the end compare with
what the reference's own blocks computed, stored under tests/golden/ (tests/golden/make_block_goldens.py), and run
everywhere."""
import numpy as np
import pytest

from tests import lua_reference_env as E
import os
import re

from tests.lua_interp import LuaTable
from tests.test_lua_exec import MockLib, read

needs_reference = pytest.mark.skipif(not E.available(), reason="LuaRadio tree not present (LUARADIO_REFERENCE)")
GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

MOCK_ENDS = """
local block = require('radio.core.block')
local types = require('radio.types')
local Source = block.factory("MockSource")
function Source:instantiate(rate, data_type)
    self.rate = rate
    self:add_type_signature({}, {block.Output("out", data_type or types.ComplexFloat32)})
end
function Source:get_rate() return self.rate end
function Source:process() return nil end
local Sink = block.factory("MockSink")
function Sink:instantiate(data_type) self:add_type_signature({block.Input("in", data_type or types.Float32)}, {}) end
function Sink:process(x) end
return {Source = Source, Sink = Sink}
"""


def env(monkeypatch):
    monkeypatch.delenv("LUARADIO_DISABLE_CUDA", raising=False)
    monkeypatch.delenv("LUARADIO_CUDA_DEVICE", raising=False)
    monkeypatch.delenv("LUARADIO_B200_SUPERCHUNK", raising=False)
    from tests.lua_interp import Interp
    cdef = Interp().run(read(os.path.join(E.LUA, "cdef.lua")))[0]
    lib = MockLib(set(re.findall(r"\b(lrb200_\w+)\s*\(", cdef.hash["cdef"])))
    it, types = E.make_env(lib)
    it.modules["mock_ends"] = MOCK_ENDS
    return it, lib, types


def taps_of(it, data, n):
    """float32 cells of a Float32 vector's data (tests/lua_reference_env.py: Float32Types)"""
    return np.array([it.f32._fstore[(id(it.f32.get_cell(data, i)), "value")] for i in range(n)], np.float64)


@needs_reference
def test_reference_classes_load_and_the_glue_patches_them(monkeypatch):
    it, lib, types = env(monkeypatch)
    radio = it.require("radio")
    for name in list(E.REAL_BLOCKS) + list(E.REAL_COMPOSITES) + ["CompositeBlock"]:
        assert isinstance(radio.hash.get(name), LuaTable), name
    it.call(it.require("radio_b200.blocks_patch"), [radio])
    assert it.require("radio.core.platform").hash["features"].hash["cuda"] is True
    b200 = it.require("radio_b200.platform")
    # subclasses made by the reference's class.factory (which CACHES the parent's functions at creation) still reach the GPU
    # form: new methods through the metatable chain, process functions through the explicit FIRFilterBlock.* / IIRFilterBlock.*
    # lookups in instantiate()
    for sub in ("LowpassFilterBlock", "HighpassFilterBlock", "BandpassFilterBlock", "ComplexBandpassFilterBlock"):
        assert it.index(radio.hash[sub], "make_device_handle") is it.index(radio.hash["FIRFilterBlock"], "make_device_handle")
    for sub in ("SinglepoleLowpassFilterBlock", "SinglepoleHighpassFilterBlock", "FMDeemphasisFilterBlock"):
        assert it.index(radio.hash[sub], "make_device_handle") is it.index(radio.hash["IIRFilterBlock"], "make_device_handle")
    lp = it.call(radio.hash["LowpassFilterBlock"], [128, 15e3])[0]
    sigs = lp.hash["signatures"].array()
    assert len(sigs) == 2 and all(s.hash["process_func"] is b200.hash["process"] for s in sigs)
    de = it.call(radio.hash["FMDeemphasisFilterBlock"], [75e-6])[0]
    assert all(s.hash["process_func"] is b200.hash["process"] for s in de.hash["signatures"].array())


@needs_reference
def test_wbfm_mono_example_through_the_reference_prepare_to_run(monkeypatch):
    """examples/rtlsdr_wbfm_mono.lua:11-28 with a mock source and sink: after the reference's own _prepare_to_run() the seven
    concrete blocks are ONE GPUChainBlock, initialised from taps the reference's initialize() methods designed at the rates
    the rate links report."""
    it, lib, types = env(monkeypatch)
    top, conns, order, chain = it.run("""
        local radio = require('radio')
        require('radio_b200.blocks_patch')(radio)
        local ends = require('mock_ends')
        local source = ends.Source(1102500)
        local tuner = radio.TunerBlock(-250e3, 200e3, 5)
        local fm_demod = radio.FrequencyDiscriminatorBlock(1.25)
        local af_filter = radio.LowpassFilterBlock(128, 15e3)
        local af_deemphasis = radio.FMDeemphasisFilterBlock(75e-6)
        local af_downsampler = radio.DownsamplerBlock(5)
        local sink = ends.Sink()
        local top = radio.CompositeBlock()
        top:connect(source, tuner, fm_demod, af_filter, af_deemphasis, af_downsampler, sink)
        local all_connections, evaluation_order = top:_prepare_to_run()
        return top, all_connections, evaluation_order, top._b200_substitutes[1]
    """)
    names = [b.hash["name"] if "name" in b.hash else it.index(b, "name") for b in order.array()]
    assert names == ["MockSource", "GPUChainBlock", "MockSink"]
    assert len(conns.hash) == 2 and top.hash["_b200_substitutes"].length() == 1
    members = [it.index(b, "name") for b in chain.hash["blocks"].array()]
    assert members == ["FrequencyTranslatorBlock", "LowpassFilterBlock", "DownsamplerBlock", "FrequencyDiscriminatorBlock",
                       "LowpassFilterBlock", "FMDeemphasisFilterBlock", "DownsamplerBlock"]
    # every pipe of the collapsed graph was initialised by the reference, the chain reports the final rate
    assert all(i.hash["pipe"].hash["initialized"] for i in conns.hash)
    assert it.call(it.index(chain, "get_rate"), [chain]) == [1102500 / 25]
    # library calls: the probe, then -- no HOST handle for any member -- the chain's graph
    calls = [c[0] for c in lib.calls]
    assert calls[:2] == ["lrb200_device_count", "lrb200_init"]
    creates = ["lrb200_rotator_create", "lrb200_fir_create_crcf", "lrb200_downsample_create", "lrb200_discrim_create",
               "lrb200_fir_create_rrrf", "lrb200_iir_create_rrrf", "lrb200_downsample_create"]
    expect = ["lrb200_graph_create"]
    for c in creates:
        expect += [c, "lrb200_graph_append"]
    assert calls[2:] == expect + ["lrb200_graph_commit"]
    by_name = {}
    for nm, args in lib.calls:
        by_name.setdefault(nm, []).append(args)
    assert all(a[-1] == 1 for nm in creates for a in by_name[nm])                   # DEVICE pointers
    assert by_name["lrb200_rotator_create"][0][0] == pytest.approx(-250e3 / 1102500)
    assert by_name["lrb200_discrim_create"][0][0] == pytest.approx(2 * np.pi * 1.25)       # gain = 2 pi modulation_index, as the header says
    assert [a[:2] for a in by_name["lrb200_downsample_create"]] == [(5, 8), (5, 4)]
    # the taps are the reference's own designs (filter_utils.lua run by the interpreter) at the right rates
    from luaradio_b200.utilities import filter_utils as fu
    t1 = taps_of(it, by_name["lrb200_fir_create_crcf"][0][0], 128)
    t2 = taps_of(it, by_name["lrb200_fir_create_rrrf"][0][0], 128)
    assert by_name["lrb200_fir_create_crcf"][0][1] == 128 and by_name["lrb200_fir_create_rrrf"][0][1] == 128
    np.testing.assert_allclose(t1, np.asarray(fu.firwin_lowpass(128, 100e3 / (1102500 / 2)), np.float64), atol=1e-7)
    np.testing.assert_allclose(t2, np.asarray(fu.firwin_lowpass(128, 15e3 / (220500 / 2)), np.float64), atol=1e-7)
    b, n_b, a, n_a, _ = by_name["lrb200_iir_create_rrrf"][0]
    from oracle import lr_oracle as O
    ob, oa = O.fm_deemphasis_taps(75e-6, 220500.0)
    assert (n_b, n_a) == (2, 2)
    np.testing.assert_allclose(taps_of(it, b, 2), ob, rtol=1e-6)
    np.testing.assert_allclose(taps_of(it, a, 2), oa, rtol=1e-6)
    # process() of the chain is what the reference's run loop will call (bound by Block:differentiate)
    patch = it.require("radio_b200.composite_patch")
    assert chain.hash["process"] is patch.hash["GPUChainBlock"].hash["process"]
    assert chain.hash["initialize"] is patch.hash["GPUChainBlock"].hash["initialize"]


@needs_reference
def test_composites_stereo_and_am_synchronous_through_the_reference(monkeypatch):
    """The reference's own WBFMStereoDemodulator and AMSynchronousDemodulator composites: their concrete blocks become one
    GPUDagBlock each, and the reference's rate validation and initialize pass over the members."""
    it, lib, types = env(monkeypatch)
    top, order = it.run("""
        local radio = require('radio')
        local types = require('radio.types')
        require('radio_b200.blocks_patch')(radio)
        local ends = require('mock_ends')
        local top = radio.CompositeBlock()
        local demod = radio.WBFMStereoDemodulator()
        top:connect(ends.Source(220500), demod)
        top:connect(demod, 'left', ends.Sink(), 'in')
        top:connect(demod, 'right', ends.Sink(), 'in')
        local all_connections, evaluation_order = top:_prepare_to_run()
        return top, evaluation_order
    """)
    names = sorted(it.index(b, "name") for b in order.array())
    assert names == ["GPUDagBlock", "MockSink", "MockSink", "MockSource"]
    dag = top.hash["_b200_substitutes"].hash[1]
    assert dag.hash["blocks"].length() == 14 and dag.hash["ext_out"].length() == 2
    calls = [c[0] for c in lib.calls]
    assert calls.count("lrb200_dag_create") == 1 and calls[-1] == "lrb200_dag_set_outputs"
    assert calls.count("lrb200_pll_create") == 1 and calls.count("lrb200_binary_create") == 3 and calls.count("lrb200_delay_create") == 1
    pll = [a for nm, a in lib.calls if nm == "lrb200_pll_create"][0]
    assert pll == (100, 18950.0, 19050.0, 2, 220500, 1)          # wbfmstereodemodulator.lua: PLLBlock(100, 19e3-50, 19e3+50, 2) in Hz, the member's rate, DEVICE
    # AM synchronous
    it, lib, types = env(monkeypatch)
    top, order = it.run("""
        local radio = require('radio')
        require('radio_b200.blocks_patch')(radio)
        local ends = require('mock_ends')
        local top = radio.CompositeBlock()
        top:connect(ends.Source(1e6), radio.AMSynchronousDemodulator(100e3, 5e3), ends.Sink())
        local all_connections, evaluation_order = top:_prepare_to_run()
        return top, evaluation_order
    """)
    assert sorted(it.index(b, "name") for b in order.array()) == ["GPUDagBlock", "MockSink", "MockSource"]
    assert [c[0] for c in lib.calls].count("lrb200_dag_add_graph") >= 1


@needs_reference
def test_without_the_cuda_feature_the_reference_runs_untouched(monkeypatch):
    it, lib, types = env(monkeypatch)
    monkeypatch.setenv("LUARADIO_DISABLE_CUDA", "1")
    order = it.run("""
        local radio = require('radio')
        require('radio_b200.blocks_patch')(radio)
        local ends = require('mock_ends')
        local top = radio.CompositeBlock()
        top:connect(ends.Source(1e6), radio.FrequencyTranslatorBlock(1e5), radio.DownsamplerBlock(2), ends.Sink(require('radio.types').ComplexFloat32))
        top:_validate_inputs()
        top:_differentiate()
        local all_connections = top:_crawl_connections()
        local n = 0
        for _ in pairs(all_connections) do n = n + 1 end
        return n
    """)
    assert order == [3] and lib.calls == []


@needs_reference
def test_reference_run_loop_drives_the_chain(monkeypatch):
    """top:start() through the reference's own start() (forced single-process by the glue), _prepare_to_run() and the
    round-robin run loop (composite.lua:647-707, Block:run_once block.lua:493-556) with mock pipes: every source vector is
    one lrb200_graph_execute on the chain, the sink receives the chain's output vectors, and cleanup() flushes the chain."""
    it, lib, types = env(monkeypatch)
    top, sink, chain = it.run("""
        local radio = require('radio')
        require('radio_b200.blocks_patch')(radio)
        local block = require('radio.core.block')
        local types = require('radio.types')
        local Source = block.factory("CountingSource")
        function Source:instantiate(rate, vectors)
            self.rate, self.left = rate, vectors
            self:add_type_signature({}, {block.Output("out", types.ComplexFloat32)})
        end
        function Source:get_rate() return self.rate end
        function Source:initialize() self.out = types.ComplexFloat32.vector(8192) end
        function Source:process()
            if self.left == 0 then return nil end
            self.left = self.left - 1
            return self.out
        end
        local Sink = block.factory("CountingSink")
        function Sink:instantiate() self:add_type_signature({block.Input("in", types.Float32)}, {}) end
        function Sink:initialize() self.vectors, self.samples = 0, 0 end
        function Sink:process(x) self.vectors, self.samples = self.vectors + 1, self.samples + x.length end
        local sink = Sink()
        local top = radio.CompositeBlock()
        top:connect(Source(1102500, 3), radio.TunerBlock(-250e3, 200e3, 5), radio.FrequencyDiscriminatorBlock(1.25),
                    radio.LowpassFilterBlock(128, 15e3), radio.FMDeemphasisFilterBlock(75e-6), radio.DownsamplerBlock(5), sink)
        top:start()            -- the user script says start() / run(): multiprocess by default in the reference
        return top, sink, top._b200_substitutes[1]
    """)
    calls = [c[0] for c in lib.calls]
    i0 = calls.index("lrb200_graph_commit") + 1
    # three source vectors -> three executes; then the run loop ends on the source's EOF and cleanup() flushes the chain
    assert calls[i0:] == ["lrb200_graph_max_output", "lrb200_graph_execute"] * 3 + ["lrb200_graph_max_output", "lrb200_graph_flush"]
    ex = [a for nm, a in lib.calls if nm == "lrb200_graph_execute"]
    assert all(a[0] is chain.hash["graph"] and a[2] == 8192 for a in ex)
    # the flushed tail (the mock library reports 3 samples) was written to the chain's output pipe after the loop ended, and
    # the sink downstream took one more turn on it before its own cleanup
    assert sink.hash["vectors"] == 4 and sink.hash["samples"] == 3 * 8192 + 3
    out_pipe = chain.hash["outputs"].hash[1].hash["pipes"].hash[1]
    assert out_pipe.hash["queue"] == []


def test_pll_oracle_pinned_against_the_reference_pll_lua_executed():
    """The reference ships no pll_spec, so the oracle's PLL used to be an unpinned restatement.  The reference's OWN
    radio/blocks/signal/pll.lua (instantiate, initialize, the process() loop: VCO, phase detector, loop filter, clamp, wrap)
    was executed statement by statement in the interpreter on float32-faithful sample cells (tests/lua_reference_env.py:
    Float32Types; stored in tests/golden/blocks_ref_executed.npz) and is compared with oracle/lr_oracle.py: PLL on a 19 kHz
    pilot in noise, in two calls (state carried), through acquisition and lock."""
    from oracle import lr_oracle as O
    g = np.load(os.path.join(GOLDEN_DIR, "blocks_ref_executed.npz"))
    rate = 220500.0
    x = g["pll_x"]
    ref = O.PLL(100, 18950, 19050, 2, rate)
    for part, got_out, got_err in zip(np.split(x, 2), np.split(g["pll_out"], 2), np.split(g["pll_err"], 2)):
        exp_out, exp_err = ref.process(part)
        assert np.max(np.abs(got_err - exp_err)) <= 1e-7 and np.max(np.abs(got_out - exp_out)) <= 1e-7
        assert np.array_equal(got_err, exp_err) and np.array_equal(got_out, exp_out)          # the same float32 cells, bit for bit
    # the loop did something: it pulled in from the band centre (19 000 Hz) towards the 19 011 Hz pilot and the error settled
    assert abs(float(np.mean(exp_err[-400:]))) < 0.05 and np.std(exp_err[:200]) > np.std(exp_err[-200:]) * 0.5
    f_locked = float(g["pll_freq_locked"]) * rate / (2 * np.pi)
    assert 19000.5 < f_locked < 19030 and f_locked == pytest.approx(ref.freq * rate / (2 * np.pi), abs=1e-9)


REF_CHAIN = """
    local radio = require('radio')
    local block = require('radio.core.block')
    local types = require('radio.types')
    local Source = block.factory("ArraySource")
    function Source:instantiate(rate, vectors)
        self.rate, self.vectors, self.k = rate, vectors, 0
        self:add_type_signature({}, {block.Output("out", types.ComplexFloat32)})
    end
    function Source:get_rate() return self.rate end
    function Source:process()
        self.k = self.k + 1
        return self.vectors[self.k]            -- nil after the last one: EOF
    end
    local Sink = block.factory("CollectSink")
    function Sink:instantiate() self:add_type_signature({block.Input("in", types.Float32)}, {}) end
    function Sink:initialize() self.got = {} end
    function Sink:process(x)
        -- the upstream block reuses its output vector: copy the cells out
        local copy = types.Float32.vector(x.length)
        for i = 0, x.length - 1 do copy.data[i] = x.data[i] end
        self.got[#self.got + 1] = copy
    end
    return function (vectors)
        local sink = Sink()
        local top = radio.CompositeBlock()
        top:connect(Source(1102500, vectors), radio.TunerBlock(-250e3, 200e3, 5), radio.FrequencyDiscriminatorBlock(1.25),
                    radio.LowpassFilterBlock(128, 15e3), radio.FMDeemphasisFilterBlock(75e-6), radio.DownsamplerBlock(5), sink)
        top:start(false)
        return sink.got
    end
"""


def test_oracle_chain_against_the_reference_chain_executed():
    """SURVEY 8c lists "no full WBFM chain vector" among the gaps the reference's golden vectors leave.  The stock reference
    ran the whole examples/rtlsdr_wbfm_mono.lua chain itself (tests/golden/make_chain_golden.py, REF_CHAIN above): its
    pure-Lua process() branches (the ones it uses without VOLK / liquid: frequencytranslator.lua:91-112,
    firfilter.lua:228-307, downsampler.lua:45-56, frequencydiscriminator.lua:66-90, iirfilter.lua:111-181), its composites,
    its CompositeBlock run loop -- executed in the test interpreter on float32-faithful sample cells, fed in three ragged
    vectors -- and the numpy oracle's chain is compared with what the reference's sink received
    (tests/golden/wbfm_chain_ref_executed.npz).  (The pure-Lua FIR accumulates in float32 cells, the oracle in float64: hence
    a tolerance -- the reference specs' own 1e-6; the measured difference is 4.5e-8.)"""
    from oracle import lr_oracle as O
    g = np.load(os.path.join(GOLDEN_DIR, "wbfm_chain_ref_executed.npz"))
    rate = 1102500.0
    n = 1650
    rng = np.random.default_rng(11)
    t = np.arange(n)
    audio = np.sin(2 * np.pi * 3000.0 / rate * t)
    x = (0.9 * np.exp(1j * (2 * np.pi * 250e3 / rate * t + 2 * np.pi * 75e3 / rate * np.cumsum(audio)))
         + 0.02 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))).astype(np.complex64)
    assert np.array_equal(x, g["x"]) and list(g["splits"]) == [0, 700, 701, n]
    y = g["y"]
    ref = O.Chain(O.tuner(-250e3, 200e3, 5, rate), O.FrequencyDiscriminator(1.25), O.lowpass_filter(128, 15e3, rate / 5, False),
                  O.IIRFilter(*O.fm_deemphasis_taps(75e-6, rate / 5), False), O.Downsampler(5)).process(x)
    assert len(y) == len(ref) == n // 25
    scale = max(1.0, float(np.max(np.abs(ref))))
    err = float(np.max(np.abs(y - ref)))
    print("reference-executed chain vs oracle: max |diff| = %.3g over %d outputs" % (err, len(y)))
    assert err <= 1e-6 * scale, err                                      # measured: 4.5e-8 (float32 rounding of the accumulations)
    assert np.max(np.abs(ref)) > 1e-3                                    # a live signal came out of the filters' transient


@needs_reference
def test_top_spec_topology_through_the_reference_run_loop(monkeypatch):
    """tests/top_spec.lua:14-55's shape: two sources into MultiplyConjugateBlock (two outside feeds: it stays a block of its
    own, HOST-pointer handle, process(x, y) -> lrb200_block_execute_multi), then Lowpass -> FrequencyDiscriminator ->
    DecimatorBlock as one chain; driven by the reference's own run loop."""
    it, lib, types = env(monkeypatch)
    top, sink = it.run("""
        local radio = require('radio')
        require('radio_b200.blocks_patch')(radio)
        local block = require('radio.core.block')
        local types = require('radio.types')
        local Source = block.factory("CountingSource")
        function Source:instantiate(rate, vectors)
            self.rate, self.left = rate, vectors
            self:add_type_signature({}, {block.Output("out", types.ComplexFloat32)})
        end
        function Source:get_rate() return self.rate end
        function Source:initialize() self.out = types.ComplexFloat32.vector(4096) end
        function Source:process()
            if self.left == 0 then return nil end
            self.left = self.left - 1
            return self.out
        end
        local Sink = block.factory("CountingSink")
        function Sink:instantiate() self:add_type_signature({block.Input("in", types.Float32)}, {}) end
        function Sink:initialize() self.vectors = 0 end
        function Sink:process(x) self.vectors = self.vectors + 1 end
        local sink, mixer = Sink(), radio.MultiplyConjugateBlock()
        local top = radio.CompositeBlock()
        top:connect(Source(1e6, 2), 'out', mixer, 'in1')
        top:connect(Source(1e6, 2), 'out', mixer, 'in2')
        top:connect(mixer, radio.LowpassFilterBlock(16, 100e3), radio.FrequencyDiscriminatorBlock(5), radio.DecimatorBlock(25, {num_taps = 16}), sink)
        top:start()
        return top, sink
    """)
    subs = top.hash["_b200_substitutes"].array()
    assert len(subs) == 1 and [it.index(b, "name") for b in subs[0].hash["blocks"].array()] == \
        ["LowpassFilterBlock", "FrequencyDiscriminatorBlock", "LowpassFilterBlock", "DownsamplerBlock"]
    calls = [c[0] for c in lib.calls]
    assert calls.count("lrb200_binary_create") == 1
    create = [a for nm, a in lib.calls if nm == "lrb200_binary_create"][0]
    assert create == ("multiplyconjugate", 1, 0)                          # its own HOST-pointer handle
    assert calls.count("lrb200_block_execute_multi") == 2 and calls.count("lrb200_graph_execute") == 2
    em = [a for nm, a in lib.calls if nm == "lrb200_block_execute_multi"][0]
    assert em[2] == 2 and em[3] == 4096 and em[5] == 1
    assert calls[-2:] == ["lrb200_graph_max_output", "lrb200_graph_flush"] and sink.hash["vectors"] == 3      # two vectors + the flushed tail


def test_discriminator_first_sample_signed_zero_artefact():
    """frequencydiscriminator.lua:33,72: the first sample is multiplied by conj(ComplexFloat32()) and atan2f sees a product of
    signed zeros -- pi / gain when both parts of the first sample are negative, 0 in the three other quadrants.  The
    reference's own pure-Lua process() executed on float32-faithful cells (stored in tests/golden/blocks_ref_executed.npz),
    the oracle, and (on the GPU) both the stand-alone and the fused discriminator must agree on it
    (tests/test_gpu_stream.py::test_wbfm_mono_chain_reference_executed_golden*)."""
    from oracle import lr_oracle as O
    g = np.load(os.path.join(GOLDEN_DIR, "blocks_ref_executed.npz"))
    gain = 2 * np.pi * 1.25
    for (re, im, first), x, got in zip(((0.3, 0.2, 0.0), (-0.3, 0.2, 0.0), (0.3, -0.2, 0.0), (-0.3, -0.2, np.pi / gain)),
                                       g["disc_x"], g["disc_y"]):
        assert np.array_equal(x, np.array([complex(re, im), complex(0.1, 0.4), complex(-0.2, 0.1)], np.complex64))
        exp = O.FrequencyDiscriminator(1.25).process(x)
        assert np.max(np.abs(got - exp)) <= 3e-8, (re, im, got, exp)          # one float32 ulp in the gain scaling
        assert abs(float(got[0]) - first) <= 1e-7 and abs(float(exp[0]) - first) <= 1e-7, (re, im, got[0], exp[0])


@needs_reference
def test_entry_point_module(monkeypatch):
    """require('radio_b200')(radio): true with the backend active and the classes patched, false (and nothing touched) with the
    kill switch."""
    it, lib, types = env(monkeypatch)
    active, has = it.run("""
        local radio = require('radio')
        local active = require('radio_b200')(radio)
        return active, radio.DownsamplerBlock.make_device_handle ~= nil
    """)
    assert active is True and has is True
    monkeypatch.setenv("LUARADIO_DISABLE_CUDA", "1")
    it, lib, types = env(monkeypatch)
    monkeypatch.setenv("LUARADIO_DISABLE_CUDA", "1")
    active, has = it.run("""
        local radio = require('radio')
        local active = require('radio_b200')(radio)
        return active, radio.DownsamplerBlock.make_device_handle ~= nil
    """)
    assert active is False and has is False and lib.calls == []
