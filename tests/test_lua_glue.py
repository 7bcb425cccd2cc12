"""Static checks of the LuaJIT glue (lua/radio_b200/*.lua).  LuaJIT is not installed in the build image (the glue's logic
is executed under a test interpreter in tests/test_lua_exec.py); these tests make it reviewable as well: the FFI declarations are GENERATED from include/lrb200.h
and must be current, every lrb200_* symbol the Lua code calls must be declared (LuaJIT raises "missing declaration"
otherwise), every helper / method it calls must be defined by the glue or be part of the reference's block API, and the
block structure of every file must balance."""
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LUA = os.path.join(ROOT, "lua", "radio_b200")
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_lua_cdef  # noqa: E402

from luaradio_b200 import _lib  # noqa: E402

# methods of the reference's own classes that the glue calls (radio/core/block.lua:238-390,516-532; radio/core/vector.lua:108-136;
# radio/core/pipe.lua:495-615; radio/core/platform.lua:277-285)
REFERENCE_METHODS = {
    "add_type_signature", "get_input_type", "get_output_type", "get_rate", "differentiate", "resize", "write", "vector",
    "run_once",
}


def lua_files():
    return sorted(f for f in os.listdir(LUA) if f.endswith(".lua"))


def strip_lua(text):
    """Lua source without comments and string literals (long brackets included)."""
    text = re.sub(r"--\[\[.*?\]\]", " ", text, flags=re.S)
    text = re.sub(r"\[\[.*?\]\]", '""', text, flags=re.S)
    text = re.sub(r"--[^\n]*", " ", text)
    text = re.sub(r'"(?:\\.|[^"\\])*"', '""', text)
    text = re.sub(r"'(?:\\.|[^'\\])*'", "''", text)
    return text


def test_cdef_is_generated_from_the_header_and_current():
    assert subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_lua_cdef.py"), "--check"]).returncode == 0, \
        "lua/radio_b200/cdef.lua is stale: run python tools/gen_lua_cdef.py"
    header = gen_lua_cdef.header_statements(open(gen_lua_cdef.HEADER).read())
    body = open(os.path.join(LUA, "cdef.lua")).read()
    body = body[body.index("[[") + 2: body.index("]]")]
    declared = [gen_lua_cdef.normalise(s) for s in body.split(";") if s.strip()]
    assert declared == header                                   # prototypes textually equal after normalisation
    fns = gen_lua_cdef.function_names(header)
    assert sorted(fns) == _lib.EXPORTED_SYMBOLS                  # == what ctypes binds == what the .so exports (test_cpu_host)
    # the two sample types are LuaRadio's own (radio/types): the cdef must not redefine them
    assert "typedef struct {" not in body


def test_every_library_call_in_the_glue_is_declared():
    declared = set(gen_lua_cdef.function_names(gen_lua_cdef.header_statements(open(gen_lua_cdef.HEADER).read())))
    used = {}
    for f in lua_files():
        if f == "cdef.lua":
            continue
        text = strip_lua(open(os.path.join(LUA, f)).read())
        for m in re.finditer(r"\b(lrb200_\w+)\b", text):
            used.setdefault(m.group(1), set()).add(f)
    assert used, "no library calls found: the scan is broken"
    missing = {k: sorted(v) for k, v in used.items() if k not in declared}
    assert not missing, "called from Lua but not in the cdef: %s" % missing
    # the blocks of the hot path are all bound
    for need in ("lrb200_fir_create_crcf", "lrb200_rotator_create", "lrb200_discrim_create", "lrb200_downsample_create",
                 "lrb200_iir_create_rrrf", "lrb200_graph_execute", "lrb200_graph_commit", "lrb200_graph_flush",
                 "lrb200_mulconst_create", "lrb200_upsample_create"):
        assert need in used, need


def test_helpers_and_methods_the_glue_calls_exist():
    texts = {f: strip_lua(open(os.path.join(LUA, f)).read()) for f in lua_files() if f != "cdef.lua"}
    # helpers of radio_b200.platform (module table M) used as b200.<name>
    plat = texts["platform.lua"]
    defined_m = set(re.findall(r"function M\.(\w+)", plat)) | set(re.findall(r"\bM\.(\w+)\s*=", plat)) | \
        set(re.findall(r"\b(\w+)\s*=\s*decl\.constants", plat))
    for f, t in texts.items():
        for name in re.findall(r"\bb200\.(\w+)", t):
            assert name in defined_m, "%s uses b200.%s which radio_b200/platform.lua does not define" % (f, name)
    # methods called with ':' -- defined somewhere in the glue, or part of the reference API
    defined_methods = set()
    for t in texts.values():
        defined_methods |= set(re.findall(r"function \w+(?:\.\w+)*:(\w+)\s*\(", t))
    for f, t in texts.items():
        for obj, name in re.findall(r"\b(\w+(?:\[[^\]]*\])?(?:\.\w+)*):(\w+)\s*\(", t):
            assert name in defined_methods or name in REFERENCE_METHODS, "%s calls %s:%s() which nothing defines" % (f, obj, name)
    # the scheduler hook is really installed, and the block hook really defines make_device_handle
    assert "make_device_handle" in defined_methods
    comp = texts["composite_patch.lua"]
    assert re.search(r"function CompositeBlock:start\(", comp) and re.search(r"function CompositeBlock:_crawl_connections\(", comp)
    assert "composite_patch').install(radio)" in open(os.path.join(LUA, "blocks_patch.lua")).read()
    # module-level functions used inside composite_patch are defined there
    for name in re.findall(r"\bM\.(\w+)\(", comp):
        assert re.search(r"function M\.%s\(" % name, comp), name


def test_lua_block_structure_balances():
    for f in lua_files():
        words = re.findall(r"[A-Za-z_]\w*", strip_lua(open(os.path.join(LUA, f)).read()))
        opens = sum(words.count(w) for w in ("function", "if", "do"))
        assert opens == words.count("end"), "%s: %d block openers vs %d `end`" % (f, opens, words.count("end"))
        assert words.count("repeat") == words.count("until")
        text = strip_lua(open(os.path.join(LUA, f)).read())
        for a, b in ("()", "{}", "[]"):
            assert text.count(a) == text.count(b), "%s: unbalanced %s%s" % (f, a, b)


# (reference file, field or method the glue relies on) -- each pair was found in the LuaRadio tree by
# tests/golden/make_block_goldens.py (tests/golden/reference_hooks.json); a new one is checked there before it is listed
GLUE_RELIES_ON = [
    ("radio/blocks/signal/frequencytranslator.lua", "self.offset"), ("radio/blocks/signal/frequencydiscriminator.lua", "self.gain"),
    ("radio/blocks/signal/downsampler.lua", "self.factor"), ("radio/blocks/signal/iirfilter.lua", "self.b_taps"),
    ("radio/blocks/signal/iirfilter.lua", "self.a_taps"), ("radio/blocks/signal/hilberttransform.lua", "self.hilbert_taps"),
    ("radio/blocks/signal/multiplyconstant.lua", "self.constant"), ("radio/blocks/signal/upsampler.lua", "self.factor"),
    ("radio/blocks/signal/firfilter.lua", "self.taps"), ("radio/blocks/signal/firfilter.lua", "self.use_fft"),
    ("radio/blocks/signal/firfilter.lua", "process_fft_complex_input_real_taps"), ("radio/blocks/signal/iirfilter.lua", "process_complex"),
    ("radio/blocks/signal/multiplyconstant.lua", "process_complex_by_real"),
    ("radio/blocks/sources/iqfile.lua", "self.raw_samples"), ("radio/blocks/sources/iqfile.lua", "self.repeat_on_eof"),
    ("radio/blocks/sources/iqfile.lua", "self.file"), ("radio/blocks/sources/realfile.lua", "self.raw_samples"),
    ("radio/blocks/sinks/iqfile.lua", "self.raw_samples"), ("radio/blocks/sinks/realfile.lua", "self.raw_samples"),
    ("radio/blocks/sinks/wavfile.lua", "self.count"),
    ("radio/core/composite.lua", "function CompositeBlock:_crawl_connections"), ("radio/core/composite.lua", "function CompositeBlock:start"),
    ("radio/core/composite.lua", "function CompositeBlock:_connect_pipes"), ("radio/core/block.lua", "function Block:differentiate"),
    ("radio/core/platform.lua", "platform.load"), ("radio/core/pipe.lua", "function Pipe:write"),
    # multi-port blocks
    ("radio/blocks/signal/multiply.lua", "MultiplyBlock.process_complex"), ("radio/blocks/signal/multiply.lua", "MultiplyBlock.process_real"),
    ("radio/blocks/signal/multiplyconjugate.lua", "function MultiplyConjugateBlock:process(x, y)"),
    ("radio/blocks/signal/add.lua", "function AddBlock:process(x, y)"), ("radio/blocks/signal/subtract.lua", "function SubtractBlock:process(x, y)"),
    ("radio/blocks/signal/delay.lua", "self.num_samples"), ("radio/blocks/signal/delay.lua", "function DelayBlock:initialize"),
    ("radio/blocks/signal/delay.lua", "types.Bit"),
    ("radio/blocks/signal/pll.lua", "self.loop_bw"), ("radio/blocks/signal/pll.lua", "self.freq_min"), ("radio/blocks/signal/pll.lua", "self.freq_max"),
    ("radio/blocks/signal/pll.lua", "self.multiplier"), ("radio/blocks/signal/pll.lua", "return out, err"),
    ("radio/core/block.lua", "self.outputs[i].data_type"), ("radio/core/block.lua", "self.inputs[i].data_type"),
    ("radio/core/block.lua", "function Block:run_once"), ("radio/core/pipe.lua", "self.input = input"),
    ("radio/core/composite.lua", "function CompositeBlock:_prepare_to_run"), ("radio/core/composite.lua", "function CompositeBlock:_initialize"),
    ("radio/core/composite.lua", "return all_connections, evaluation_order"),
]


def test_fields_and_hooks_the_glue_relies_on_exist_in_the_reference():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_hooks.json")) as f:
        hooks = json.load(f)
    found = {tuple(p) for p in hooks["found"]}
    missing = [p for p in GLUE_RELIES_ON if p not in found]
    assert not missing, missing
    # every class the glue patches is registered by the reference (radio/blocks/init.lua, radio/composites/init.lua)
    reg = set(hooks["registered_blocks"])
    glue = open(os.path.join(LUA, "blocks_patch.lua")).read() + open(os.path.join(LUA, "firfilter_patch.lua")).read()
    for cls in set(re.findall(r"radio\.(\w+Block|\w+Source|\w+Sink)\b", glue)) | set(re.findall(r"\b(\w+Block) = \"", glue)):
        assert cls in reg, "%s is not a reference block" % cls


def test_glue_parses_as_lua():
    """Every file of the glue goes through a Lua 5.1 (+ LuaJIT goto) grammar (tests/lua_grammar.py, lark/Earley): a syntax
    error would stop LuaJIT at require() time.  The grammar itself is validated on files of the reference when the
    reference tree is present (they must parse), and on a few deliberately broken chunks (they must not)."""
    import pytest
    from lark.exceptions import LarkError
    from tests.lua_grammar import parse_lua
    for f in lua_files():
        parse_lua(open(os.path.join(LUA, f)).read())
    for bad in ("local x = = 1", "function f() return 1", "if x then y = 1 ende", "x = {1, 2", "lib.foo(,)", "for i = 1 do end"):
        with pytest.raises(LarkError):
            parse_lua(bad)
    ref = os.environ.get("LUARADIO_REFERENCE", "/root/reference")
    if os.path.isdir(ref):
        for rel in ("radio/blocks/signal/firfilter.lua", "radio/core/composite.lua", "radio/core/block.lua", "radio/core/pipe.lua",
                    "radio/blocks/signal/pll.lua", "radio/blocks/sources/iqfile.lua", "radio/composites/wbfmstereodemodulator.lua"):
            parse_lua(open(os.path.join(ref, rel)).read())


def test_glue_has_no_undefined_or_accidental_globals():
    """Scope analysis on the parse tree: every variable the glue reads or writes is a local declared earlier in an enclosing
    scope (`local`, parameters, `self`, loop variables) or a standard Lua / LuaJIT global -- a misspelled local would be a
    silent nil global in never-executed Lua."""
    from tests.lua_grammar import undefined_globals
    for f in lua_files():
        assert undefined_globals(open(os.path.join(LUA, f)).read()) == [], f
    # the analysis does see through to real problems
    assert undefined_globals("local a = 1\nlocal M = {}\n-- names in a comment: foo(bar)\nfunction M.f(x) return a + x - -typo end") == [("typo", 4)]


def test_cdef_text_is_valid_c_in_declaration_order(tmp_path):
    """LuaJIT's ffi.cdef is a C declaration parser: the generated text must be valid C as it stands (every typedef before its
    first use), given only the two sample types radio.types declares.  gcc -fsyntax-only stands in for the FFI parser."""
    import shutil
    import pytest
    if not shutil.which("gcc"):
        pytest.skip("gcc not available")
    from tests.lua_interp import Interp
    cdef = Interp().run(open(os.path.join(LUA, "cdef.lua")).read())[0].hash["cdef"]
    src = tmp_path / "cdef_check.c"
    src.write_text("#include <stddef.h>\n#include <stdint.h>\n"
                   "typedef struct { float real; float imag; } complex_float32_t;\n"      # radio/types/complexfloat32.lua:19-24
                   "typedef struct { float value; } float32_t;\n"                         # radio/types/float32.lua:17-21
                   + cdef + "\nint main(void) { return 0; }\n")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
