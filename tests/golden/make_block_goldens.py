#!/usr/bin/env python3
"""Golden data for tests/test_lua_reference.py and tests/test_lua_glue.py that would otherwise need a LuaRadio checkout:

  blocks_ref_executed.npz   the stock PLLBlock (radio/blocks/signal/pll.lua) and FrequencyDiscriminatorBlock
                            (radio/blocks/signal/frequencydiscriminator.lua) executed in this repo's test interpreter on
                            float32-faithful sample cells (tests/lua_reference_env.py), on the inputs the tests use
  reference_hooks.json      the (file, text) pairs of test_lua_glue.GLUE_RELIES_ON that were found in the LuaRadio tree, and
                            the block class names radio/blocks/init.lua registers

    LUARADIO_REFERENCE=<luaradio checkout> python tests/golden/make_block_goldens.py
"""
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

PLL_LUA = """
    local PLLBlock = require('radio.blocks.signal.pll')
    local types = require('radio.types')
    local blk = PLLBlock(100, 18950, 19050, 2)
    blk:differentiate({types.ComplexFloat32})
    blk.inputs[1].pipe = {get_rate = function () return 220500 end}
    blk:initialize()
    return blk
"""
DISC_LUA = """
    local Disc = require('radio.blocks.signal.frequencydiscriminator')
    local types = require('radio.types')
    return function ()
        local blk = Disc(1.25)
        blk:differentiate({types.ComplexFloat32})
        blk:initialize()
        return blk
    end
"""


def pll_input():
    """A 19 011 Hz pilot in noise at 220.5 kHz, 2 x 2400 samples (fed to the PLL in two calls)."""
    rate, n = 220500.0, 2400
    rng = np.random.default_rng(7)
    t = np.arange(2 * n)
    return (0.8 * np.exp(2j * np.pi * 19011.0 / rate * t + 0.4j)
            + 0.05 * (rng.standard_normal(2 * n) + 1j * rng.standard_normal(2 * n))).astype(np.complex64)


def disc_inputs():
    """Three samples each; the first one in each of the four quadrants."""
    return np.array([[complex(re, im), complex(0.1, 0.4), complex(-0.2, 0.1)]
                     for re, im in ((0.3, 0.2), (-0.3, 0.2), (0.3, -0.2), (-0.3, -0.2))], np.complex64)


def main():
    ref = os.environ.get("LUARADIO_REFERENCE")
    if not ref or not os.path.isdir(ref):
        sys.exit("set LUARADIO_REFERENCE to a LuaRadio checkout")
    os.environ["LUARADIO_DISABLE_CUDA"] = "1"
    from tests import lua_reference_env as E
    from tests.test_lua_glue import GLUE_RELIES_ON

    it, types = E.make_env(lib=None, cuda=False)
    x = pll_input()
    blk = it.run(PLL_LUA)[0]
    outs, errs = [], []
    for part in np.split(x, 2):
        out, err = it.call(it.index(blk, "process"), [blk, it.f32.vector_from_numpy(part)])
        outs.append(it.f32.to_numpy(out))
        errs.append(it.f32.to_numpy(err))
    xd = disc_inputs()
    make = it.run(DISC_LUA)[0]
    yd = []
    for row in xd:
        d = it.call(make, [])[0]
        yd.append(it.f32.to_numpy(it.call(it.index(d, "process"), [d, it.f32.vector_from_numpy(row)])[0]))
    path = os.path.join(GOLDEN, "blocks_ref_executed.npz")
    np.savez_compressed(path, pll_x=x, pll_out=np.concatenate(outs), pll_err=np.concatenate(errs),
                        pll_freq_locked=np.float64(blk.hash["freq_locked"]), disc_x=xd, disc_y=np.array(yd, np.float32))
    print("wrote", path)

    found = [[rel, needle] for rel, needle in GLUE_RELIES_ON if needle in open(os.path.join(ref, rel)).read()]
    missing = [p for p in GLUE_RELIES_ON if list(p) not in found]
    if missing:
        sys.exit("not in the LuaRadio tree: %s" % missing)
    reg = open(os.path.join(ref, "radio", "blocks", "init.lua")).read()
    names = sorted(set(re.findall(r"\b\w+(?:Block|Source|Sink)\b", reg)))
    path = os.path.join(GOLDEN, "reference_hooks.json")
    with open(path, "w") as f:
        f.write('{"found": [\n%s\n],\n"registered_blocks": %s}\n' % (",\n".join(json.dumps(p) for p in found), json.dumps(names)))
    print("wrote", path)


if __name__ == "__main__":
    main()
