"""Build / load the C restatement of the reference CPU path (oracle/lr_oracle.c).  Test and baseline
infrastructure only: imported by tests/, __graft_entry__ and bench.py, never by luaradio_b200/."""
import ctypes
import os
import subprocess
import tempfile
from ctypes import POINTER, c_double, c_float, c_int, c_long, c_uint32, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))


def build(native=False, out_dir=HERE):
    target = "liblr_oracle_native.so" if native else "liblr_oracle.so"
    path = os.path.join(out_dir, target)
    src = os.path.join(HERE, "lr_oracle.c")
    if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(src):
        subprocess.run(["make", "-C", HERE, "OUT=" + out_dir, path], check=True, capture_output=True)
    return path


def load(native=False):
    """`native`: the -march=native build, compiled into a temporary directory (removed again once the library is loaded)
    so that a timing run writes nothing into the source tree; the portable build if that compile fails."""
    if native:
        with tempfile.TemporaryDirectory(prefix="lr_oracle_") as d:
            try:
                lib = ctypes.CDLL(build(True, d))
            except Exception:
                lib = ctypes.CDLL(build(False))
    else:
        lib = ctypes.CDLL(build(False))
    lib.lro_wbfm_chain.restype = c_long
    lib.lro_wbfm_chain.argtypes = [c_void_p, c_long, c_uint64, c_void_p, c_int, c_int, c_double, c_float,
                                   c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_long]
    lib.lro_wbfm_chain2.restype = c_long
    lib.lro_wbfm_chain2.argtypes = lib.lro_wbfm_chain.argtypes + [c_int]
    lib.lro_fir_crcf_parallel.restype = None
    lib.lro_fir_crcf_parallel.argtypes = [c_void_p, c_long, c_void_p, c_int, c_void_p, c_int]
    lib.lro_fir_crcf_fft_parallel.restype = None
    lib.lro_fir_crcf_fft_parallel.argtypes = [c_void_p, c_long, c_void_p, c_int, c_void_p, c_int]
    lib.lro_max_threads.restype = c_int
    lib.lro_usable_cpus.restype = c_int
    lib.lro_synth_fm_iq.restype = None
    lib.lro_synth_fm_iq.argtypes = [c_void_p, c_uint64, c_long, c_uint32, c_double, c_double, c_double, c_float, c_float, c_int]
    # streaming overlap-save objects (firfilter.lua:320-398) for the pinning tests
    lib.lro_firfft_new.restype = c_void_p
    lib.lro_firfft_new.argtypes = [c_void_p, c_int, c_int, c_int]
    lib.lro_firfft_free.restype = None
    lib.lro_firfft_free.argtypes = [c_void_p]
    for nm in ("lro_firfft_process_c", "lro_firfft_process_r"):
        getattr(lib, nm).restype = c_long
        getattr(lib, nm).argtypes = [c_void_p, c_void_p, c_long, c_void_p]
    for nm in ("lro_firfft_flush_c", "lro_firfft_flush_r"):
        getattr(lib, nm).restype = c_long
        getattr(lib, nm).argtypes = [c_void_p, c_void_p]
    return lib
