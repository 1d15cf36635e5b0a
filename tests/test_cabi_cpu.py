"""CPU-side checks of the C ABI: the library loads, exports every symbol include/uavsim.h declares,
and fails loudly (no fallback) when there is no CUDA device."""
import ctypes as C
import os
import re
import subprocess

import pytest
import torch

from conftest import ROOT

from marl_uavs_targets_tracking_b200 import _cabi, default_config, params_from_config


def test_library_is_built_and_loads():
    lib = _cabi.load()
    assert lib.uavsim_abi_version() == 1


def test_every_declared_symbol_is_exported_and_bound():
    hdr = open(os.path.join(ROOT, "include", "uavsim.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(uavsim_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 15
    lib = C.CDLL(_cabi.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), "libuavsim.so does not export %s" % name
    assert declared == set(_cabi.SYMBOLS), "ctypes table and header disagree: %s" % (declared ^ set(_cabi.SYMBOLS))


def test_struct_layouts_match_the_header(tmp_path):
    """sizeof() seen by the C compiler == ctypes layout (catches field drift)."""
    src = '#include <stdio.h>\n#include "uavsim.h"\nint main(){printf("%zu %zu %zu\\n", sizeof(UavSimParams), sizeof(UavSimBuffers), sizeof(UavSimPmiWeights));return 0;}'
    exe = str(tmp_path / "uavsim_sizeof")
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=src.encode(), check=True)
    a, b, c = map(int, subprocess.check_output([exe]).split())
    assert (a, b, c) == (C.sizeof(_cabi.UavSimParams), C.sizeof(_cabi.UavSimBuffers), C.sizeof(_cabi.UavSimPmiWeights))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device error path")
def test_no_cpu_fallback():
    lib = _cabi.load()
    p = params_from_config(default_config(), 10, 10, 2000, 2000, 12)
    h = C.c_void_p()
    rc = lib.uavsim_create(C.byref(p), 4, 0, 0, C.byref(h))
    assert rc != 0 and not h.value
    assert b"cuda" in lib.uavsim_last_error().lower()
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment, UavSimError
    with pytest.raises(UavSimError):
        BatchedEnvironment(10, 10, 2000, 2000, 12, n_envs=4)


def test_argument_errors_are_reported():
    lib = _cabi.load()
    assert lib.uavsim_create(None, 4, 0, 0, None) == -1
    assert lib.uavsim_step(None, 0, 0.0, None) == -1
    assert lib.uavsim_bind(None, None) == -1
    assert b"NULL" in lib.uavsim_last_error()


def test_philox_host_build_matches_numpy_reference(tmp_path):
    """csrc/philox.cuh compiled for the host equals tests/philox_ref.py and the Random123 known answers."""
    import numpy as np
    from philox_ref import philox4x32_10, u53
    src = r'''
#include <stdio.h>
#include "philox.cuh"
int main(){ unsigned c[3][4]={{0,0,0,0},{0xffffffffu,0xffffffffu,0xffffffffu,0xffffffffu},{0x243f6a88u,0x85a308d3u,0x13198a2e,0x03707344}};
 unsigned long long k[3]={0ull,0xffffffffffffffffull,0x299f31d0a4093822ull};
 for(int i=0;i<3;i++){Philox4 r=philox4x32_10(c[i][0],c[i][1],c[i][2],c[i][3],k[i]); printf("%08x %08x %08x %08x %.17g\n",r.v[0],r.v[1],r.v[2],r.v[3],philox_u53(r.v[0],r.v[1]));}
 return 0;}'''
    exe = str(tmp_path / "uavsim_philox")
    subprocess.run(["g++", "-x", "c++", "-", "-I", os.path.join(ROOT, "marl_uavs_targets_tracking_b200", "csrc"), "-o", exe], input=src.encode(), check=True)
    lines = subprocess.check_output([exe]).decode().strip().split("\n")
    kat = ["6627e8d5 e169c58d bc57ac4c 9b00dbd8", "408f276d 41c83b0e a20bc7c6 6d5451fd", "d16cfe09 94fdcceb 5001e420 24126ea1"]
    ctrs = [(0, 0, 0, 0, 0), (0xffffffff,) * 4 + (0xffffffffffffffff,), (0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344, 0x299f31d0a4093822)]
    for line, want, c in zip(lines, kat, ctrs):
        assert line.startswith(want)
        r = philox4x32_10(*c)
        assert " ".join("%08x" % int(v) for v in r) == want
        assert float(line.split()[-1]) == float(u53(r[0], r[1]))
