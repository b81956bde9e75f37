"""The catch log and replay-by-index entry points at the C-ABI boundary, without a GPU: the struct mirrors have the C
sizes and offsets, and every new entry point rejects a NULL handle."""
import ctypes as C
import os
import subprocess

from conftest import ROOT
from radiative3d_b200 import abi, engine


def test_catch_structs_match_c(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "r3d_gpu.h"\n'
                   'int main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(r3d_catch), sizeof(r3d_catch_log_desc),'
                   ' offsetof(r3d_catch, seis), offsetof(r3d_catch, bin), offsetof(r3d_catch, type), offsetof(r3d_catch, moves),'
                   ' offsetof(r3d_catch, time), offsetof(r3d_catch, energy), offsetof(r3d_catch_log_desc, seis),'
                   ' offsetof(r3d_catch_log_desc, capacity));'
                   'printf("%llu\\n", (unsigned long long)R3D_CATCH_LOG_MAX);return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    v = list(map(int, out))
    assert v[0] == abi.CATCH_DTYPE.itemsize == 64
    assert v[1] == C.sizeof(abi.CatchLogDesc)
    f = abi.CATCH_DTYPE.fields
    assert v[2:8] == [f["seis"][1], f["bin"][1], f["type"][1], f["moves"][1], f["time"][1], f["energy"][1]]
    assert v[8] == abi.CatchLogDesc.seis.offset and v[9] == abi.CatchLogDesc.capacity.offset
    assert v[10] == abi.R3D_CATCH_LOG_MAX


def test_null_handle_is_rejected():
    L = engine.load_library()
    idx = (C.c_uint64 * 2)(1, 2)
    n = C.c_uint64()
    d = abi.CatchLogDesc(n_seis=0, bin_lo=0, bin_hi=1, capacity=16)
    assert L.r3d_set_catch_log(None, C.byref(d)) == abi.R3D_EINVAL
    assert L.r3d_set_catch_log(None, None) == abi.R3D_EINVAL
    assert L.r3d_fetch_catch_log(None, None, 0, C.byref(n), C.byref(n)) == abi.R3D_EINVAL
    fin = (abi.PhononFinal * 2)()
    assert L.r3d_trace_indices(None, idx, 2, 1, fin) == abi.R3D_EINVAL
    ev = (C.c_uint8 * (2 * abi.EVENT_DTYPE.itemsize))()
    assert L.r3d_trace_events_indices(None, idx, 2, 1, abi.R3D_EV_ALL, ev, 2, C.byref(n)) == abi.R3D_EINVAL


def test_catch_log_desc_helper():
    d, keep = abi.catch_log_desc([3, 1], 2, 5, 100)
    assert (d.n_seis, d.bin_lo, d.bin_hi, d.capacity) == (2, 2, 5, 100) and list(keep) == [3, 1]
    assert d.seis[0] == 3 and d.seis[1] == 1
    d, _ = abi.catch_log_desc(None, 0, 7, 1)
    assert d.n_seis == 0 and not d.seis
