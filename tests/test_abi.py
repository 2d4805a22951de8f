"""CPU-side checks of the drop-in boundary: the C-ABI library builds, loads, and exports every symbol that
include/mcgra.h declares (no compute calls -- there is no GPU here)."""
import ctypes
import os
import re
import shutil

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def native():
    import __graft_entry__ as g
    g.build()
    from mcgra_b200 import _native
    return _native


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "mcgra.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(?:int|int64_t)\s+(mcgra_\w+)\s*\(", src)))


def test_header_symbols_are_exported(native):
    lib = ctypes.CDLL(native.LIB_PATH)
    names = declared_symbols()
    assert len(names) >= 20
    for name in names:
        assert hasattr(lib, name), f"{name} declared in include/mcgra.h but not exported"
    assert set(names) == set(native.exported_symbols()), "ctypes table and header disagree"


def test_version_and_tile_count(native):
    L = native.lib()
    assert L.mcgra_version() >= 1
    assert L.mcgra_tiles_in_rows(0, 4) == 10
    assert L.mcgra_tiles_in_rows(2, 4) == 7


# bench.py's large_parity restores {0: 5, 1: 3, 2: 2} after its exact-engine run, so these must stay the defaults
DEFAULT_ENGINES = {0: 5, 1: 3, 2: 2, 4: 1, 5: 1, 6: 1}


def test_fresh_library_reports_default_engines(native, tmp_path):
    # a copy under another path is loaded as a second instance, with engine state no earlier test has touched
    fresh = tmp_path / "libmcgra_fresh.so"
    shutil.copyfile(native.LIB_PATH, fresh)
    L = ctypes.CDLL(str(fresh))
    assert {which: L.mcgra_get_engine(which) for which in DEFAULT_ENGINES} == DEFAULT_ENGINES
    assert [L.mcgra_get_engine(which) for which in (-1, 3, 7)] == [-1, -1, -1]


def test_set_engine_accepts_only_known_values(native):
    L = native.lib()
    accepted = {0: [0, 5], 1: [0, 2, 3, 100, 101, 999], 2: [0, 1, 2], 4: [0, 1, 100, 101, 999], 5: [0, 1], 6: [0, 1]}
    rejected = [(3, 1), (3, 2), (3, 116), (0, 3), (0, 1), (0, 101), (1, 1), (1, 4), (1, 1007), (1, 1000), (1, -1),
                (2, 3), (2, -1), (4, 2), (4, 1000), (5, 2), (6, 2), (6, 101), (7, 0), (-1, 0)]
    saved = {which: L.mcgra_get_engine(which) for which in accepted}
    try:
        for which, values in accepted.items():
            for value in values:
                assert L.mcgra_set_engine(which, value) == 0, (which, value)
                if value < 100:                     # 100 + cap sets the grid cap and leaves the engine as it is
                    engine = value
                assert L.mcgra_get_engine(which) == engine, (which, value)
        for which, value in rejected:
            before = L.mcgra_get_engine(which)
            assert L.mcgra_set_engine(which, value) == -1, (which, value)
            assert L.mcgra_get_engine(which) == before, (which, value)
    finally:
        for which, value in saved.items():
            assert L.mcgra_set_engine(which, value) == 0
        assert L.mcgra_set_engine(1, 100) == 0 and L.mcgra_set_engine(4, 100) == 0     # grid caps off


def test_struct_sizes_match_c(native):
    # the C structs are passed by pointer; their size must match what nvcc laid out (probe via a tiny C check)
    import subprocess, tempfile, textwrap
    code = textwrap.dedent("""
        #include <stdio.h>
        #include "mcgra.h"
        int main(){ printf("%zu %zu %zu %zu\\n", sizeof(mcgra_elem_args), sizeof(mcgra_node_args), sizeof(mcgra_fold_args), sizeof(mcgra_ensemble_args)); return 0; }
    """)
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "s.c")
        open(src, "w").write(code)
        exe = os.path.join(td, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        sizes = [int(v) for v in subprocess.check_output([exe]).split()]
    assert sizes == [ctypes.sizeof(native.ElemArgs), ctypes.sizeof(native.NodeArgs), ctypes.sizeof(native.FoldArgs),
                     ctypes.sizeof(native.EnsembleArgs)]


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from mcgra_b200 import _native
    from mcgra_b200.engine import PGDEngine
    with pytest.raises(_native.NativeError):
        PGDEngine(4, torch.zeros(4, 16), torch.zeros(16, 16), torch.zeros(16), torch.zeros(16), torch.zeros(2, 16),
                  torch.zeros(2), torch.zeros(4, dtype=torch.long), [0, 1, 2, 3], torch.zeros(4, 16), torch.zeros(4, 2),
                  None, "MSELoss", [0] * 10, 0.01)


def test_shard_tile_rows_cover_and_balance():
    from mcgra_b200.engine import shard_tile_rows, tri
    for T in (1, 3, 21, 155, 512):
        for world in (1, 2, 4, 8):
            sh = shard_tile_rows(T, world)
            assert sh[0][0] == 0 and sh[-1][1] == T
            assert all(a[1] == b[0] for a, b in zip(sh, sh[1:]))
            if T >= 64:
                counts = [tri(b) - tri(a) for a, b in sh]
                assert max(counts) / (sum(counts) / world) < 1.1
