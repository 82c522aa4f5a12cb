"""CPU-only checks: the C-ABI library builds for sm_100a, loads, and exports every symbol
include/bbgpu.h declares (no compute calls); piece tables; host Philox replica."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def libpath():
    import bbgpu.build as b
    return b.build()


def test_library_exports_every_declared_symbol(libpath):
    hdr = open(os.path.join(ROOT, "include", "bbgpu.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = sorted(set(re.findall(r"\b(bb_[a-z_0-9]+)\s*\(", hdr)))
    assert len(names) >= 30, names
    lib = C.CDLL(libpath)
    for n in names:
        assert hasattr(lib, n), "missing symbol " + n
    lib.bb_version.restype = C.c_int
    assert lib.bb_version() == 2


def test_piece_table_matches_oracle_table(libpath):
    from bbgpu import capi
    masks, inb, nblk = capi.piece_table()
    table = json.load(open(os.path.join(ROOT, "oracle", "piece_table.json")))
    assert len(table) == 37
    for i, row in enumerate(table):
        assert int(masks[i]) == int(row["mask"], 16)
        assert int(inb[i]) == int(row["inb"], 16)
        assert int(nblk[i]) == row["n"] == len(row["cells"])
    # reference tests/test_pieces.py KATs: counts per category, SINGLE first, 3x3 last
    assert table[0]["name"] == "SINGLE" and table[36]["name"] == "SQUARE_3x3"
    assert sum(bin(int(r["inb"], 16)).count("1") for r in table) == 1623
    assert [r["n"] for r in table].count(4) == 19 and [r["n"] for r in table].count(3) == 8


def test_committed_tables_equal_fresh_derivation_from_reference(tmp_path):
    """The three generated tables against a fresh derivation from the reference's PIECE_LIST as stored in
    tests/golden/reference_pieces.json (written by tools/gen_piece_tables.py --golden)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("gen", os.path.join(ROOT, "tools", "gen_piece_tables.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    rows = gen.derive(json.load(open(os.path.join(ROOT, "tests", "golden", "reference_pieces.json"))))
    table = json.load(open(os.path.join(ROOT, "oracle", "piece_table.json")))
    assert len(rows) == len(table) == 37
    for r, t in zip(rows, table):
        assert r["name"] == t["name"] and r["mask"] == int(t["mask"], 16) and r["inb"] == int(t["inb"], 16)
        assert [list(c) for c in r["cells"]] == t["cells"]
    for write, committed in ((gen.write_json, os.path.join("oracle", "piece_table.json")),
                             (gen.write_oracle_header, os.path.join("oracle", "bb_piece_cells.h")),
                             (gen.write_cuda_inc, os.path.join(gen.PKG, "csrc", "bb_piece_table.inc"))):
        write(rows, str(tmp_path / "out"))
        assert (tmp_path / "out").read_text() == open(os.path.join(ROOT, committed)).read(), committed


def test_philox_known_answers():
    from bbgpu import philox
    h = lambda t: [int(x) for x in t]
    assert h(philox.philox4x32_10(0, 0, 0, 0, 0, 0)) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    f = 0xffffffff
    assert h(philox.philox4x32_10(f, f, f, f, f, f)) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert h(philox.philox4x32_10(0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344, 0xa4093822, 0x299f31d0)) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    t = philox.candidate_trios(42, [0, 1], 3)
    assert t.shape == (2, 3, 3) and t.max() < 37
    assert t[0, 0].tolist() == [22, 17, 2]


def test_product_has_no_oracle_import():
    """The product path must not route through the oracle."""
    pkg = os.path.join(ROOT, "block-blast-ai---reinforcement-learning-agent_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "bboracle" not in src, f


def test_c_abi_error_paths_return_codes_not_crashes(libpath):
    """Argument errors are reported through return codes + bb_last_error() before any CUDA call
    (so this runs without a GPU); invalid ACTIONS are not errors (block_blast_env.py:240-245)."""
    lib = C.CDLL(libpath)
    lib.bb_last_error.restype = C.c_char_p
    vp, i64, u64, u32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_uint32
    lib.bb_env_create.argtypes = [C.POINTER(vp), i64, u64, i64, vp, u32]
    h = vp()
    assert lib.bb_env_create(None, 8, 0, 0, None, 0) < 0 and b"out is NULL" in lib.bb_last_error()
    assert lib.bb_env_create(C.byref(h), 0, 0, 0, None, 0) < 0 and b"n_envs" in lib.bb_last_error()
    assert lib.bb_env_create(C.byref(h), -5, 0, 0, None, 0) < 0
    assert lib.bb_env_create(C.byref(h), 8, 0, -1, None, 0) < 0 and b"offset" in lib.bb_last_error()
    assert h.value is None
    lib.bb_env_step.argtypes = [vp] * 12
    assert lib.bb_env_step(*([None] * 12)) < 0 and b"env is NULL" in lib.bb_last_error()
    lib.bb_env_reset.argtypes = [vp] * 4
    assert lib.bb_env_reset(None, None, None, None) < 0
    lib.bb_env_step_random.argtypes = [vp, C.c_int32, vp, vp, vp, vp, vp, vp, vp]
    assert lib.bb_env_step_random(None, 1, None, None, None, None, None, None, None) < 0
    lib.bb_env_set_trios.argtypes = [vp, vp, i64, vp]
    assert lib.bb_env_set_trios(None, None, 0, None) < 0 and b"env is NULL" in lib.bb_last_error()
    lib.bb_env_step_host_dense.argtypes = [vp] * 4
    assert lib.bb_env_step_host_dense(None, None, None, None) < 0
    lib.bb_env_fetch_step_info.argtypes = [vp] * 5
    assert lib.bb_env_fetch_step_info(None, None, None, None, None) < 0
    off5, off8, tot, pre = (i64 * 5)(), (i64 * 8)(), i64(), i64()
    lib.bb_env_host_dense_layout.argtypes = [i64, C.POINTER(i64), C.POINTER(i64)]
    assert lib.bb_env_host_dense_layout(10, off5, C.byref(tot)) == 0 and tot.value == 12210 and list(off5) == [0, 2560, 10240, 12160, 12200]
    assert lib.bb_env_host_dense_layout(0, off5, C.byref(tot)) < 0
    lib.bb_env_host_layout.argtypes = [i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]
    assert lib.bb_env_host_layout(10, off8, C.byref(tot), C.byref(pre)) == 0
    assert pre.value == 416 and tot.value == 416 + 120 and list(off8) == [0, 240, 320, 360, 416, 456, 496, 400]
    lib.bb_gather_minibatch.argtypes = [vp, i64, i64] + [vp] * 9 + [C.c_int] + [vp] * 6
    assert lib.bb_gather_minibatch(None, 4, 8, *([None] * 9), 0, *([None] * 6)) < 0 and b"NULL" in lib.bb_last_error()
    assert lib.bb_gather_minibatch(None, 4, 0, *([None] * 9), 0, *([None] * 6)) < 0
    lib.bb_env_destroy.argtypes = [vp]
    assert lib.bb_env_destroy(None) == 0                      # destroying nothing is fine
    lib.bb_env_num_envs.argtypes = [vp]
    lib.bb_env_num_envs.restype = i64
    assert lib.bb_env_num_envs(None) == -1
    lib.bb_gae.argtypes = [vp, vp, vp, vp, C.c_double, C.c_double, vp, vp, vp, i64, i64, vp]
    assert lib.bb_gae(None, None, None, None, 0.99, 0.95, None, None, None, 4, 4, None) < 0 and b"NULL" in lib.bb_last_error()
    assert lib.bb_gae(None, None, None, None, 0.99, 0.95, None, None, None, -1, 4, None) < 0
    lib.bb_masked_sample.argtypes = [vp, C.c_int, vp, i64, u64, u64, C.c_int, vp, vp, vp, i64, i64, vp, vp]
    assert lib.bb_masked_sample(None, 0, None, 0, 0, 0, 0, None, None, None, 4, 0, None, None) < 0
    one = (C.c_char * 64)()
    assert lib.bb_masked_sample(one, 7, one, 1, 0, 0, 0, one, None, None, 0, 0, None, None) < 0 and b"dtype" in lib.bb_last_error()
    assert lib.bb_masked_sample(one, 0, one, 1, 0, 0, 9, one, None, None, 0, 0, None, None) < 0 and b"mode" in lib.bb_last_error()
    lib.bb_unpack_obs.argtypes = [vp, vp, vp, i64, vp, C.c_int, vp, C.c_int, i64, vp]
    assert lib.bb_unpack_obs(None, None, None, 0, one, 0, None, 0, 1, None) < 0          # obs without board/pieces
    assert lib.bb_unpack_obs(one, one, one, 1, one, 5, None, 0, 1, None) < 0 and b"obs_dtype" in lib.bb_last_error()
    assert lib.bb_unpack_obs(one, one, None, 1, None, 0, one, 2, 1, None) < 0           # dense mask without mask
    assert lib.bb_unpack_obs(one, one, one, 1, None, 0, None, 0, -3, None) < 0
