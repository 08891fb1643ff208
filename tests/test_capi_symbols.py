"""The C-ABI library loads without a GPU and exports every symbol include/rqae_b200.h declares."""
import ctypes
import os
import re

from rqae_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "rqae_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rqae_[a-z0-9_]+)\s*\(", src)))


def test_header_and_binding_list_agree():
    assert header_symbols() == sorted(_lib.SYMBOLS)


def header_prototypes():
    """name -> (return type, [parameter types]) of every function include/rqae_b200.h declares, as C text."""
    src = open(os.path.join(ROOT, "include", "rqae_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = {}
    for ret, name, params in re.findall(r"([\w ]+\*?)\s*\b(rqae_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", src):
        params = [] if params.strip() == "void" else [re.sub(r"\s*\w+$", "", p.strip()) for p in params.split(",")]
        protos[name] = (" ".join(ret.split()), [" ".join(p.split()) for p in params])
    return protos


def test_binding_types_match_the_header():
    c = ctypes
    known = {"int": c.c_int, "int64_t": c.c_int64, "size_t": c.c_size_t, "float": c.c_float, "const char*": c.c_char_p,
             "int*": c.POINTER(c.c_int), "double*": c.POINTER(c.c_double)}   # int* / double*: out-parameters

    def ctype(decl):   # any other pointer is a data pointer
        return known.get(decl, c.c_void_p if decl.endswith("*") else None)

    protos = header_prototypes()
    assert sorted(protos) == header_symbols()
    for name, (ret, params) in protos.items():
        restype, argtypes = _lib.BINDINGS[name]
        assert restype is ctype(ret), f"{name}: returns {ret}, bound as {restype}"
        assert len(argtypes) == len(params), f"{name}: {len(params)} parameters, {len(argtypes)} bound"
        for k, (decl, bound) in enumerate(zip(params, argtypes)):
            assert bound is ctype(decl), f"{name}: parameter {k} is {decl}, bound as {bound}"


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in header_symbols():
        assert hasattr(lib, name), f"{name} missing from librqae_b200.so"


def test_host_only_entry_points():
    lib = _lib.load()
    assert b"sm_100a" in lib.rqae_version()
    assert lib.rqae_strerror(0) == b"ok" and lib.rqae_strerror(2).startswith(b"unsupported")
    # packed size model: header + biases + search table + (nq+1) stages of E*256*36 bytes
    n = lib.rqae_packed_bytes(1024, 2304, 4, 625)
    assert n >= 1025 * 9 * 256 * 36 and n < 1025 * 9 * 256 * 36 + (1 << 16)
    assert lib.rqae_packed_bytes(2048, 3584, 4, 625) >= 2049 * 14 * 256 * 36
    assert lib.rqae_packed_bytes(8, 2304, 8, 625) == 0      # codebook_dim != 4
    assert lib.rqae_packed_bytes(8, 5000, 4, 625) == 0      # dim beyond the compiled shapes
    # argument validation happens before any CUDA call
    assert lib.rqae_forward_f32(None, None, 1, 8, 8, 256, 4, 625, None, 4, None, 2, 8, None, None, None, None) == 1
    assert lib.rqae_decode_f32(None, None, 8, 8, 256, 4, 625, None, 2, 8, None, None, 4, None, None) == 1


def test_mining_entry_points_validate_before_touching_the_gpu():
    import ctypes
    import numpy as np
    lib = _lib.load()
    cuts = np.array([2, 4, 1023], dtype=np.int32)
    n = lib.rqae_intensity_workspace_bytes(cuts.ctypes.data, 3, 1024, 1 << 20)
    # schedule + tables + 8 feature tiles x (1+1+64) K-blocks x 16 KB + layer-major int16 codes
    assert n >= 8 * 66 * 16384 + 1024 * (1 << 20) * 2 and n < 8 * 66 * 16384 + 1024 * (1 << 20) * 2 + (1 << 16)
    bad = np.array([4, 2], dtype=np.int32)                       # not ascending
    assert lib.rqae_intensity_workspace_bytes(bad.ctypes.data, 2, 8, 100) == 0
    assert lib.rqae_intensity_workspace_bytes(cuts.ctypes.data, 0, 8, 100) == 0
    one = ctypes.c_void_p(4096)
    assert lib.rqae_intensity_f16(None, 625, one, 0, 1024, 8, one, 1024, 1, one, cuts.ctypes.data, 3, one, 256, one, n, None) == 1
    assert lib.rqae_intensity_f16(one, 5000, one, 0, 1024, 8, one, 1024, 1, one, cuts.ctypes.data, 3, one, 256, one, n, None) == 2
    assert lib.rqae_intensity_f16(one, 625, one, 0, 16, 8, one, 1024, 1, one, cuts.ctypes.data, 3, one, 256, one, n, None) == 1   # stride < layers
    assert lib.rqae_intensity_f16(one, 625, one, 0, 1024, 8, one, 1024, 1, one, cuts.ctypes.data, 3, one, 100, one, n, None) == 1  # out rows too short
    assert lib.rqae_intensity_f16(one, 625, one, 0, 1024, 8, one, 1024, 1, one, cuts.ctypes.data, 3, one, 256, one, 16, None) == 5  # workspace too small
    assert lib.rqae_select_top_middle_bottom_f16(one, 4, 256, 200, 300, one, None, None) == 1      # k > n
    assert lib.rqae_select_top_middle_bottom_f16(one, 4, 512, 400, 300, one, None, None) == 2      # k > 256
    assert lib.rqae_select_top_middle_bottom_f16(one, 4, 250, 250, 10, one, None, None) == 1       # rows not 16-byte aligned
    assert lib.rqae_select_top_middle_bottom_f16(one, 0, 256, 250, 10, one, None, None) == 0       # nothing to do


def test_search_entry_points_validate_before_touching_the_gpu():
    import ctypes
    lib = _lib.load()
    assert lib.rqae_search_table_bytes(1023, 625) == 1023 * 625 * 128 * 2
    assert lib.rqae_search_table_bytes(0, 625) == 0
    one = ctypes.c_void_p(4096)
    tb = lib.rqae_search_table_bytes(16, 625)
    assert lib.rqae_search_build_table_f16(None, 625, one, 16, 7, 16, one, tb, None) == 1
    assert lib.rqae_search_build_table_f16(one, 625, one, 8, 7, 16, one, tb, None) == 1        # query rows shorter than n_layers
    assert lib.rqae_search_build_table_f16(one, 625, one, 16, 129, 16, one, tb, None) == 2     # more than 128 query positions
    assert lib.rqae_search_build_table_f16(one, 625, one, 16, 7, 16, one, tb - 1, None) == 5   # table too small
    assert lib.rqae_search_accumulate_f16(one, 625, one, 3, 16, 8, 0, 4, 1, one, None) == 1    # unknown code dtype
    assert lib.rqae_search_accumulate_f16(one, 625, one, 1, 16, 8, 4, 4, 0, one, None) == 1    # empty layer range
    assert lib.rqae_search_accumulate_f16(one, 625, one, 1, 16, 8, 4, 24, 0, one, None) == 1   # range beyond the code rows
    assert lib.rqae_search_accumulate_f16(one, 625, one, 1, 16, 0, 0, 4, 1, one, None) == 0    # no tokens: nothing to do
    assert lib.rqae_search_position_max_f16(one, 24, 7, 7, one, 20, None) == 1                 # rows shorter than n_seq
    assert lib.rqae_search_position_max_f16(one, 24, 7, 7, one, 28, None) == 1                 # row stride not a multiple of 8
    assert lib.rqae_search_position_max_f16(one, 24, 7, 200, one, 24, None) == 2               # more than 128 query positions


def test_tensor_core_search_entry_points_validate_before_touching_the_gpu():
    import ctypes
    import numpy as np
    lib = _lib.load()
    # the block-major store copy: ceil(n_seq / 2) units x ceil(layers / 8) blocks x 256 rows x 16 bytes
    assert lib.rqae_search_tc_store_bytes(36864, 1024) == 18432 * 128 * 256 * 16
    assert lib.rqae_search_tc_store_bytes(9, 150) == 5 * 19 * 256 * 16
    assert lib.rqae_search_tc_store_bytes(0, 1024) == 0
    cuts = np.array([4, 6, 8, 12, 16, 24, 32, 48, 64, 128, 256, 512, 1023], dtype=np.int32)    # server.py:167
    # 131 K-blocks of 8 layers: a range end inside a block costs a K-block of its own
    assert lib.rqae_search_tc_workspace_bytes(cuts.ctypes.data, 13) == 4096 + 131 * 16384
    bad = np.array([8, 8], dtype=np.int32)
    assert lib.rqae_search_tc_workspace_bytes(bad.ctypes.data, 2) == 0                         # not strictly ascending
    one = ctypes.c_void_p(4096)
    wb = lib.rqae_search_tc_workspace_bytes(cuts.ctypes.data, 13)
    assert lib.rqae_search_tc_pack_store(one, 0, 1024, 10, 200, 1024, 625, one, 1 << 40, None) == 2    # more than 128 positions
    assert lib.rqae_search_tc_pack_store(one, 0, 512, 10, 127, 1024, 625, one, 1 << 40, None) == 1     # code rows shorter than the layers
    assert lib.rqae_search_tc_pack_store(one, 0, 1024, 10, 127, 1024, 625, one, 16, None) == 5         # store copy too small
    args = (one, 10, 127, 1024, one, one, 1024, 625, one, 1024, 127, cuts.ctypes.data, 13, one)
    assert lib.rqae_search_tc_maxima_f16(*args[:10], 200, *args[11:], 16, one, wb, None) == 2          # more than 128 query positions
    assert lib.rqae_search_tc_maxima_f16(*args, 8, one, wb, None) == 1                                 # rows shorter than the 10 sequences
    assert lib.rqae_search_tc_maxima_f16(*args, 16, one, 64, None) == 5                                # workspace too small
    assert lib.rqae_search_tc_maxima_f16(*args[:6], 512, *args[7:], 16, one, wb, None) == 1            # factor tables shorter than the layers
    assert lib.rqae_search_rows_f16(one, 625, one, 0, 1024, 10, 127, one, 127, 50, cuts.ctypes.data, 60, 10, one, None) == 2  # more than 64 ranges
    assert lib.rqae_search_rows_f16(one, 625, one, 0, 512, 10, 127, one, 127, 50, cuts.ctypes.data, 0, 13, one, None) == 1    # code rows shorter than the last range
    assert lib.rqae_search_rows_f16(one, 625, one, 0, 1024, 10, 127, one, 127, 0, cuts.ctypes.data, 0, 13, one, None) == 0    # nothing selected


def test_host_widening_pool_matches_numpy():
    """The widening step of the narrow host pipeline (int16 -> int32 / int64, AVX2 streaming stores, persistent worker
    pool) on its own: every thread count, unaligned destinations, sizes around the split and vector widths."""
    import numpy as np
    lib = _lib.load()
    rng = np.random.default_rng(0)
    for n in (0, 1, 15, 16, 17, 65535, 65536, 65537, 300001, 1 << 20):
        src = rng.integers(0, 625, size=n + 8, dtype=np.int16)
        for dtype, code in ((np.int32, 1), (np.int64, 2)):
            for threads in (1, 2, 3, 8):
                for off in (0, 1):
                    dst = np.full(n + 8, -7, dtype=dtype)
                    rc = lib.rqae_widen_codes_host(src[off:].ctypes.data, dst[off:].ctypes.data, n, code, threads)
                    assert rc == 0
                    assert np.array_equal(dst[off:off + n], src[off:off + n].astype(dtype))
                    assert (dst[:off] == -7).all() and (dst[off + n:] == -7).all()
    # changing the thread count between calls re-creates the pool: new workers must wait for a NEW job
    big = rng.integers(0, 625, size=1 << 18, dtype=np.int16)
    for threads in (8, 2, 5, 1, 8, 3):
        dst = np.empty(1 << 18, np.int64)
        assert lib.rqae_widen_codes_host(big.ctypes.data, dst.ctypes.data, 1 << 18, 2, threads) == 0
        assert np.array_equal(dst, big.astype(np.int64))
        del dst
    assert lib.rqae_widen_codes_host(None, None, 4, 2, 1) == 1
    assert lib.rqae_widen_codes_host(None, None, 0, 0, 1) == 1      # int16 is not a widening target
    assert lib.rqae_forward_host_config(3, 0) == 1 and lib.rqae_forward_host_config(-1, -1) == 0
    # int16 codes cannot hold a 40000-row codebook: refused before any CUDA call
    one = ctypes.c_void_p(4096)
    assert lib.rqae_forward_f32(one, one, 0, 8, 8, 256, 4, 40000, one, 4, one, 0, 8, None, None, None, None) == 1
