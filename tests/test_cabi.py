"""The C-ABI library builds for sm_100a here (nvcc cross-compiles without a GPU), loads, and exports
every symbol include/cutie_b200.h declares.  No compute calls (no GPU in this suite)."""
import ctypes
import os
import re
import subprocess

from tests.conftest import ROOT


def _declared():
    src = open(os.path.join(ROOT, 'include', 'cutie_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(cutie_[a-z0-9_]+)\s*\(', src)))


def test_abi_v2_library_builds_loads_and_exports_header_symbols():
    import __graft_entry__ as ge
    ge.build()
    lib = ctypes.CDLL(ge.LIB)
    names = _declared()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f'{n} declared in include/cutie_b200.h but not exported'
    assert lib.cutie_b200_abi_version() == 2
    lib.cutie_b200_last_error.restype = ctypes.c_char_p
    assert lib.cutie_b200_last_error() is not None


def test_argument_validation_needs_no_gpu():
    """Invalid arguments are rejected before any CUDA call and set the thread-local error string."""
    import __graft_entry__ as ge
    ge.build()
    lib = ctypes.CDLL(ge.LIB)
    lib.cutie_b200_last_error.restype = ctypes.c_char_p
    st = lib.cutie_obj_summary_accumulate(None, None, ctypes.c_int64(4), None)
    assert st == -1 and b'cutie_obj_summary_accumulate' in lib.cutie_b200_last_error()
    st = lib.cutie_qt_self_attention(None, None, ctypes.c_int64(16), ctypes.c_int64(256), 16, 8, None, None)
    assert st == -1


def test_query_chain_op_list_is_validated_on_the_host():
    """cutie_qt_chain checks its op list (counts, phase order, per-kind required pointers and sizes, the two coupled
    optional arguments of each op) before any CUDA call; cutie_consolidate_partial wants both statistics or neither."""
    import __graft_entry__ as ge
    from cutie_b200.kernels import _QtOp
    ge.build()
    lib = ctypes.CDLL(ge.LIB)
    lib.cutie_b200_last_error.restype = ctypes.c_char_p
    sync = (ctypes.c_uint32 * 4)()
    one = ctypes.c_void_p(0x1000)                      # never dereferenced: validation fails first

    def call(ops, n=None, sync_ws=sync):
        arr = (_QtOp * max(len(ops), 1))(*ops)
        return lib.cutie_qt_chain(arr, ctypes.c_int(len(ops) if n is None else n), None, None, ctypes.c_int(0), sync_ws, None)

    def linear(phase=0, **kw):
        o = _QtOp()
        o.kind, o.phase = 0, phase
        o.inp[0], o.inp[1], o.out[0] = one, one, one
        o.i[:] = (48, 256, 256, 256, 0, 0)
        for k, v in kw.items():
            setattr(o, k, v)
        return o
    assert call([], n=0) == -1 and b'cutie_qt_chain' in lib.cutie_b200_last_error()
    assert call([linear()] * 17) == -1
    assert call([linear()], sync_ws=None) == -1
    assert call([linear(phase=1), linear(phase=0)]) == -1 and b'phases' in lib.cutie_b200_last_error()
    bad = linear(); bad.kind = 9
    assert call([bad]) == -1 and b'unknown op' in lib.cutie_b200_last_error()
    no_w = linear(); no_w.inp[1] = None
    assert call([no_w]) == -1
    half_ln = linear(); half_ln.inp[3] = one           # ln_w without ln_b
    assert call([half_ln]) == -1 and b'ln_w' in lib.cutie_b200_last_error()
    xhat_without_ln = linear(); xhat_without_ln.out[1] = one
    assert call([xhat_without_ln]) == -1
    attn = linear(); attn.kind = 2; attn.i[0] = 40     # self attention: M must be a multiple of 16
    assert call([attn]) == -1
    comb = linear(); comb.kind = 3; comb.inp[2] = one; comb.i[:] = (2000, 256, 3, 0, 0, 0)    # > 1024 pixel tiles
    assert call([comb]) == -1 and b'pixel tiles' in lib.cutie_b200_last_error()
    fold = linear(); fold.kind = 1; fold.out[1] = one  # dots without bias_vec
    assert call([fold]) == -1
    # consolidate_partial: out_max without out_sumexp
    f = lib.cutie_consolidate_partial
    st = f(1, None, None, None, None, None, None, None, ctypes.c_int64(0), None, ctypes.c_int64(0), None, ctypes.c_int64(0),
           ctypes.c_int64(1), ctypes.c_int64(1), ctypes.c_int64(64), ctypes.c_int64(256), None, None, None, ctypes.c_int64(0),
           one, None, None, ctypes.c_int64(1), None)
    assert st == -1 and b'out_max' in lib.cutie_b200_last_error()


def test_sass_is_sm100a():
    import __graft_entry__ as ge
    ge.build()
    out = subprocess.run(['/usr/local/cuda/bin/cuobjdump', '-lelf', ge.LIB], capture_output=True, text=True).stdout
    assert 'sm_100a' in out


def test_affinity_plan_rule_is_pure_host_logic():
    """Which plan cutie_affinity_topk_img runs for a bank size (no GPU needed): exact scan below the threshold or when
    the bank has fewer than 2k tokens, the FP16 image filter at and above it."""
    import __graft_entry__ as ge
    ge.build()
    lib = ctypes.CDLL(ge.LIB)
    plan = lambda n, k=30: lib.cutie_affinity_plan(ctypes.c_int64(n), k)
    lib.cutie_set_tc_min_tokens(ctypes.c_int64(-1))
    assert plan(100) == 0 and plan(1620) == 0 and plan(4860) == 0 and plan(6143) == 0
    assert plan(6144) == 1 and plan(8100) == 1 and plan(65537) == 1 and plan(413100) == 1 and plan(20_000_000) == 1
    lib.cutie_set_tc_min_tokens(ctypes.c_int64(256))
    assert plan(333) == 1 and plan(256) == 1 and plan(255) == 0 and plan(4099) == 1
    assert plan(59) == 0 and plan(300, 151) == 0 and plan(300, 150) == 1      # fewer than 2k tokens: exact scan
    lib.cutie_set_tc_min_tokens(ctypes.c_int64(1 << 40))
    assert plan(413100) == 0
    lib.cutie_set_tc_min_tokens(ctypes.c_int64(-1))
    assert plan(413100) == 1
