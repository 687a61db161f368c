"""The C-ABI library loads on a CPU-only box and exports every symbol include/raft_b200.h declares."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "raft_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from raft_b200 import capi
    names = _declared()
    assert len(names) >= 25
    lib = ctypes.CDLL(capi.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in raft_b200.h but not exported"
    assert set(names) == set(capi.SIGNATURES), set(names) ^ set(capi.SIGNATURES)


def test_library_reads_only_the_documented_knobs():
    """The environment variables the library reads: the switches README.md lists, nothing left over from tuning."""
    from raft_b200 import capi
    names = set(re.findall(rb"RAFT_B200_[A-Z0-9_]+", open(capi.LIB_PATH, "rb").read()))
    assert names == {b"RAFT_B200_" + k for k in (b"NO_PDL", b"NO_HOIST", b"NO_STASH", b"NO_SPLITK", b"NO_SPLITK_CLUSTER",
                                                   b"NO_FUSED_STATS", b"LOOKUP_V5", b"SPLITK_CLOSING_BARRIER")}, names


def test_host_only_queries():
    from raft_b200 import capi
    lib = capi.lib
    assert lib.rb_version() >= 100
    assert lib.rb_update_num_convs(0) == 15 and lib.rb_update_num_convs(1) == 9
    assert lib.rb_update_conv_name(0, 5) == b"update_block/gru/convz1"
    assert lib.rb_update_conv_name(1, 8) == b"update_block/flow_head/conv2"
    # pyramid size at things@440x1024 = 261.3 MB (SURVEY section 6)
    assert capi.size_query(lib.rb_corr_pyramid_bytes, 1, 55, 128) == 4 * 7040 * (55 * 128 + 27 * 64 + 13 * 32 + 6 * 16) + 256
    # error path: status code + message, no abort
    out = ctypes.c_size_t()
    assert lib.rb_corr_pyramid_bytes(1, 4, 4, ctypes.byref(out)) == -1
    assert b"too small" in lib.rb_last_error()
    assert lib.rb_set_math_mode(7) == -2
    # argument checks come before any CUDA call: unsupported stride / even kernel -> RB_ERR_UNSUPPORTED on a CPU-only box
    buf = (ctypes.c_float * 16)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert lib.rb_conv2d_strided(p, p, None, p, 1, 8, 8, 4, 4, 3, 3, 3, 0, p, 64, None) == -3
    assert b"stride" in lib.rb_last_error()
    assert lib.rb_conv2d_strided(p, p, None, p, 1, 8, 8, 4, 4, 2, 2, 1, 0, p, 64, None) == -3
    assert lib.rb_update_packed_conv(0, 12, None, None, None, None, None, None, None, None) == -2

