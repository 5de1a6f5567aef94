"""CPU suite: argument checking of the plan-level C entry (sdk_plan_*, include/sdb200.h) -- no device work."""
import ctypes as C

import pytest

from stable_diffusion_pytorch_b200 import _lib


@pytest.fixture()
def plan():
    lib = _lib.lib()
    h = C.c_void_p()
    assert lib.sdk_plan_create(C.byref(h)) == 0
    yield lib, h
    assert lib.sdk_plan_destroy(h) == 0


def _args(*v):
    return (C.c_uint64 * max(len(v), 1))(*v)


def test_add_launch_checks_name_and_arity(plan):
    lib, h = plan
    assert lib.sdk_plan_num_launches(h, 0) == 0
    # sdk_layernorm(x, gamma, beta, eps, out, out_dtype, rows, C, stream): 8 arguments before the stream
    assert lib.sdk_plan_add_launch(h, 0, b"sdk_layernorm", _args(1, 2, 3, 0x3727C5AC, 4, 1, 128, 320), 8) == 0
    assert lib.sdk_plan_num_launches(h, 0) == 1
    assert lib.sdk_plan_add_launch(h, 0, b"sdk_layernorm", _args(1, 2, 3), 3) == -1
    assert b"8 arguments" in lib.sdk_last_error()
    assert lib.sdk_plan_add_launch(h, 0, b"sdk_tc_gemm_create", _args(1, 2), 2) == -3          # not a launch-type entry point
    assert lib.sdk_plan_add_launch(h, 99, b"sdk_layernorm", _args(1, 2, 3, 0, 4, 1, 128, 320), 8) == -1
    # a handle launch needs an adopted handle
    assert lib.sdk_plan_add_launch(h, 0, b"sdk_tc_gemm_launch", _args(0xdead0), 1) == -1
    assert b"adopt" in lib.sdk_last_error()
    assert lib.sdk_plan_num_launches(h, 0) == 1 and lib.sdk_plan_num_launches(h, 1) == 0 and lib.sdk_plan_num_launches(h, 99) == -1


def test_every_recorded_entry_point_is_in_the_binding_table():
    """The Python transcription looks the argument types up in _lib.SIGNATURES: every launch-type entry point must be there."""
    lib = _lib.lib()
    h = C.c_void_p()
    assert lib.sdk_plan_create(C.byref(h)) == 0
    launchers = [n for n, sig in _lib.SIGNATURES.items()
                 if sig and sig[-1] is _lib.P and not n.startswith(("sdk_plan_", "sdk_stream_")) and "create" not in n
                 and "destroy" not in n and n not in ("sdk_tc_gemm_set_workspace", "sdk_tc_gemm_info", "sdk_tc_gemm_set_debug", "sdk_tc_gemm_set_stats",
                                                      "sdk_tc_gemm_workspace_bytes", "sdk_linear_ln_info", "sdk_device_info")]
    known = 0
    for n in launchers:
        nargs = len(_lib.SIGNATURES[n]) - 1
        rc = lib.sdk_plan_add_launch(h, 1, n.encode(), _args(*([0] * nargs)), nargs)
        if n in ("sdk_tc_gemm_launch", "sdk_attention_tc_launch", "sdk_linear_ln_launch", "sdk_conv_gemm_f32"):
            assert rc == -1, n                                     # known, but needs a handle / struct
        else:
            assert rc == 0, (n, lib.sdk_last_error())
            known += 1
    assert known >= 25
    lib.sdk_plan_destroy(h)


def test_regions_and_adopt_checks(plan):
    lib, h = plan
    assert lib.sdk_plan_add_region(h, 0x10000, 4096, 0, b"") == 0
    assert lib.sdk_plan_add_region(h, 0x10000, 4096, 0, b"again") == 0               # same buffer twice: harmless
    assert lib.sdk_plan_add_region(h, 0x10800, 4096, 1, b"") == -1                   # partial overlap
    assert lib.sdk_plan_add_region(h, 0x20000, 0, 1, b"") == -1
    p, n = C.c_void_p(), C.c_int64()
    assert lib.sdk_plan_region(h, b"again", C.byref(p), C.byref(n)) == 0 and p.value == 0x10000 and n.value == 4096
    assert lib.sdk_plan_region(h, b"nope", C.byref(p), C.byref(n)) == -1
    d = _lib.LinearLnDesc()
    assert lib.sdk_plan_adopt(h, 3, 0, C.byref(d), C.sizeof(d), _args(0, 0), 2) == -1         # null handle
    assert lib.sdk_plan_adopt(h, 7, 0x1234, C.byref(d), C.sizeof(d), _args(0, 0), 2) == -1    # unknown kind
    assert lib.sdk_plan_adopt(h, 1, 0x1234, C.byref(d), C.sizeof(d), _args(0, 0), 2) == -1    # descriptor size of another kind


def test_load_rejects_missing_and_foreign_files(tmp_path):
    lib = _lib.lib()
    h = C.c_void_p()
    assert lib.sdk_plan_load(str(tmp_path / "missing.engine").encode(), C.byref(h)) == -1
    f = tmp_path / "junk.engine"
    f.write_bytes(b"not an engine file at all" * 10)
    assert lib.sdk_plan_load(str(f).encode(), C.byref(h)) == -1
    assert b"engine file" in lib.sdk_last_error()


def test_slots_encode_floats_and_negative_ints():
    from stable_diffusion_pytorch_b200.program import LaunchProgram
    s = LaunchProgram._slots("sdk_gather_row", (0x1000, 20160, 50, 0x2000, -1, 0x3000))
    assert list(s) == [0x1000, 20160, 50, 0x2000, 0xFFFFFFFFFFFFFFFF, 0x3000]
    s = LaunchProgram._slots("sdk_layernorm", (1, 2, 3, 1e-5, 4, 1, 128, 320))
    assert s[3] == 0x3727C5AC
    with pytest.raises(RuntimeError):
        LaunchProgram._slots("sdk_layernorm", (1, 2, 3))


def test_save_load_roundtrip_and_truncation(tmp_path):
    """The engine file format without a GPU: a plan whose launches carry no device memory saves and loads on the CPU; every
    truncation of the file is rejected cleanly (no crash, no partial plan)."""
    lib = _lib.lib()
    h = C.c_void_p()
    assert lib.sdk_plan_create(C.byref(h)) == 0
    assert lib.sdk_plan_add_launch(h, 2, b"sdk_zero", _args(0, 0), 2) == 0
    assert lib.sdk_plan_add_launch(h, 2, b"sdk_x0_from_eps", _args(0, 0, 0x3F7F0000, 0x3D8C7E28, 0, 0), 6) == 0
    assert lib.sdk_plan_add_launch(h, 5, b"sdk_gather_row", _args(0, 20160, 50, 0, 0xFFFFFFFFFFFFFFFF, 0), 6) == 0
    path = tmp_path / "tiny.engine"
    assert lib.sdk_plan_save(h, str(path).encode()) == 0, lib.sdk_last_error()
    assert lib.sdk_plan_destroy(h) == 0
    data = path.read_bytes()
    assert data[:8] == b"SDB200PL" and len(data) < 4096
    h2 = C.c_void_p()
    assert lib.sdk_plan_load(str(path).encode(), C.byref(h2)) == 0, lib.sdk_last_error()
    assert [lib.sdk_plan_num_launches(h2, i) for i in (0, 2, 5)] == [0, 2, 1]
    assert lib.sdk_plan_destroy(h2) == 0
    for cut in list(range(0, len(data), 7)) + [len(data) - 1]:
        f = tmp_path / f"cut{cut}.engine"
        f.write_bytes(data[:cut])
        h3 = C.c_void_p()
        assert lib.sdk_plan_load(str(f).encode(), C.byref(h3)) == -1, cut
    # a corrupted launch name is rejected too
    bad = bytearray(data)
    i = bad.find(b"sdk_zero")
    bad[i:i + 8] = b"sdk_zerx"
    f = tmp_path / "bad.engine"
    f.write_bytes(bytes(bad))
    assert lib.sdk_plan_load(str(f).encode(), C.byref(C.c_void_p())) == -1
