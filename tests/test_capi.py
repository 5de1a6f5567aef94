"""CPU suite, part 3: the C-ABI boundary.  The built library must load and export every symbol that
include/sdb200.h declares, and the ctypes binding table must cover exactly that set (no compute calls)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "sdb200.h")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"typedef struct.*?}\s*\w+;", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sdk_\w+)\s*\(", src)))


def test_header_declares_entry_points():
    names = declared_functions()
    for must in ("sdk_ddim_step", "sdk_ddpm_step", "sdk_tc_gemm_launch", "sdk_attention_bf16", "sdk_groupnorm_stats",
                 "sdk_layernorm", "sdk_conv_gemm_f32", "sdk_last_error"):
        assert must in names
    assert len(names) >= 25


def test_library_exports_every_declared_symbol():
    from stable_diffusion_pytorch_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    h = ctypes.CDLL(_lib.LIB_PATH)
    missing = [n for n in declared_functions() if not hasattr(h, n)]
    assert not missing, f"declared in sdb200.h but not exported: {missing}"


def test_binding_table_matches_header():
    from stable_diffusion_pytorch_b200 import _lib
    assert sorted(_lib.SIGNATURES) == declared_functions()
    lib = _lib.lib()                       # resolves every symbol with its argtypes
    assert lib.sdk_version() >= 100
    assert lib.sdk_last_error() is not None


def test_struct_layouts_match_header():
    """ctypes mirrors of the two parameter structs have the field order of the header."""
    from stable_diffusion_pytorch_b200 import _lib
    src = open(HEADER).read()
    for cname, mirror in (("SdkConvParams", _lib.ConvParams), ("SdkTcGemmDesc", _lib.TcGemmDesc), ("SdkLinearLnDesc", _lib.LinearLnDesc), ("SdkAttentionTcDesc", _lib.AttentionTcDesc)):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (cname, cname), src, flags=re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        fields = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            names = decl.split(None, 1)[1] if not decl.startswith("const") else decl.split(None, 2)[2]
            for n in names.split(","):
                fields.append(n.replace("*", "").strip().split("[")[0])
        assert fields == [f[0] for f in mirror._fields_], (cname, fields)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from stable_diffusion_pytorch_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.ExtensionMissing, match="no CPU/PyTorch fallback"):
        _lib.lib()


def test_tune_cache_roundtrip(tmp_path, monkeypatch):
    """Measured GEMM tilings persist as JSON keyed by GPU model + layer shape; 2-element entries of older files still load.
    New measurements are MERGED into the per-user file (never the package's committed cache), keeping other writers' entries."""
    import hashlib
    import json
    from stable_diffusion_pytorch_b200.program import LaunchProgram
    f = tmp_path / "user" / "tune.json"
    f.parent.mkdir()
    f.write_text(json.dumps({"NVIDIA B200|2|64|64|320|1|320|3|0|0|0|0|1|1": [160, 1], "NVIDIA B200|1|1|8192|960|1|320|1|0|0|1|0|0|0": [128, 3, 0]}))
    shipped = hashlib.sha1(open(LaunchProgram._tune_shipped, "rb").read()).hexdigest()
    monkeypatch.setenv("SDB200_TC_TUNE_FILE", str(f))
    monkeypatch.setattr(LaunchProgram, "_tune_loaded", False)
    monkeypatch.setattr(LaunchProgram, "_tune_cache", {})
    LaunchProgram._tune_load()
    assert LaunchProgram._tune_cache["NVIDIA B200|2|64|64|320|1|320|3|0|0|0|0|1|1"] == (160, 1)      # the user file wins over the shipped one
    # another process added an entry meanwhile: the merge keeps it
    cur = json.loads(f.read_text())
    cur["other-rank"] = [32, 4, 0]
    f.write_text(json.dumps(cur))
    LaunchProgram._tune_save("k", (64, 2, 0))
    after = json.loads(f.read_text())
    assert after["k"] == [64, 2, 0] and after["other-rank"] == [32, 4, 0]
    assert hashlib.sha1(open(LaunchProgram._tune_shipped, "rb").read()).hexdigest() == shipped       # package file untouched


def test_context_version_helpers():
    """inference_mode tensors have no version counter (reference inpaint runs under it, models/diffusion.py:328): the context
    cache must treat them as changed instead of raising."""
    import torch
    from stable_diffusion_pytorch_b200.unet import same_context, tensor_version
    a = torch.zeros(3)
    v = tensor_version(a)
    assert same_context(a, a, v)
    a.add_(1)
    assert not same_context(a, a, v)
    with torch.inference_mode():
        b = torch.zeros(3)
    assert tensor_version(b) is None
    assert not same_context(b, b, None)
