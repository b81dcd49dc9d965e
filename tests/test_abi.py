"""CPU: the C-ABI library loads and exports every symbol include/llama2_b200.h declares;
argument validation and the no-fallback rule hold without a GPU (no compute calls here)."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest


def test_library_exports_every_declared_symbol(l2b):
    lib = l2b.load_library()
    names = l2b.exported_symbols()
    assert len(names) >= 20
    out = subprocess.run(["nm", "-D", "--defined-only", l2b.lib_path()], capture_output=True, text=True,
                         check=True).stdout
    defined = {line.split()[-1] for line in out.splitlines() if " T " in line}
    for n in names:
        assert n in defined, f"{n} declared in llama2_b200.h but not exported"
        assert hasattr(lib, n)
    assert lib.l2b_abi_version() == 2


def test_library_is_sm100a_only(l2b):
    out = subprocess.run(["cuobjdump", "-lelf", l2b.lib_path()], capture_output=True, text=True).stdout
    archs = {tok for line in out.splitlines() for tok in line.replace(".", " ").split() if tok.startswith("sm_")}
    assert archs == {"sm_100a"}, archs


def test_status_strings(l2b):
    lib = l2b.load_library()
    assert lib.l2b_status_string(0) == b"ok"
    for code in range(-7, 0):
        assert lib.l2b_status_string(code) not in (b"", b"unknown status")


def test_create_rejects_bad_arguments_before_touching_cuda(l2b):
    from llama2_zig_b200.binding import L2BConfig, FP
    lib = l2b.load_library()
    h = C.c_void_p()
    cfg = L2BConfig(288, 768, 6, 6, 6, 32000, 256, 1)
    data = np.zeros(8, np.float32)
    # NULL weights
    assert lib.l2b_create(C.byref(h), C.byref(cfg), None, 0, None, None, 1) == -1
    # n_gpus must be 1, 2, 4 or 8 (SURVEY.md 8b), and the shape must shard over it (6 kv heads % 4)
    assert lib.l2b_create(C.byref(h), C.byref(cfg), data.ctypes.data_as(FP), 8, None, None, 3) == -2
    assert lib.l2b_create(C.byref(h), C.byref(cfg), data.ctypes.data_as(FP), 8, None, None, 4) == -2
    assert b"n_kv_heads" in lib.l2b_last_error(None)
    # head_size > 256: the attention kernels write one output element per thread (ADVICE r1)
    wide = L2BConfig(1024, 2048, 2, 2, 2, 1000, 64, 1)
    assert lib.l2b_create(C.byref(h), C.byref(wide), data.ctypes.data_as(FP), 8, None, None, 1) == -2
    assert b"head_size" in lib.l2b_last_error(None)
    # unsupported shapes (head_size not a multiple of 4; dim not divisible by heads)
    bad = L2BConfig(36, 768, 6, 6, 6, 32000, 256, 1)
    assert lib.l2b_create(C.byref(h), C.byref(bad), data.ctypes.data_as(FP), 8, None, None, 1) == -2
    bad2 = L2BConfig(290, 768, 6, 6, 6, 32000, 256, 1)
    assert lib.l2b_create(C.byref(h), C.byref(bad2), data.ctypes.data_as(FP), 8, None, None, 1) == -2
    neg = L2BConfig(288, 768, 0, 6, 6, 32000, 256, 1)
    assert lib.l2b_create(C.byref(h), C.byref(neg), data.ctypes.data_as(FP), 8, None, None, 1) == -1
    # payload shorter than the checkpoint layout requires
    assert lib.l2b_create(C.byref(h), C.byref(cfg), data.ctypes.data_as(FP), 8, None, None, 1) == -1
    assert b"shorter" in lib.l2b_last_error(None)
    assert not h.value


def test_no_cpu_fallback_when_no_device(l2b):
    """Without a GPU the product must fail loudly (L2B_ERR_NO_DEVICE), never compute on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from llama2_zig_b200.checkpoint import shape_checkpoint
    ck = shape_checkpoint((64, 172, 2, 4, 2, 96, 32))
    ck.data = l2b.synth_checkpoint_host(ck, 1)
    with pytest.raises(l2b.L2BError) as e:
        l2b.Transformer(ck)
    assert e.value.status == -4
    with pytest.raises(l2b.L2BError):
        l2b.matmul(np.zeros(3, np.float32), np.ones(3, np.float32), np.ones(9, np.float32))


def test_checkpoint_floats_matches_real_file(l2b, tmp_path):
    """stories15M.bin's own 28-byte header, padded with zeros to the real file's size (sparse)."""
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    with open(os.path.join(golden, "stories15M_t0_tokens.json")) as f:
        size = json.load(f)["checkpoint_bytes"]
    path = tmp_path / "stories15M.bin"
    with open(os.path.join(golden, "stories15M_header.bin"), "rb") as f, open(path, "wb") as out:
        out.write(f.read())
        out.truncate(size)
    ck = l2b.read_checkpoint(str(path))
    assert ck.shape_tuple == (288, 768, 6, 6, 6, 32000, 256) and ck.shared_weights
    assert l2b.checkpoint_floats(ck) == ck.data.size == (os.path.getsize(path) - 28) // 4


def test_product_never_references_the_oracle():
    """oracle/ is test infrastructure: nothing under the product package may import, link or
    dlopen it."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "llama2.zig_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h", "Makefile")):
                text = open(os.path.join(dirpath, fn), errors="replace").read()
                assert "liborc" not in text and "oracle_lib" not in text and "llama2_oracle" not in text, (dirpath, fn)
