"""CPU: the C++ twin of the reference's Zig host (llama2.zig_b200/host) — loader, tokenizer and
sampler behave like src/main.zig.  The tokenizer checks are the reference's own `bpe` test
(src/main.zig:1152-1180) replayed on the shipped tokenizer.bin."""
import ctypes as C
import hashlib
import lzma
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOKENIZER_SHA256 = "74f899535f8f99cdeac697474b697f3fa40467b8376dab7b6c4d8c753f28ae9f"


@pytest.fixture(scope="module")
def host():
    path = os.path.join(ROOT, "llama2.zig_b200", "lib", "libllama2_host.so")
    if not os.path.exists(path):
        pytest.skip("host twin not built")
    C.CDLL(os.path.join(ROOT, "llama2.zig_b200", "lib", "libllama2_b200.so"), mode=C.RTLD_GLOBAL)
    lib = C.CDLL(path)
    lib.l2h_tokenizer_load.argtypes = [C.c_char_p, C.c_int32, C.POINTER(C.c_void_p)]
    lib.l2h_tokenizer_free.argtypes = [C.c_void_p]
    lib.l2h_tokenizer_max_token_len.argtypes = [C.c_void_p]
    lib.l2h_tokenizer_token.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]
    lib.l2h_tokenizer_token.restype = C.c_void_p
    lib.l2h_tokenizer_lookup.argtypes = [C.c_void_p, C.c_char_p, C.c_int32]
    lib.l2h_tokenizer_encode.argtypes = [C.c_void_p, C.c_char_p, C.c_int32, C.POINTER(C.c_int32), C.c_int32]
    lib.l2h_argmax.argtypes = [C.POINTER(C.c_float), C.c_int32]
    lib.l2h_softmax.argtypes = [C.POINTER(C.c_float), C.c_int32]
    lib.l2h_sample.argtypes = [C.POINTER(C.c_float), C.c_int32]
    lib.l2h_sample_top_p.argtypes = [C.POINTER(C.c_float), C.c_int32, C.c_float, C.c_void_p]
    lib.l2h_seed.argtypes = [C.c_uint64]
    return lib


@pytest.fixture(scope="module")
def tokenizer(tmp_path_factory):
    """The reference's shipped tokenizer.bin, stored xz-compressed under tests/golden."""
    with lzma.open(os.path.join(ROOT, "tests", "golden", "tokenizer.bin.xz")) as f:
        data = f.read()
    assert hashlib.sha256(data).hexdigest() == TOKENIZER_SHA256
    path = tmp_path_factory.mktemp("tokenizer") / "tokenizer.bin"
    path.write_bytes(data)
    return str(path)


def test_bpe(host, tokenizer):
    """test "bpe", src/main.zig:1152-1180."""
    tk = C.c_void_p()
    assert host.l2h_tokenizer_load(tokenizer.encode(), 32000, C.byref(tk)) == 0
    assert host.l2h_tokenizer_lookup(tk, "æ".encode(), 2) == 233
    n = C.c_int32()
    p = host.l2h_tokenizer_token(tk, 100, C.byref(n))
    assert C.string_at(p, n.value) == b"a"
    assert host.l2h_tokenizer_max_token_len(tk) == 27
    assert host.l2h_tokenizer_lookup(tk, b"a", 1) == 100
    text = b"A man dying of thirst is suddenly a mineral water critic?"
    out = (C.c_int32 * 128)()
    k = host.l2h_tokenizer_encode(tk, text, len(text), out, 128)
    assert list(out[:k]) == [68, 767, 27116, 310, 266, 765, 338, 11584, 263, 1375, 13537, 4094, 11164, 66]
    utf = "中".encode()
    k = host.l2h_tokenizer_encode(tk, utf, len(utf), out, 128)
    assert list(out[:k]) == [30275]
    host.l2h_tokenizer_free(tk)


def test_sampler_helpers(host):
    FP = C.POINTER(C.c_float)
    x = np.array([0, 5, 5, 1], dtype=np.float32)
    assert host.l2h_argmax(x.ctypes.data_as(FP), 4) == 1                     # first max wins (:720)
    y = np.array([1, 2, 3, 4], dtype=np.float32)
    host.l2h_softmax(y.ctypes.data_as(FP), 4)
    s = np.float32(0)
    for v in y:
        s = np.float32(s + v)
    assert s == 1.0                                                         # test "softmax" :1141-1150
    host.l2h_seed(7)
    probs = np.array([0.0, 0.0, 1.0, 0.0], dtype=np.float32)
    assert host.l2h_sample(probs.ctypes.data_as(FP), 4) == 2
    scratch = (C.c_uint64 * 8)()
    peaked = np.array([0.01, 0.97, 0.01, 0.01], dtype=np.float32)
    for _ in range(20):
        assert host.l2h_sample_top_p(peaked.ctypes.data_as(FP), 4, 0.9, scratch) == 1


def test_tokenizer_hash_lookup_equals_first_match_scan(host, tokenizer):
    """SURVEY 8f.4: the O(1) lookup must answer exactly like the reference's linear scan (:208-215):
    the FIRST id whose bytes match — the shipped vocabulary has 204 duplicated strings."""
    tk = C.c_void_p()
    assert host.l2h_tokenizer_load(tokenizer.encode(), 32000, C.byref(tk)) == 0
    first, dups = {}, 0
    n = C.c_int32()
    for i in range(32000):
        p = host.l2h_tokenizer_token(tk, i, C.byref(n))
        s = C.string_at(p, n.value)
        if s in first:
            dups += 1
        first.setdefault(s, i)
    assert dups == 204
    for s, i in first.items():
        assert host.l2h_tokenizer_lookup(tk, s, len(s)) == i
    assert host.l2h_tokenizer_lookup(tk, b"\xff\xfe-not-a-token", 14) == -1
    host.l2h_tokenizer_free(tk)


def test_top_p_on_prefiltered_candidates_equals_full_sampler(host):
    """The host half of the split sampler (:770-797 on the device's candidate list) picks the same
    token as sample_top_p on the full distribution (:752-798) for the same PRNG state."""
    FP = C.POINTER(C.c_float)

    class PI(C.Structure):
        _fields_ = [("prob", C.c_float), ("index", C.c_int32)]

    host.l2h_sample_top_p_candidates.argtypes = [C.POINTER(PI), C.c_int32, C.c_float]
    rng = np.random.default_rng(3)
    n, p = 32000, 0.9
    for trial in range(20):
        logits = (rng.standard_normal(n) * 3).astype(np.float32)
        probs = np.exp(logits - logits.max()).astype(np.float32)
        probs /= probs.sum(dtype=np.float32)
        cutoff = np.float32((np.float32(1) - np.float32(p)) / (np.float32(n) - np.float32(1)))
        keep = np.nonzero(probs >= cutoff)[0]
        cand = (PI * keep.size)(*[PI(float(probs[i]), int(i)) for i in keep])
        scratch = (C.c_uint64 * n)()
        host.l2h_seed(100 + trial)
        a = host.l2h_sample_top_p(probs.ctypes.data_as(FP), n, p, scratch)
        host.l2h_seed(100 + trial)
        b = host.l2h_sample_top_p_candidates(cand, keep.size, p)
        assert a == b
