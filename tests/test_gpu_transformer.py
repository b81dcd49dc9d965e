"""GPU: transformer() parity through the C ABI (l2b_forward & friends) against the oracle.

Tolerances are the north star's: tokens identical at temperature 0, per-step logits within
1e-4 relative (measured as max|diff| / max|logit| per step)."""
import hashlib
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REL_TOL = 1e-4


def rel_err(got, want):
    return float(np.max(np.abs(got.astype(np.float64) - want)) / (np.max(np.abs(want)) + 1e-30))


def teacher_tokens(n, vocab):
    return [(1 + 7919 * p) % vocab for p in range(n)]      # SURVEY.md 8d


def is_argmax_within_tol(idx, logits):
    """idx is an argmax of `logits` up to REL_TOL: a near-tie may legitimately break either way when
    the summation order differs (as test_stories110m_full_depth_full_context allows)."""
    return float(logits[idx]) >= float(np.max(logits)) - REL_TOL * float(np.max(np.abs(logits)))


def stories15m_synthetic(l2b):
    """stories15M's shape with bench.py's synthetic weights (seed 15): the 61 MB checkpoint is not stored
    in the repository, and these tests need a model of that shape, not its trained weights."""
    from llama2_zig_b200.checkpoint import shape_checkpoint
    ck = shape_checkpoint("stories15M")
    ck.data = l2b.synth_checkpoint_host(ck, 15)
    return ck


def make_pair(l2b, oracle, shape, seed):
    from llama2_zig_b200.checkpoint import shape_checkpoint
    ck = shape_checkpoint(shape)
    ck.data = l2b.synth_checkpoint_host(ck, seed)
    om = oracle.OracleModel(oracle.make_config(*ck.shape_tuple), ck.data, ck.shared_weights, W=8, kind="strict")
    return ck, om


def test_stories15m_logits_and_tokens_match_oracle(l2b, oracle, stories15m):
    """configs[1]: stories15M.bin fp32 on 1xB200, -t 0, 256-token decode, bit-exact tokens."""
    with open(os.path.join(GOLDEN, "stories15M_t0_tokens.json")) as f:
        gold = json.load(f)
    ck = l2b.read_checkpoint(stories15m, mmap=False)
    cfg, shared, data = oracle.read_checkpoint(stories15m)
    om = oracle.OracleModel(cfg, data, shared, W=8, kind="strict")
    worst = 0.0
    with l2b.Transformer(ck) as t:
        token, toks = 1, []
        for pos in range(ck.seq_len):
            got = t.forward(token, pos)
            want = om.forward(token, pos)
            worst = max(worst, rel_err(got, want))
            nxt = int(np.argmax(got))
            assert nxt == int(np.argmax(want)), f"argmax differs at pos {pos}"
            if nxt == 1:
                break
            toks.append(nxt)
            token = nxt
    assert worst <= REL_TOL, worst
    assert toks == gold["tokens"]
    assert hashlib.sha256(np.array(toks, "<u4").tobytes()).hexdigest() == gold["sha256_le_u32"]


def test_stories15m_golden_logits_fixture(l2b, stories15m):
    """Same check against the committed fixture only (no oracle in the loop)."""
    gold = np.load(os.path.join(GOLDEN, "stories15M_logits.npz"))
    with open(os.path.join(GOLDEN, "stories15M_t0_tokens.json")) as f:
        toks = json.load(f)["tokens"] + [1]
    ck = l2b.read_checkpoint(stories15m, mmap=False)
    with l2b.Transformer(ck) as t:
        token = 1
        for pos in range(int(gold["positions"].max()) + 1):
            lg = t.forward(token, pos)
            if pos in gold["positions"]:
                scale = np.max(np.abs(gold[f"p{pos}_top_val"]))
                assert np.max(np.abs(lg[::16] - gold[f"p{pos}_strided"])) / scale <= REL_TOL
                assert np.max(np.abs(lg[gold[f"p{pos}_top_idx"]] - gold[f"p{pos}_top_val"])) / scale <= REL_TOL
                assert int(np.argmax(lg)) == int(gold[f"p{pos}_top_idx"][0])
            token = toks[pos]


def test_stories15m_argmax_and_generate_paths(l2b, stories15m):
    """l2b_forward_argmax and the on-device loop l2b_generate_argmax reproduce the stream."""
    with open(os.path.join(GOLDEN, "stories15M_t0_tokens.json")) as f:
        gold = json.load(f)
    ck = l2b.read_checkpoint(stories15m, mmap=False)
    with l2b.Transformer(ck) as t:
        token, toks = 1, []
        for pos in range(256):
            nxt = t.forward_argmax(token, pos)
            if nxt == 1:
                break
            toks.append(nxt)
            token = nxt
        assert toks == gold["tokens"]
        t.reset()
        out = t.generate_argmax(1, 0, 256, stop_on_bos=True)
        assert out[-1] == 1 and out[:-1].tolist() == gold["tokens"]
        assert len(out) == gold["forward_calls"]
        # without BOS-stop the loop runs all 256 positions; prefix is unchanged
        t.reset()
        out2 = t.generate_argmax(1, 0, 256, stop_on_bos=False)
        assert len(out2) == 256 and out2[:222].tolist() == out.tolist()
        # prompt forcing (src/main.zig:999-1000): forced tokens are fed, the rest free-runs
        t.reset()
        forced = np.full(256, -1, np.int32)
        forced[:5] = gold["tokens"][:5]
        out3 = t.generate_argmax(1, 0, 40, forced=forced, stop_on_bos=True)
        assert out3.tolist() == gold["tokens"][:40]


def test_rope_table_from_host_is_used(l2b, oracle):
    """rope_cos/rope_sin passed through the ABI (host libm) give the same result as the
    library's own table here (same libm); a deliberately wrong table must change the logits."""
    ck = stories15m_synthetic(l2b)
    hs = ck.dim // ck.n_heads
    import ctypes as C
    lib = oracle.load("strict")
    cos = np.zeros((ck.seq_len, hs // 2), np.float32)
    sin = np.zeros_like(cos)
    a, b = C.c_float(), C.c_float()
    for p in range(ck.seq_len):
        for j in range(hs // 2):
            lib.orc_rope_angle(2 * j, hs, p, C.byref(a), C.byref(b))
            cos[p, j], sin[p, j] = a.value, b.value
    with l2b.Transformer(ck) as t0, l2b.Transformer(ck, rope_cos=cos, rope_sin=sin) as t1, \
            l2b.Transformer(ck, rope_cos=np.ones_like(cos), rope_sin=np.zeros_like(sin)) as t2:
        for pos, tok in enumerate([1, 9038, 2501, 263]):
            l0, l1, l2_ = t0.forward(tok, pos), t1.forward(tok, pos), t2.forward(tok, pos)
            assert np.array_equal(l0, l1)
        assert not np.array_equal(l0, l2_)


@pytest.mark.parametrize("shape,seed,steps", [
    ((64, 172, 2, 4, 2, 96, 32), 3, 32),            # GQA branch (:314-320), odd-ish hidden, full context
    ((128, 344, 3, 4, 1, -200, 48), 4, 48),         # MQA + unshared classifier (:112, :942-944)
    ((288, 768, 6, 6, 6, 32000, 256), 15, 40),      # stories15M shape, synthetic weights
    ((768, 2048, 2, 12, 12, 32000, 1024), 110, 12), # stories110M shape, 2 layers
    ((4096, 11008, 1, 32, 32, -32000, 2048), 7, 6), # llama2-7B shape, 1 layer, unshared classifier
])
def test_synthetic_models_match_oracle_teacher_forced(l2b, oracle, shape, seed, steps):
    """Synthetic weights have no argmax margin, so compare logits under teacher forcing
    (SURVEY.md 7 'hard parts') and never free-run."""
    ck, om = make_pair(l2b, oracle, shape, seed)
    toks = teacher_tokens(steps, ck.vocab_size)
    with l2b.Transformer(ck) as t:
        for pos, tok in enumerate(toks):
            got = t.forward(tok, pos)
            want = om.forward(tok, pos)
            assert rel_err(got, want) <= REL_TOL, (pos, rel_err(got, want))
        # RunState parity of the last step (src/main.zig:119-135)
        kc = t.state("key_cache")
        np.testing.assert_allclose(kc, om.state("key_cache"), rtol=0, atol=1e-4 * np.max(np.abs(om.state("key_cache"))))
        vc = t.state("value_cache")
        np.testing.assert_allclose(vc, om.state("value_cache"), rtol=0, atol=1e-4 * np.max(np.abs(om.state("value_cache"))))


def test_device_synthetic_weights_equal_host_mirror(l2b, oracle):
    """l2b_create_synthetic (weights generated in HBM) == l2b_create on the host mirror of the
    same generator: the two contexts must produce bit-identical logits."""
    from llama2_zig_b200.checkpoint import shape_checkpoint
    ck = shape_checkpoint((128, 344, 3, 4, 2, -200, 48))
    ck.data = l2b.synth_checkpoint_host(ck, 21)
    with l2b.Transformer(ck) as a, l2b.Transformer(shape_checkpoint(ck.shape_tuple[:5] + (-200, 48)), synthetic_seed=21) as b:
        for pos, tok in enumerate(teacher_tokens(10, 200)):
            assert np.array_equal(a.forward(tok, pos), b.forward(tok, pos))


def test_long_context_attention_splits(l2b, oracle):
    """Full 1024-position context on a 1-layer 110M-shaped model: exercises the split-KV
    attention path at every length and the last position (maximum size edge case)."""
    ck, om = make_pair(l2b, oracle, (768, 2048, 1, 12, 12, 512, 1024), 5)
    toks = teacher_tokens(1024, 512)
    with l2b.Transformer(ck) as t:
        for pos, tok in enumerate(toks):
            got = t.forward(tok, pos)
            if pos % 97 == 0 or pos >= 1020 or pos in (63, 64, 65, 127, 128, 129):
                want = om.forward(tok, pos)
                assert rel_err(got, want) <= REL_TOL, (pos, rel_err(got, want))
            else:
                om.forward(tok, pos)


def test_call_order_and_argument_errors(l2b):
    ck = stories15m_synthetic(l2b)
    with l2b.Transformer(ck) as t:
        with pytest.raises(l2b.L2BError) as e:
            t.forward(1, 5)                      # skips ahead of the KV cache
        assert e.value.status == -7
        with pytest.raises(l2b.L2BError) as e:
            t.forward(32000, 0)                  # token out of range
        assert e.value.status == -1
        with pytest.raises(l2b.L2BError) as e:
            t.forward(1, 256)                    # pos == seq_len
        assert e.value.status == -1
        a = t.forward(1, 0)
        b = t.forward(1, 0)                      # re-running a position is allowed and idempotent
        assert np.array_equal(a, b)


def test_determinism_and_reset(l2b):
    ck = stories15m_synthetic(l2b)
    with l2b.Transformer(ck) as t:
        run1 = [t.forward(tok, pos) for pos, tok in enumerate([1, 9038, 2501, 263, 931])]
        t.reset()
        run2 = [t.forward(tok, pos) for pos, tok in enumerate([1, 9038, 2501, 263, 931])]
        for a, b in zip(run1, run2):
            assert np.array_equal(a, b)
        w, kv = t.step_bytes(0)
        assert w == 60_766_848                  # SURVEY.md 8d weight bytes per token
        assert kv == 4 * 6 * 2 * 288


# ---------------------------------------------------------------------------------------------
# Full-depth parity on the configurations that are benchmarked (VERDICT r1 "missing" #1): depth is
# where reordering error accumulates (src/main.zig:303).
# ---------------------------------------------------------------------------------------------
def test_stories110m_full_depth_full_context(l2b, oracle):
    """configs[2]: all 12 layers of the stories110M shape, synthetic weights (seed 110 = bench.py's),
    teacher-forced over the WHOLE 1024-position context; logits compared at >= 40 positions that
    include the attention-split boundaries 255/256/257, 511/512/513 and the last position 1023."""
    ck, om = make_pair(l2b, oracle, (768, 2048, 12, 12, 12, 32000, 1024), 110)
    toks = teacher_tokens(1024, ck.vocab_size)
    check = set(range(0, 1024, 32)) | {1, 2, 3, 255, 256, 257, 511, 512, 513, 767, 768, 769, 1021, 1022, 1023}
    worst = 0.0
    with l2b.Transformer(ck) as t:
        for pos, tok in enumerate(toks):
            got = t.forward(tok, pos)
            want = om.forward(tok, pos)
            if pos in check:
                e = rel_err(got, want)
                worst = max(worst, e)
                assert e <= REL_TOL, (pos, e)
                assert int(np.argmax(got)) == int(np.argmax(want)) or e < 1e-6   # synthetic logits can tie
    assert len(check) >= 40
    print(f"stories110M 12 layers x 1024 positions: max rel logit err {worst:.2e}")


@pytest.mark.slow
def test_llama2_7b_full_depth(l2b, oracle):
    """configs[3]: all 32 layers of llama2-7B (synthetic fp32 weights, seed 7 = bench.py's; unshared
    classifier), 4 teacher-forced positions against the strict oracle.  The GPU context is created
    from the HOST payload (27 GB through the pinned double-buffered upload, SURVEY 8f.3), and a
    second one from the on-device generator must give bit-identical logits."""
    import psutil
    if psutil.virtual_memory().available < 45 * (1 << 30):
        pytest.skip("needs ~30 GB of free host memory for the 7B payload")
    from llama2_zig_b200.checkpoint import shape_checkpoint
    ck = shape_checkpoint("llama2-7B")
    cfg = oracle.make_config(*ck.shape_tuple)
    ck.data = oracle.synth_checkpoint(cfg, ck.shared_weights, 7, "strict")      # multi-threaded generator, == the device's
    om = oracle.OracleModel(cfg, ck.data, ck.shared_weights, W=8, kind="strict")
    toks = teacher_tokens(4, ck.vocab_size)
    want = [om.forward(tok, pos) for pos, tok in enumerate(toks)]
    om.close()
    with l2b.Transformer(ck) as t:
        ms, nbytes = t.load_stats()
        assert nbytes >= 26_000_000_000 and ms > 0
        print(f"llama2-7B upload: {nbytes / 1e9:.2f} GB in {ms / 1e3:.2f} s = {nbytes / ms / 1e6:.2f} GB/s")
        got = [t.forward(tok, pos) for pos, tok in enumerate(toks)]
    ck.data = None
    for pos in range(4):
        e = rel_err(got[pos], want[pos])
        assert e <= REL_TOL, (pos, e)
    with l2b.Transformer(shape_checkpoint("llama2-7B"), synthetic_seed=7) as t2:
        for pos, tok in enumerate(toks):
            assert np.array_equal(t2.forward(tok, pos), got[pos]), pos


def test_forward_sample_matches_host_sampler_steps(l2b, oracle):
    """l2b_forward_sample: transformer() + logits/=T + softmax + top-p prefilter (:996, :1005-1012)
    against the oracle's logits pushed through the reference's own host-side steps."""
    import ctypes as C
    FP = C.POINTER(C.c_float)
    ck, om = make_pair(l2b, oracle, "stories15M", 15)
    lib = oracle.load("strict")
    with l2b.Transformer(ck) as t:
        tok = 1
        for pos, (temp, top_p) in enumerate([(1.0, 0.9), (0.8, 0.9), (1.0, 0.0), (1.5, 0.5), (0.5, 1.0), (1.0, 0.95)]):
            probs, cand = t.forward_sample(tok, pos, temp, top_p)
            raw = om.forward(tok, pos)
            nxt = int(np.argmax(raw))
            want = raw.copy()
            if temp != 1.0:
                want = (want / np.float32(temp)).astype(np.float32)
            ref64 = np.exp(want.astype(np.float64) - want.max())
            ref64 /= ref64.sum()
            lib.orc_softmax(want.ctypes.data_as(FP), want.size)
            # The bar is the exact softmax (1e-4, the north star's tolerance).  The reference itself sums the
            # 32000 exponentials sequentially in fp32 (:697-701): once the running sum has absorbed the
            # dominant term (~1.0), terms below its half-ulp (6e-8) are rounded away one by one, so on a sharp
            # distribution (p_max near 1, e.g. the trained stories15M at T = 0.5: 0.985) its normalisation is
            # off by up to ~1e-3.  The device's tree sum does not reproduce that loss; against the restatement
            # the bar is therefore 2e-3.  The argmax is compared up to a near-tie, the candidate set exactly.
            assert np.max(np.abs(probs - ref64)) <= 1e-4 * np.max(ref64)
            assert np.max(np.abs(probs - want)) <= 2e-3 * np.max(want)
            assert int(np.argmax(probs)) == nxt or is_argmax_within_tol(int(np.argmax(probs)), raw)
            if top_p in (0.0, 1.0):
                assert cand is None
            else:
                cutoff = np.float32((np.float32(1.0) - np.float32(top_p)) / (np.float32(want.size) - np.float32(1.0)))
                keep = np.nonzero(probs >= cutoff)[0]
                assert np.array_equal(cand["index"], keep.astype(np.int32))
                assert np.array_equal(cand["prob"], probs[keep])
            tok = nxt


def test_logits_buffer_is_zero_copy_state_logits(l2b):
    """A host that adopts l2b_logits_buffer() as state.logits (src/main.zig:149) gets the same
    logits as one that passes its own buffer."""
    ck = stories15m_synthetic(l2b)
    with l2b.Transformer(ck) as t:
        buf = t.logits_buffer()
        for pos, tok in enumerate([1, 9038, 2501]):
            own = t.forward(tok, pos)
            t.forward_into(tok, pos, buf)
            assert np.array_equal(own, buf)
        ms, nbytes = t.load_stats()
        assert nbytes == 60_816_028 - 28 - 4 * 2 * 256 * 24 and ms > 0      # stories15M.bin less header and freq_cis tables


def test_prefill_equals_token_by_token(l2b, oracle):
    """SURVEY 8f.2: l2b_prefill (all prompt positions on the device, classifier skipped where the
    reference discards the logits, src/main.zig:996-1000) leaves the same KV cache and returns the
    same logits as feeding the prompt through l2b_forward one token at a time — bit for bit."""
    with open(os.path.join(GOLDEN, "stories15M_t0_tokens.json")) as f:
        gold = json.load(f)["tokens"]
    prompt = [1] + gold[:23]                      # BOS + 23 story tokens
    ck, om = make_pair(l2b, oracle, "stories15M", 15)
    with l2b.Transformer(ck) as a, l2b.Transformer(ck) as b:
        for pos, tok in enumerate(prompt):
            want = a.forward(tok, pos)
            ref = om.forward(tok, pos)
        got = b.prefill(prompt, 0)
        assert np.array_equal(got, want)
        assert rel_err(got, ref) <= REL_TOL
        n = 6 * 256 * 288
        assert np.array_equal(a.state("key_cache")[:n], b.state("key_cache")[:n])
        assert np.array_equal(a.state("value_cache")[:n], b.state("value_cache")[:n])
        # continue decoding after a logits-free prefill of a longer prompt
        b.reset()
        assert b.prefill(prompt + gold[23:40], 0, want_logits=False) is None
        for pos in range(len(prompt), len(prompt) + 17):
            a.forward(gold[pos - 1], pos)
            om.forward(gold[pos - 1], pos)
        nxt_a = a.forward_argmax(gold[40], 41)
        nxt_b = b.forward_argmax(gold[40], 41)
        ref = om.forward(gold[40], 41)
        assert nxt_a == nxt_b
        assert nxt_a == int(np.argmax(ref)) or is_argmax_within_tol(nxt_a, ref)
        with pytest.raises(l2b.L2BError):
            b.prefill([1] * 300, 0)               # runs past seq_len


def test_batched_prefill_on_bandwidth_bound_shapes(l2b, oracle):
    """SURVEY 8f.2 on llama2-7B shapes (2 layers): l2b_prefill runs 4 prompt positions per pass over
    the weights (csrc/l2b_prefill.cuh).  KV cache and the next logits must equal the token-by-token
    path (same per-row summation order => expected bit-identical; bar 1e-6) and the oracle (1e-4)."""
    ck, om = make_pair(l2b, oracle, (4096, 11008, 2, 32, 32, -32000, 2048), 7)
    toks = teacher_tokens(12, ck.vocab_size)           # 11 silent positions = 2 full chunks + 3, then 1 with logits
    with l2b.Transformer(ck) as a, l2b.Transformer(ck) as b:
        for pos, tok in enumerate(toks):
            want = a.forward(tok, pos)
            ref = om.forward(tok, pos)
        got = b.prefill(toks, 0)
        ms, launches = b.last_timing()
        assert rel_err(got, ref) <= REL_TOL
        assert rel_err(got, want) <= 1e-6
        kv_a, kv_b = a.state("key_cache"), b.state("key_cache")
        va, vb = a.state("value_cache"), b.state("value_cache")
        S, kvd = 2048, 4096
        for l in range(2):
            sl = slice(l * S * kvd, l * S * kvd + 12 * kvd)
            assert np.max(np.abs(kv_a[sl] - kv_b[sl])) <= 1e-6 * np.max(np.abs(kv_a[sl]))
            assert np.max(np.abs(va[sl] - vb[sl])) <= 1e-6 * np.max(np.abs(va[sl]))
        print("batched prefill bit-identical to token-by-token:", bool(np.array_equal(got, want) and np.array_equal(kv_a[:12 * kvd], kv_b[:12 * kvd])))
        # decoding continues from the prefilled cache
        nxt = teacher_tokens(13, ck.vocab_size)[12]
        assert rel_err(b.forward(nxt, 12), a.forward(nxt, 12)) <= 1e-6


def test_batched_prefill_long_prompt_with_attention_splits(l2b):
    """A prompt longer than one attention split (> 256 positions on a 7B-shaped context): the batched
    prefill's attention runs with timeline splits and a per-(position, head) last-arriver merge.  Checked
    GPU against GPU: the same positions fed one by one (which the oracle tests pin) must give the same
    logits afterwards, and a second chunked call must continue a partly filled cache."""
    from llama2_zig_b200.checkpoint import shape_checkpoint
    shape = (4096, 11008, 2, 32, 32, -32000, 2048)
    toks = teacher_tokens(331, 32000)
    with l2b.Transformer(shape_checkpoint(shape), synthetic_seed=3) as a, \
            l2b.Transformer(shape_checkpoint(shape), synthetic_seed=3) as b:
        for pos, tok in enumerate(toks):
            want = a.forward(tok, pos)
        assert b.prefill(toks[:200], 0, want_logits=False) is None      # 50 chunks of 4
        got = b.prefill(toks[200:], 200)                                 # continues at pos 200, crosses 256; 131 = 32 chunks + 3
        assert rel_err(got, want) <= 1e-6
        assert int(np.argmax(got)) == int(np.argmax(want))
