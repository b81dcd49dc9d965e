"""Several decode streams over one copy of the weights: l2b_create_stream, l2b_forward_batch,
l2b_generate_argmax_batch.

Every batched result is compared with the same stream run alone: the stream context is reset and
replayed one token at a time, so no second copy of the weights is needed.  On llama2-7B shapes the
batch shares each pass over the weights (csrc/l2b_prefill.cuh) with the decode kernels' per-row
summation order, so the bar is 1e-6 and bit-identity is printed; on small shapes the batch calls run
each stream's own step and must match bit for bit."""
import ctypes as C

import numpy as np
import pytest

SHAPE_7B_2L = (4096, 11008, 2, 32, 32, -32000, 2048)
REL_TOL = 1e-4
BATCH_TOL = 1e-6


def rel_err(got, want):
    return float(np.max(np.abs(got.astype(np.float64) - want)) / (np.max(np.abs(want)) + 1e-30))


def prompt(n, k, vocab):
    """A distinct teacher-forced token sequence per stream k (SURVEY.md 8d's generator, shifted)."""
    return [(1 + 7919 * p + 104729 * k) % vocab for p in range(n)]


def replay(t, toks):
    """The stream alone, from an empty cache, one l2b_forward per token: last logits."""
    t.reset()
    for pos, tok in enumerate(toks):
        out = t.forward(tok, pos)
    return out


def kv_rows(t, n_layers, seq_len, kv_dim, n_pos):
    k, v = t.state("key_cache"), t.state("value_cache")
    rows = [slice(l * seq_len * kv_dim, l * seq_len * kv_dim + n_pos * kv_dim) for l in range(n_layers)]
    return np.concatenate([k[s] for s in rows]), np.concatenate([v[s] for s in rows])


# ---- argument checks that need no device (the library answers before any CUDA call) -------------
def test_batch_argument_checks_without_device(l2b):
    lib = l2b.load_library()
    toks = (C.c_int32 * 9)(*([1] * 9))
    pos = (C.c_int32 * 9)()
    logits = (C.c_float * 9)()
    out = (C.c_int32 * 9)()
    done = (C.c_int32 * 9)()
    streams = (C.c_void_p * 9)()
    assert lib.l2b_forward_batch(None, 1, toks, pos, logits) == -1                  # NULL stream list
    assert lib.l2b_generate_argmax_batch(None, 1, toks, pos, 1, None, 0, out, done) == -1
    for n in (0, 9, -1):
        assert lib.l2b_forward_batch(streams, n, toks, pos, logits) == -1
        assert lib.l2b_generate_argmax_batch(streams, n, toks, pos, 1, None, 0, out, done) == -1
    assert lib.l2b_forward_batch(streams, 2, toks, pos, logits) == -1               # NULL stream in the list
    h = C.c_void_p()
    assert lib.l2b_create_stream(C.byref(h), None) == -1                            # NULL base
    assert lib.l2b_create_stream(None, None) == -1
    assert h.value is None


# ---- GPU ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def seven(l2b):
    """A 2-layer llama2-7B-shaped model (seed 7) with a base context and 7 streams over its weights."""
    from llama2_zig_b200.checkpoint import shape_checkpoint
    ck = shape_checkpoint(SHAPE_7B_2L)
    base = l2b.Transformer(ck, synthetic_seed=7)
    streams = [base] + [base.new_stream() for _ in range(7)]
    yield ck, streams
    for s in reversed(streams):
        s.close()


@pytest.mark.gpu
def test_forward_batch_equals_each_stream_alone(l2b, oracle, seven):
    ck, all_streams = seven
    streams = all_streams[:4]
    V, S, kvd, L = ck.vocab_size, ck.seq_len, 4096, 2
    lens = [5, 9, 12, 17]
    seqs = [prompt(n + 1, k, V) for k, n in enumerate(lens)]
    for t, toks, n in zip(streams, seqs, lens):
        t.reset()
        assert t.prefill(toks[:n], 0, want_logits=False) is None
    got = l2b.forward_batch(streams, [s[-1] for s in seqs], lens)
    assert got.shape == (4, V)
    ms, launches = streams[0].last_timing()
    assert ms > 0 and launches > 0
    batched_kv = [kv_rows(t, L, S, kvd, n + 1) for t, n in zip(streams, lens)]
    identical = True
    for k, (t, toks, n) in enumerate(zip(streams, seqs, lens)):
        want = replay(t, toks)
        assert rel_err(got[k], want) <= BATCH_TOL, k
        ka, va = kv_rows(t, L, S, kvd, n + 1)
        kb, vb = batched_kv[k]
        assert np.max(np.abs(ka - kb)) <= BATCH_TOL * np.max(np.abs(ka)), k
        assert np.max(np.abs(va - vb)) <= BATCH_TOL * np.max(np.abs(va)), k
        identical = identical and np.array_equal(got[k], want) and np.array_equal(ka, kb) and np.array_equal(va, vb)
    print("forward_batch bit-identical to each stream alone:", identical)
    # one stream against the strict oracle
    data = l2b.synth_checkpoint_host(ck, 7)
    om = oracle.OracleModel(oracle.make_config(*ck.shape_tuple), data, ck.shared_weights, W=8, kind="strict")
    for pos, tok in enumerate(seqs[1]):
        ref = om.forward(tok, pos)
    om.close()
    assert rel_err(got[1], ref) <= REL_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 3, 4, 5, 8])
def test_generate_argmax_batch_equals_each_stream_alone(l2b, seven, n):
    ck, all_streams = seven
    streams = all_streams[:n]
    V, steps = ck.vocab_size, 6
    lens = [3 + 2 * k for k in range(n)]
    seqs = [prompt(m + 1, k, V) for k, m in enumerate(lens)]
    forced = np.full((n, steps), -1, dtype=np.int32)
    for k in range(1, n, 2):                       # odd streams teacher-forced, except one free step
        forced[k] = prompt(steps, k + 50, V)
        forced[k, 2] = -1

    def start():
        for t, toks, m in zip(streams, seqs, lens):
            t.reset()
            t.prefill(toks[:m], 0, want_logits=False)

    start()
    got = l2b.generate_argmax_batch(streams, [s[-1] for s in seqs], lens, steps, forced=forced, stop_on_bos=False)
    for k, t in enumerate(streams):
        t.reset()
        t.prefill(seqs[k][:lens[k]], 0, want_logits=False)
        want = t.generate_argmax(seqs[k][-1], lens[k], steps, forced=forced[k], stop_on_bos=False)
        assert len(got[k]) == steps
        assert np.array_equal(got[k], want), (k, got[k], want)

    # stop on BOS: stream 0 is forced to emit token 1 at step 2 and stops; the others run on
    forced_bos = forced.copy()
    forced_bos[0, 2] = 1
    start()
    S, kvd = ck.seq_len, 4096
    before = streams[0].state("key_cache")
    got = l2b.generate_argmax_batch(streams, [s[-1] for s in seqs], lens, steps, forced=forced_bos, stop_on_bos=True)
    after = streams[0].state("key_cache")
    assert len(got[0]) == 3 and got[0][-1] == 1
    for l in range(2):                             # rows after the stop are untouched
        tail = slice(l * S * kvd + (lens[0] + 3) * kvd, l * S * kvd + (lens[0] + steps + 1) * kvd)
        assert np.array_equal(before[tail], after[tail])
    for k, t in enumerate(streams):
        t.reset()
        t.prefill(seqs[k][:lens[k]], 0, want_logits=False)
        want = t.generate_argmax(seqs[k][-1], lens[k], steps, forced=forced_bos[k], stop_on_bos=True)
        assert np.array_equal(got[k], want), (k, got[k], want)
        if k:
            assert len(got[k]) == steps or (len(got[k]) and got[k][-1] == 1)


@pytest.mark.gpu
def test_batch_streams_across_attention_splits(l2b, seven):
    """One stream past position 256 (attention runs with timeline splits) next to one at position 10."""
    ck, all_streams = seven
    a, b = all_streams[:2]
    V = ck.vocab_size
    sa, sb = prompt(301, 0, V), prompt(11, 1, V)
    a.reset(); b.reset()
    a.prefill(sa[:300], 0, want_logits=False)
    b.prefill(sb[:10], 0, want_logits=False)
    got = l2b.forward_batch([a, b], [sa[300], sb[10]], [300, 10])
    assert rel_err(got[0], replay(a, sa)) <= BATCH_TOL
    assert rel_err(got[1], replay(b, sb)) <= BATCH_TOL
    # a device loop that crosses the 256 boundary on one stream only
    a.reset(); b.reset()
    a.prefill(sa[:254], 0, want_logits=False)
    b.prefill(sb[:10], 0, want_logits=False)
    got = l2b.generate_argmax_batch([a, b], [sa[254], sb[10]], [254, 10], 5, stop_on_bos=False)
    a.reset(); b.reset()
    a.prefill(sa[:254], 0, want_logits=False)
    b.prefill(sb[:10], 0, want_logits=False)
    assert np.array_equal(got[0], a.generate_argmax(sa[254], 254, 5, stop_on_bos=False))
    assert np.array_equal(got[1], b.generate_argmax(sb[10], 10, 5, stop_on_bos=False))


def stories15m_base(l2b):
    from llama2_zig_b200.checkpoint import shape_checkpoint
    return l2b.Transformer(shape_checkpoint("stories15M"), synthetic_seed=15)


@pytest.mark.gpu
def test_batch_calls_on_small_shapes_equal_single_stream(l2b):
    """stories15M shape: no batched weight pass; the batch calls run each stream's own step."""
    base = stories15m_base(l2b)
    streams = [base, base.new_stream(), base.new_stream()]
    V = base.ck.vocab_size
    lens = [4, 7, 2]
    seqs = [prompt(m + 1, k, V) for k, m in enumerate(lens)]
    for t, s, m in zip(streams, seqs, lens):
        t.prefill(s[:m], 0, want_logits=False)
    got = l2b.forward_batch(streams, [s[-1] for s in seqs], lens)
    for k, t in enumerate(streams):
        assert np.array_equal(got[k], replay(t, seqs[k])), k
    for t, s, m in zip(streams, seqs, lens):
        t.reset()
        t.prefill(s[:m], 0, want_logits=False)
    gen = l2b.generate_argmax_batch(streams, [s[-1] for s in seqs], lens, 8, stop_on_bos=False)
    for k, t in enumerate(streams):
        t.reset()
        t.prefill(seqs[k][:lens[k]], 0, want_logits=False)
        assert np.array_equal(gen[k], t.generate_argmax(seqs[k][-1], lens[k], 8, stop_on_bos=False)), k
    for t in reversed(streams):
        t.close()


@pytest.mark.gpu
def test_streams_share_weights_and_outlive_their_base(l2b):
    from llama2_zig_b200.checkpoint import shape_checkpoint
    ck = shape_checkpoint("stories15M")
    ck.data = l2b.synth_checkpoint_host(ck, 15)
    base = l2b.Transformer(ck)                            # uploads the host payload
    a, b = base.new_stream(), base.new_stream()
    assert a.load_stats()[1] == 0 and b.load_stats()[1] == 0
    assert base.load_stats()[1] > 0
    V = base.ck.vocab_size
    sa, sb = prompt(6, 0, V), prompt(6, 1, V)
    want_a, want_b = replay(a, sa), replay(b, sb)
    assert np.array_equal(replay(base, sa), want_a)       # a stream computes what its base computes
    base.close()                                          # the weights stay while a stream uses them
    assert np.array_equal(replay(a, sa), want_a)
    a.reset()                                             # resetting one stream leaves the other's cache alone
    a.forward(sb[0], 0)
    assert np.array_equal(b.forward(sb[5], 5), want_b)
    a.close()
    assert np.array_equal(b.forward(sb[5], 5), want_b)
    b.close()


@pytest.mark.gpu
def test_batch_call_errors(l2b):
    base = stories15m_base(l2b)
    other = stories15m_base(l2b)
    s = base.new_stream()
    for t in (base, s, other):
        t.forward(1, 0)

    def status(fn, *a, **kw):
        with pytest.raises(l2b.L2BError) as e:
            fn(*a, **kw)
        return e.value.status

    assert status(l2b.forward_batch, [base, other], [1, 1], [1, 1]) == -1          # different weights
    assert status(l2b.forward_batch, [base, base], [1, 1], [1, 1]) == -1           # listed twice
    assert status(l2b.forward_batch, [base] * 9, [1] * 9, [0] * 9) == -1           # n > L2B_MAX_BATCH
    assert status(l2b.forward_batch, [base, s], [1, 32000], [1, 1]) == -1          # token out of range
    assert status(l2b.forward_batch, [base, s], [1, 1], [1, 256]) == -1            # pos == seq_len
    assert status(l2b.forward_batch, [base, s], [1, 1], [1, 5]) == -7              # skips ahead of the cache
    assert status(l2b.generate_argmax_batch, [base, s], [1, 1], [1, 5], 3) == -7
    assert status(l2b.generate_argmax_batch, [base, other], [1, 1], [1, 1], 3) == -1
    got = l2b.forward_batch([base, s], [1, 1], [1, 1])                             # still usable afterwards
    assert np.array_equal(got[0], got[1])
    for t in (s, base, other):
        t.close()


@pytest.mark.gpu
def test_create_stream_over_two_gpus_is_unsupported(l2b):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from llama2_zig_b200.checkpoint import shape_checkpoint
    with l2b.Transformer(shape_checkpoint("stories15M"), synthetic_seed=15, n_gpus=2) as t:
        with pytest.raises(l2b.L2BError) as e:
            t.new_stream()
        assert e.value.status == -2


@pytest.mark.gpu
@pytest.mark.slow
def test_llama2_7b_full_depth_batch(l2b):
    """All 32 layers of llama2-7B (device-generated, seed 7): a base and 3 streams, 4 batched steps."""
    from llama2_zig_b200.checkpoint import shape_checkpoint
    ck = shape_checkpoint("llama2-7B")
    V = ck.vocab_size
    base = l2b.Transformer(ck, synthetic_seed=7)
    streams = [base] + [base.new_stream() for _ in range(3)]
    lens = [1, 2, 3, 4]
    seqs = [prompt(m + 4, k, V) for k, m in enumerate(lens)]
    for t, s, m in zip(streams, seqs, lens):
        t.prefill(s[:m], 0, want_logits=False)
    got = []
    for i in range(4):
        got.append(l2b.forward_batch(streams, [s[m + i] for s, m in zip(seqs, lens)], [m + i for m in lens]))
    for k, t in enumerate(streams):
        t.reset()
        for pos, tok in enumerate(seqs[k]):
            out = t.forward(tok, pos)
            if pos >= lens[k]:
                assert rel_err(got[pos - lens[k]][k], out) <= BATCH_TOL, (k, pos)
    for t in reversed(streams):
        t.close()
