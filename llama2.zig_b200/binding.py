"""ctypes binding of include/llama2_b200.h (the C ABI that replaces transformer()).

Function names follow the reference (/root/reference/src/main.zig): `Transformer.forward`
is `transformer(token, pos, ...)` (:285), and the module-level `matmul`, `rmsnorm`,
`softmax`, `vector_weighted_sum_rows` run the same device code on host buffers so the
reference's unit tests (:1078-1150) can be replayed against the GPU.
"""
import ctypes as C
import os
import re

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)


class L2BError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"l2b status {status}: {message}")
        self.status = status


class L2BConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("dim", "hidden_dim", "n_layers", "n_heads", "n_kv_heads", "vocab_size", "seq_len",
                 "shared_weights")]


class L2BKernelTime(C.Structure):
    _fields_ = [("name", C.c_char * 24), ("layer", C.c_int32), ("ms", C.c_float), ("bytes", C.c_uint64)]


class L2BProbIndex(C.Structure):
    _fields_ = [("prob", C.c_float), ("index", C.c_int32)]


class L2BShard(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world_size", C.c_int32), ("device", C.c_int32),
                ("reserved", C.c_int32), ("comm_id", C.c_uint8 * 128)]


FP = C.POINTER(C.c_float)
IP = C.POINTER(C.c_int32)
U64P = C.POINTER(C.c_uint64)


def lib_path():
    return os.path.join(_HERE, "lib", "libllama2_b200.so")


def header_path():
    return os.path.join(_ROOT, "include", "llama2_b200.h")


def exported_symbols():
    """Names of every function include/llama2_b200.h declares."""
    with open(header_path()) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(l2b_[a-z0-9_]+)\s*\(", text)))


_lib = None


def load_library():
    """dlopen the CUDA library.  Raises L2BError if it has not been built: no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise L2BError(-3, f"{path} not built (run __graft_entry__.build()); there is no CPU fallback")
    lib = C.CDLL(path)
    vp = C.c_void_p
    lib.l2b_create.argtypes = [C.POINTER(vp), C.POINTER(L2BConfig), FP, C.c_uint64, FP, FP, C.c_int32]
    lib.l2b_create_sharded.argtypes = [C.POINTER(vp), C.POINTER(L2BConfig), FP, C.c_uint64, FP, FP,
                                       C.POINTER(L2BShard)]
    lib.l2b_create_synthetic.argtypes = [C.POINTER(vp), C.POINTER(L2BConfig), C.c_uint64,
                                         C.POINTER(L2BShard)]
    lib.l2b_create_synthetic_group.argtypes = [C.POINTER(vp), C.POINTER(L2BConfig), C.c_uint64, C.c_int32]
    lib.l2b_create_stream.argtypes = [C.POINTER(vp), vp]
    lib.l2b_forward_batch.argtypes = [C.POINTER(vp), C.c_int32, IP, IP, FP]
    lib.l2b_generate_argmax_batch.argtypes = [C.POINTER(vp), C.c_int32, IP, IP, C.c_int32, IP, C.c_int32, IP, IP]
    lib.l2b_destroy.argtypes = [vp]
    lib.l2b_destroy.restype = None
    lib.l2b_reset.argtypes = [vp]
    lib.l2b_forward.argtypes = [vp, C.c_int32, C.c_int32, FP]
    lib.l2b_forward_argmax.argtypes = [vp, C.c_int32, C.c_int32, IP]
    lib.l2b_forward_pinned.argtypes = [vp, C.c_int32, C.c_int32, C.POINTER(FP)]
    lib.l2b_generate_argmax.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, IP, C.c_int32, IP, IP]
    lib.l2b_prefill.argtypes = [vp, IP, C.c_int32, C.c_int32, FP]
    lib.l2b_logits_buffer.argtypes = [vp]
    lib.l2b_logits_buffer.restype = FP
    lib.l2b_forward_sample.argtypes = [vp, C.c_int32, C.c_int32, C.c_float, C.c_float, FP,
                                       C.POINTER(L2BProbIndex), C.c_int32, IP]
    lib.l2b_load_stats.argtypes = [vp, C.POINTER(C.c_double), U64P]
    lib.l2b_op_fused_matmul.argtypes = [C.c_int32, FP, FP, FP, FP, FP, C.c_int32, C.c_int32, C.c_int32]
    lib.l2b_op_sample_prep.argtypes = [C.c_int32, FP, C.c_int32, C.c_float, C.c_float,
                                       C.POINTER(L2BProbIndex), C.c_int32, IP]
    lib.l2b_last_error.argtypes = [vp]
    lib.l2b_last_error.restype = C.c_char_p
    lib.l2b_status_string.argtypes = [C.c_int32]
    lib.l2b_status_string.restype = C.c_char_p
    lib.l2b_abi_version.restype = C.c_int32
    lib.l2b_read_state.argtypes = [vp, C.c_int32, FP, C.c_uint64, U64P]
    lib.l2b_last_timing.argtypes = [vp, FP, IP]
    lib.l2b_step_bytes.argtypes = [vp, C.c_int32, U64P, U64P]
    lib.l2b_profile_step.argtypes = [vp, C.c_int32, C.c_int32, C.POINTER(L2BKernelTime), C.c_int32, IP]
    lib.l2b_comm_unique_id.argtypes = [C.POINTER(C.c_uint8 * 128)]
    lib.l2b_synth_fill_host.argtypes = [FP, C.c_uint64, C.c_uint64, C.c_uint64, C.c_double,
                                        C.c_double, C.c_float, C.c_float]
    lib.l2b_synth_fill_host.restype = None
    lib.l2b_synth_checkpoint_host.argtypes = [C.POINTER(L2BConfig), C.c_uint64, FP, C.c_uint64]
    lib.l2b_checkpoint_floats.argtypes = [C.POINTER(L2BConfig)]
    lib.l2b_checkpoint_floats.restype = C.c_uint64
    lib.l2b_op_matmul.argtypes = [C.c_int32, FP, FP, FP, C.c_int32, C.c_int32]
    lib.l2b_op_rmsnorm.argtypes = [C.c_int32, FP, FP, FP, C.c_int32]
    lib.l2b_op_softmax.argtypes = [C.c_int32, FP, C.c_int32]
    lib.l2b_op_weighted_sum_rows.argtypes = [C.c_int32, FP, C.c_int32, FP, C.c_int32, FP, C.c_int32]
    lib.l2b_op_attention_head.argtypes = [C.c_int32, FP, FP, FP, FP, C.c_int32, C.c_int32, C.c_int32]
    _lib = lib
    return lib


def _f32(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(FP)


def _check(rc, ctx=None):
    if rc != 0:
        lib = load_library()
        msg = lib.l2b_last_error(ctx).decode() or lib.l2b_status_string(rc).decode()
        raise L2BError(rc, msg)


def make_config(ck):
    """L2BConfig from a Checkpoint-like object (dim, hidden_dim, ..., shared_weights)."""
    return L2BConfig(ck.dim, ck.hidden_dim, ck.n_layers, ck.n_heads, ck.n_kv_heads, ck.vocab_size,
                     ck.seq_len, 1 if ck.shared_weights else 0)


def checkpoint_floats(ck):
    return int(load_library().l2b_checkpoint_floats(C.byref(make_config(ck))))


def comm_unique_id():
    buf = (C.c_uint8 * 128)()
    _check(load_library().l2b_comm_unique_id(C.byref(buf)))
    return bytes(buf)


def synth_checkpoint_host(ck, seed):
    """Host copy of the synthetic payload l2b_create_synthetic puts on the device."""
    lib = load_library()
    cfg = make_config(ck)
    n = int(lib.l2b_checkpoint_floats(C.byref(cfg)))
    data = np.empty(n, dtype=np.float32)
    _check(lib.l2b_synth_checkpoint_host(C.byref(cfg), seed, data.ctypes.data_as(FP), n))
    return data


STATE_IDS = {"x": 0, "xb": 1, "hb": 2, "q": 3, "key_cache": 4, "value_cache": 5, "logits": 6}


class Transformer:
    """Device-resident Weights + RunState and the `transformer(token, pos)` step.

    `ck` is a checkpoint.Checkpoint.  With `ck.data` set the payload is uploaded
    (l2b_create / l2b_create_sharded); with `synthetic_seed` the weights are generated on the
    device (l2b_create_synthetic).
    """

    def __init__(self, ck, synthetic_seed=None, rank=0, world_size=1, device=0, comm_id=None,
                 rope_cos=None, rope_sin=None, n_gpus=1, _stream_of=None):
        """n_gpus > 1: ONE process drives n_gpus GPUs (l2b_create(.., n_gpus)); rank/world_size:
        one process per GPU (l2b_create_sharded)."""
        self.lib = load_library()
        self.ck = ck
        self.cfg = make_config(ck)
        self.h = C.c_void_p()
        if _stream_of is not None:           # new_stream(): l2b_create_stream over another context's weights
            _check(self.lib.l2b_create_stream(C.byref(self.h), _stream_of.h), _stream_of.h)
            self._logits = np.empty(ck.vocab_size, dtype=np.float32)
            return
        shard = None
        assert n_gpus == 1 or world_size == 1
        if world_size > 1 or device != 0 or rank != 0:
            shard = L2BShard(rank, world_size, device, 0)
            if comm_id is not None:
                C.memmove(shard.comm_id, comm_id, 128)
        if synthetic_seed is not None and n_gpus > 1:
            rc = self.lib.l2b_create_synthetic_group(C.byref(self.h), C.byref(self.cfg), synthetic_seed, n_gpus)
        elif synthetic_seed is not None:
            rc = self.lib.l2b_create_synthetic(C.byref(self.h), C.byref(self.cfg), synthetic_seed,
                                               C.byref(shard) if shard else None)
        else:
            data = ck.data
            if data is None:
                raise ValueError("checkpoint has no payload and no synthetic_seed was given")
            if not (isinstance(data, np.ndarray) and data.dtype == np.float32 and data.flags["C_CONTIGUOUS"]):
                data = np.ascontiguousarray(data, dtype=np.float32)
            self._keep = data
            cp = data.ctypes.data_as(FP)
            rcos = rsin = None
            if rope_cos is not None:
                self._rc, rcos = _f32(rope_cos)
                self._rs, rsin = _f32(rope_sin)
            if shard is None:
                rc = self.lib.l2b_create(C.byref(self.h), C.byref(self.cfg), cp, data.size, rcos, rsin, n_gpus)
            else:
                rc = self.lib.l2b_create_sharded(C.byref(self.h), C.byref(self.cfg), cp, data.size, rcos,
                                                 rsin, C.byref(shard))
        if rc != 0:
            self.h = C.c_void_p()
            _check(rc, None)
        self._logits = np.empty(ck.vocab_size, dtype=np.float32)

    # -- lifecycle
    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.l2b_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def reset(self):
        _check(self.lib.l2b_reset(self.h), self.h)

    def new_stream(self):
        """Another decode stream over this context's device weights (l2b_create_stream): its own KV
        cache and run state, no upload.  The weights live as long as any context that uses them."""
        return Transformer(self.ck, _stream_of=self)

    # -- the hot path
    def forward(self, token, pos):
        """transformer(token, pos): returns state.logits (a fresh copy)."""
        _check(self.lib.l2b_forward(self.h, int(token), int(pos), self._logits.ctypes.data_as(FP)), self.h)
        return self._logits.copy()

    def forward_into(self, token, pos, out):
        _check(self.lib.l2b_forward(self.h, int(token), int(pos), out.ctypes.data_as(FP)), self.h)

    def forward_pinned(self, token, pos):
        p = FP()
        _check(self.lib.l2b_forward_pinned(self.h, int(token), int(pos), C.byref(p)), self.h)
        return np.ctypeslib.as_array(p, shape=(self.ck.vocab_size,))

    def forward_argmax(self, token, pos):
        nxt = C.c_int32()
        _check(self.lib.l2b_forward_argmax(self.h, int(token), int(pos), C.byref(nxt)), self.h)
        return nxt.value

    def prefill(self, tokens, pos0=0, want_logits=True):
        """tokens[i] at position pos0+i, all on the device (src/main.zig:996-1000 without the host loop);
        returns the logits of the last position, or None with want_logits=False."""
        toks = np.ascontiguousarray(tokens, dtype=np.int32)
        out = self._logits if want_logits else None
        _check(self.lib.l2b_prefill(self.h, toks.ctypes.data_as(IP), toks.size, int(pos0),
                                    out.ctypes.data_as(FP) if want_logits else None), self.h)
        return self._logits.copy() if want_logits else None

    def logits_buffer(self):
        """The library's pinned logits buffer as a numpy view (state.logits of the host, zero copy)."""
        return np.ctypeslib.as_array(self.lib.l2b_logits_buffer(self.h), shape=(self.ck.vocab_size,))

    def forward_sample(self, token, pos, temperature, top_p, cand_cap=8192):
        """transformer() + logits/=T, softmax (:1005-1008) and the top-p prefilter (:761-768) on the
        device.  Returns (probs, candidates or None); candidates is a structured array
        (prob, index) in index order, or None when top_p is 0/1 or too many passed the filter."""
        probs = np.empty(self.ck.vocab_size, dtype=np.float32)
        cand = (L2BProbIndex * cand_cap)()
        n = C.c_int32()
        _check(self.lib.l2b_forward_sample(self.h, int(token), int(pos), float(temperature), float(top_p),
                                           probs.ctypes.data_as(FP), cand, cand_cap, C.byref(n)), self.h)
        if n.value <= 0:
            return probs, None
        arr = np.frombuffer(cand, dtype=[("prob", "<f4"), ("index", "<i4")], count=n.value).copy()
        return probs, arr

    def load_stats(self):
        ms = C.c_double()
        nb = C.c_uint64()
        _check(self.lib.l2b_load_stats(self.h, C.byref(ms), C.byref(nb)), self.h)
        return ms.value, nb.value

    def generate_argmax(self, token, pos, n_steps, forced=None, stop_on_bos=True):
        out = np.full(max(n_steps, 1), -1, dtype=np.int32)
        done = C.c_int32()
        fp = None
        if forced is not None:
            forced = np.ascontiguousarray(forced, dtype=np.int32)
            assert forced.size >= n_steps
            fp = forced.ctypes.data_as(IP)
        _check(self.lib.l2b_generate_argmax(self.h, int(token), int(pos), int(n_steps), fp,
                                            1 if stop_on_bos else 0, out.ctypes.data_as(IP),
                                            C.byref(done)), self.h)
        return out[:done.value].copy()

    # -- introspection
    def state(self, name):
        n = C.c_uint64()
        ck = self.ck
        cap = max(ck.vocab_size, 2 * ck.n_layers * ck.seq_len * ck.dim, ck.hidden_dim)
        buf = np.empty(cap, dtype=np.float32)
        _check(self.lib.l2b_read_state(self.h, STATE_IDS[name], buf.ctypes.data_as(FP), cap, C.byref(n)), self.h)
        return buf[:n.value].copy()

    def last_timing(self):
        ms = C.c_float()
        k = C.c_int32()
        _check(self.lib.l2b_last_timing(self.h, C.byref(ms), C.byref(k)), self.h)
        return ms.value, k.value

    def profile_step(self, token, pos):
        """Per-kernel (name, layer, ms, algorithmic bytes) of one real step (CUDA events)."""
        cap = 8 * self.ck.n_layers + 8
        arr = (L2BKernelTime * cap)()
        n = C.c_int32()
        _check(self.lib.l2b_profile_step(self.h, int(token), int(pos), arr, cap, C.byref(n)), self.h)
        return [(arr[i].name.decode(), arr[i].layer, arr[i].ms, arr[i].bytes) for i in range(n.value)]

    def step_bytes(self, pos):
        w = C.c_uint64()
        kv = C.c_uint64()
        _check(self.lib.l2b_step_bytes(self.h, int(pos), C.byref(w), C.byref(kv)), self.h)
        return w.value, kv.value


# ---- several decode streams over one copy of the weights -------------------------------------

def _batch_args(streams, tokens, positions):
    n = len(streams)
    hs = (C.c_void_p * max(n, 1))(*[s.h.value for s in streams])
    toks = np.ascontiguousarray(tokens, dtype=np.int32)
    pos = np.ascontiguousarray(positions, dtype=np.int32)
    if toks.size != n or pos.size != n:
        raise ValueError("one token and one position per stream")
    return n, hs, toks, pos


def _batch_check(rc, streams):
    _check(rc, streams[0].h if streams else None)


def forward_batch(streams, tokens, positions):
    """One transformer() step on each stream (l2b_forward_batch): tokens[k] at positions[k] on
    streams[k], all Transformers over the same weights.  Returns (n, vocab) logits."""
    lib = load_library()
    n, hs, toks, pos = _batch_args(streams, tokens, positions)
    vocab = streams[0].ck.vocab_size if streams else 1
    out = np.empty((max(n, 1), vocab), dtype=np.float32)
    rc = lib.l2b_forward_batch(hs, n, toks.ctypes.data_as(IP), pos.ctypes.data_as(IP), out.ctypes.data_as(FP))
    _batch_check(rc, streams)
    return out[:n]


def generate_argmax_batch(streams, tokens, positions, n_steps, forced=None, stop_on_bos=True):
    """Transformer.generate_argmax for every stream at once on the device
    (l2b_generate_argmax_batch).  forced: (n, n_steps) ints, -1 = free-running, or None.  Returns a
    list with each stream's chosen tokens."""
    lib = load_library()
    n, hs, toks, pos = _batch_args(streams, tokens, positions)
    width = max(int(n_steps), 1)
    out = np.full((max(n, 1), width), -1, dtype=np.int32)
    done = np.zeros(max(n, 1), dtype=np.int32)
    fp = None
    if forced is not None:
        forced = np.ascontiguousarray(forced, dtype=np.int32).reshape(n, -1)
        if forced.shape[1] != n_steps:
            raise ValueError("forced must be (n, n_steps)")
        fp = forced.ctypes.data_as(IP)
    rc = lib.l2b_generate_argmax_batch(hs, n, toks.ctypes.data_as(IP), pos.ctypes.data_as(IP), int(n_steps), fp,
                                       1 if stop_on_bos else 0, out.ctypes.data_as(IP), done.ctypes.data_as(IP))
    _batch_check(rc, streams)
    return [out[k, :done[k]].copy() for k in range(n)]


# ---- reference-named single ops on host buffers (device = cuda:0) ---------------------------

def matmul(xout, x, w, device=0):
    """matmul(xout, x, w): W (d,n) @ x (n,) -> xout (d,)   (src/main.zig:485-498)."""
    x, xp = _f32(x)
    w, wp = _f32(w)
    d, n = xout.size, x.size
    assert w.size == d * n and w.size > 0            # asserts :534-536
    assert xout.dtype == np.float32
    _check(load_library().l2b_op_matmul(device, xout.ctypes.data_as(FP), xp, wp, d, n))
    return xout


def fused_matmul(x, gamma, w, d, resid=None, kernel=0, device=0):
    """W(d,n) . rmsnorm(x, gamma) (gamma None => W . x) through one GEMV kernel flavour
    (0 auto, 1 latency kernel, 2 register-fed streaming kernel, 3 TMA-ring kernel): the fused
    prologue (src/main.zig:432-468 + :485-498) and, with `resid`, the fused residual add
    (:395/:422: returns resid + W . xs) of the hot path in isolation."""
    x, xp = _f32(x)
    w, wp = _f32(w)
    gp = None
    if gamma is not None:
        gamma, gp = _f32(gamma)
    n = x.size
    assert w.size == d * n
    out = np.zeros(d, dtype=np.float32)
    rp = None
    if resid is not None:
        r = np.ascontiguousarray(resid, dtype=np.float32).copy()
        rp = r.ctypes.data_as(FP)
    _check(load_library().l2b_op_fused_matmul(device, out.ctypes.data_as(FP), xp, gp, wp, rp, d, n, kernel))
    return r if resid is not None else out


def sample_prep(logits, temperature, top_p, cand_cap=8192, device=0):
    """logits/=T, softmax, top-p prefilter on the device (src/main.zig:1005-1008, :761-768).
    Returns (probs, candidates-or-None, n_passed)."""
    probs = np.ascontiguousarray(logits, dtype=np.float32).copy()
    cand = (L2BProbIndex * cand_cap)()
    n = C.c_int32()
    _check(load_library().l2b_op_sample_prep(device, probs.ctypes.data_as(FP), probs.size, float(temperature),
                                             float(top_p), cand, cand_cap, C.byref(n)))
    arr = None
    if n.value > 0:
        arr = np.frombuffer(cand, dtype=[("prob", "<f4"), ("index", "<i4")], count=min(n.value, cand_cap)).copy()
    return probs, arr, n.value


def rmsnorm(o, x, w, device=0):
    """rmsnorm(o, x, w)   (src/main.zig:432-468)."""
    x, xp = _f32(x)
    w, wp = _f32(w)
    assert o.size == x.size == w.size                # asserts :433-434
    _check(load_library().l2b_op_rmsnorm(device, o.ctypes.data_as(FP), xp, wp, x.size))
    return o


def softmax(x, device=0):
    """softmax(x) in place   (src/main.zig:687-706)."""
    assert x.dtype == np.float32 and x.size > 0      # assert :688
    _check(load_library().l2b_op_softmax(device, x.ctypes.data_as(FP), x.size))
    return x


def vector_weighted_sum_rows(xout, rows, row_stride, weights, device=0):
    """vector_weighted_sum_rows(xout, rows, row_stride, weights)   (src/main.zig:657-685)."""
    rows, rp = _f32(rows)
    weights, wp = _f32(weights)
    assert xout.size > 0 and weights.size > 0 and row_stride >= xout.size      # :658-660
    assert rows.size >= (weights.size - 1) * row_stride + xout.size            # :661
    _check(load_library().l2b_op_weighted_sum_rows(device, xout.ctypes.data_as(FP), xout.size, rp,
                                                   row_stride, wp, weights.size))
    return xout


def attention_head(q, keys, values, device=0):
    """One head of src/main.zig:361-389 over keys/values of shape (n_pos, kv_stride)."""
    q, qp = _f32(q)
    keys, kp = _f32(keys)
    values, vp_ = _f32(values)
    n_pos, stride = keys.shape
    out = np.empty(q.size, dtype=np.float32)
    _check(load_library().l2b_op_attention_head(device, out.ctypes.data_as(FP), qp, kp, vp_, q.size,
                                                stride, n_pos))
    return out
