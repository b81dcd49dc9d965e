#!/usr/bin/env python
"""bench.py — tokens/s of the llama2.zig decode hot path on B200, with its HBM roofline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload ...]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W

Workloads (BASELINE.json `configs`):
  llama2-7B    synthetic fp32, 256 positions, teacher-forced          (configs[3]/[4]) THE HEADLINE AT EVERY N
               (the metric names it and it fits one GPU, so the 1/2/4/8-GPU curve is one workload);
               N > 1: tensor-parallel, row/column shards + all-reduce of the hidden vector fused
               into the wo / w2 GEMV kernels over NVLink peer memory
  stories15M   real stories15M.bin (assets/), -t 0, 256 positions    (configs[1])   under `also` at N=1
  stories110M  synthetic, 1024 positions, teacher-forced              (configs[2])   under `also` at N=1
`--workload X` or L2B_BENCH_WORKLOAD=X makes another workload the headline line.

A "step" is ONE decode run of the workload's positions from an empty KV cache.
  value      = positions / time with everything resident in HBM: the on-device loop
               (l2b_generate_argmax: argmax fused in the classifier, no host round trip).
  e2e.value  = the same positions through the reference-facing call with HOST buffers: the
               C++ twin of the reference's loop (src/main.zig:995-1042) calling
               l2b_forward(ctx, token, pos, host_logits) and sampling (argmax) on the host, so
               every position pays its H2D (token,pos) and D2H (vocab*4 bytes of logits).
  roofline   = dominant kernel's algorithmic bytes / its CUDA-event duration inside real steps,
               against the measured HBM copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline = the oracle's -O3 build (a C port of the reference, NOT the Zig binary: no Zig
               toolchain exists here) on one host core, on a bounded sample.
`--impl reference` times that CPU port alone and prints the same JSON shape.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# rank 0 must print exactly ONE line on stdout: keep NCCL's version banner off it
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"

WORKLOADS = {
    #               shape key      positions  real file?
    "stories15M": ("stories15M", 256, True),
    "stories110M": ("stories110M", 1024, False),
    "llama2-7B": ("llama2-7B", 256, False),
}
SYNTH_SEED = {"stories15M": 15, "stories110M": 110, "llama2-7B": 7}
L2_FLUSH_BYTES = 256 << 20   # > 126 MB L2
KV_SAMPLE = 1 << 20          # floats kept per cache by --dump-outputs
SYNTH_DESC = "synthetic (counter-based N(0,s) weights, same generator on GPU and CPU; teacher-forced tokens)"


def teacher_tokens(n, vocab):
    return np.array([(1 + 7919 * p) % vocab for p in range(n)], dtype=np.int32)   # SURVEY.md 8d


def bench_config(workload, positions, world):
    """The `config` object of the JSON line: identical keys and values for the GPU arm and the
    reference arm (the driver compares them)."""
    return {"workload": workload, "positions_per_step": positions, "temperature": 0,
            "parallelism": "tp%d" % world if world > 1 else "single GPU",
            "l2": "L2 flushed (256 MiB memset) before every timed step" if workload != "llama2-7B"
                  else "inputs (26 GB of weights) exceed L2; L2 also flushed before every timed step",
            "step": "one decode run of positions_per_step positions from an empty KV cache"}


def pick_workload(args):
    w = args.workload
    if w == "auto":
        w = os.environ.get("L2B_BENCH_WORKLOAD", "llama2-7B")
    if w not in WORKLOADS:
        raise SystemExit(f"unknown workload {w}")
    return w


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _loop(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._loop, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle's fast build (a C port of src/main.zig:285-713), one thread.
# ----------------------------------------------------------------------------------------------
class CpuPort:
    """The oracle's fast build on one host core; the model is built once, samples are timed on it."""

    def __init__(self, workload):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        from llama2_zig_b200.checkpoint import shape_checkpoint

        self.workload = workload
        shape_key, self.positions, real = WORKLOADS[workload]
        real_path = os.path.join(ROOT, "assets", "stories15M.bin")
        if real and os.path.exists(real_path):
            cfg, shared, data = O.read_checkpoint(real_path, "fast")
            self.forced = None
        else:
            ck = shape_checkpoint(shape_key)
            cfg, shared = O.make_config(*ck.shape_tuple), ck.shared_weights
            data = O.synth_checkpoint(cfg, shared, SYNTH_SEED[workload], "fast")
            self.forced = teacher_tokens(self.positions + 1, ck.vocab_size)[1:]
        self.m = O.OracleModel(cfg, data, shared, W=8, kind="fast")
        t0 = time.perf_counter()
        self.m.forward(1, 0)
        self.per_tok = time.perf_counter() - t0

    def sample(self, budget_s):
        """Times a bounded sample (as many positions from pos 0 as fit the budget, <= one run)."""
        n = int(max(2, min(self.positions, budget_s / max(self.per_tok, 1e-9))))
        t0 = time.perf_counter()
        calls, _, _ = self.m.generate(1, n, forced=None if self.forced is None else self.forced[:n],
                                      stop_on_bos=False)
        dt = time.perf_counter() - t0
        return {"value": calls / dt, "unit": "tokens/s", "cores": 1, "kind": "port",
                "sample": f"{calls} positions of {self.workload} from pos 0 (oracle -O3 -mavx2 -mfma build, W=8, "
                          f"1 thread; C restatement of src/main.zig:285-713, not the Zig binary)",
                "seconds": dt}

    def close(self):
        self.m.close()


def cpu_port_run(workload, budget_s=12.0):
    port = CpuPort(workload)
    r = port.sample(budget_s)
    port.close()
    return r


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (the C port; the Zig binary
    cannot be built here) on the host, same workload / config / metric as the GPU arm.  A step is a
    bounded SAMPLE of the workload (the first n positions of the run) so that `--steps K --warmup W`
    ends within a few minutes; tokens/s is per sample, ms_per_step is scaled to the full run."""
    if rank != 0:
        return
    workload = pick_workload(args)
    positions = WORKLOADS[workload][1]
    total_budget = float(os.environ.get("L2B_BENCH_CPU_BUDGET_S", 150.0))
    warmup = max(args.warmup, 0)
    budget = total_budget / max(1, args.steps + warmup)
    port = CpuPort(workload)
    for _ in range(warmup):
        port.sample(budget)
    vals, r = [], None
    for _ in range(args.steps):
        r = port.sample(budget)
        vals.append(r["value"])
    port.close()
    v = float(np.mean(vals))
    sampled = int(r["sample"].split()[0])
    line = {"impl": "reference", "metric": "decode tokens/s", "value": v, "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup,
            "ms_per_step": 1e3 * positions / v, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32",
            "data": "stories15M.bin (real checkpoint, -t 0)" if workload == "stories15M"
                    else SYNTH_DESC,
            "config": bench_config(workload, positions, args.gpus),
            "sampled_positions_per_step": sampled,
            "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": 1, "kind": "port", "sample": r["sample"]},
            "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def step_outputs(t, positions, tokens, with_logits):
    """What the last timed step computed, as its caller would read it back: the logits of its last
    position (classifier output; single-GPU contexts only, a sharded context keeps them in per-rank
    slices), the final hidden state x (before the final rmsnorm), and the key / value cache rows of
    the positions it ran (float32), plus the token ids it returned (float64, exact).  Under teacher
    forcing those ids are the forced input, not a result.  A cache larger than KV_SAMPLE floats is
    reduced to a fixed, seeded sample so that a dump stays far below 64 MB."""
    out = {"tokens": np.asarray(tokens, dtype=np.float64), "x": t.state("x")}
    if with_logits:
        out["logits"] = t.state("logits")
    for name in ("key_cache", "value_cache"):
        cache = t.state(name)                                  # [n_layers][seq_len][kv width]
        per_layer = cache.size // t.ck.n_layers
        filled = per_layer // t.ck.seq_len * positions
        n = t.ck.n_layers * filled
        idx = np.arange(n) if n <= KV_SAMPLE else np.sort(np.random.default_rng(0).integers(0, n, KV_SAMPLE))
        out[name] = cache[idx // filled * per_layer + idx % filled]
    return out


def dump_outputs(dirname, outputs):
    """DIR/<workload>_<name>.npy for every array of step_outputs.  Inputs are seeded, so two builds
    run with the same arguments can be compared file for file."""
    os.makedirs(dirname, exist_ok=True)
    for workload, arrays in outputs.items():
        for name, a in arrays.items():
            np.save(os.path.join(dirname, f"{workload}_{name}.npy"), a)


def kernel_source_sha():
    import hashlib
    h = hashlib.sha256()
    for fn in ("l2b_device.cuh", "llama2_b200.cu"):
        with open(os.path.join(ROOT, "llama2.zig_b200", "csrc", fn), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def ncu_traffic(workload, kernel):
    """roofline.traffic = dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant
    kernel.  It can only come from an `ncu --set full` capture (never from a run under this script), so
    it is taken from profiles/r02_traffic.json — but ONLY if that capture was made from the kernel
    sources this run was built from (sha recorded by scripts/summarize_ncu.py); otherwise null."""
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        if rec.get("kernel_source_sha16") != kernel_source_sha():
            return None, None
        e = rec[workload][kernel]
        return float(e["traffic"]), e.get("source")
    except Exception:
        return None, None


def load_host_twin():
    import llama2_zig_b200 as l2b
    l2b.load_library()
    path = os.path.join(ROOT, "llama2.zig_b200", "lib", "libllama2_host.so")
    lib = C.CDLL(path)

    class GenOptions(C.Structure):
        _fields_ = [("temperature", C.c_float), ("top_p", C.c_float), ("n_steps", C.c_int32),
                    ("stop_on_bos", C.c_int32), ("use_device_argmax", C.c_int32), ("use_prefill", C.c_int32),
                    ("use_device_sampler", C.c_int32)]

    class GenResult(C.Structure):
        _fields_ = [("n_forward", C.c_int32), ("n_tokens", C.c_int32), ("secs_total", C.c_double),
                    ("secs_after_first", C.c_double), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64)]

    lib.l2h_generate.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(GenOptions), C.POINTER(C.c_int32), C.c_int32,
                                 C.c_void_p, C.POINTER(C.c_int32), C.c_int32, C.POINTER(GenResult)]
    return lib, GenOptions, GenResult


def tp_parity(t, ck, workload, rank, device, n_pos=4):
    """Outside the timed region: logits of the tensor-parallel context against a single-GPU context
    of the same synthetic weights that rank 0 builds beside its shard (BASELINE.json config 5:
    "logits vs the 1-GPU run <= 1e-4 rel").  Every rank steps the TP context (lockstep)."""
    import llama2_zig_b200 as l2b
    from llama2_zig_b200.checkpoint import shape_checkpoint
    toks = teacher_tokens(n_pos, ck.vocab_size)
    t.reset()
    tp_logits = [t.forward(int(tok), pos) for pos, tok in enumerate(toks)]
    tp_next = [t.forward_argmax(int(tok), pos) for pos, tok in enumerate(toks)]
    if rank != 0:
        return None
    worst, argmax_equal = 0.0, True
    with l2b.Transformer(shape_checkpoint(WORKLOADS[workload][0]), synthetic_seed=SYNTH_SEED[workload], device=device) as one:
        for pos, tok in enumerate(toks):
            ref = one.forward(int(tok), pos)
            worst = max(worst, float(np.max(np.abs(tp_logits[pos] - ref)) / np.max(np.abs(ref))))
            argmax_equal = argmax_equal and int(np.argmax(ref)) == int(np.argmax(tp_logits[pos])) == int(tp_next[pos])
    return {"vs": "single-GPU context of the same weights on rank 0's GPU", "positions": n_pos,
            "max_rel_logit_err": worst, "tolerance": 1e-4, "argmax_equal": bool(argmax_equal),
            "ok": bool(worst <= 1e-4 and argmax_equal)}


def run_workload(workload, args, rank, world, dist, sync, flush, clock_index):
    """Returns the result dict for one workload (all ranks participate; rank 0's dict is complete)."""
    import torch
    import llama2_zig_b200 as l2b
    from llama2_zig_b200.checkpoint import shape_checkpoint

    shape_key, positions, real = WORKLOADS[workload]
    if args.positions:
        positions = args.positions
    real_path = os.path.join(ROOT, "assets", "stories15M.bin")
    comm_id = None
    if world > 1:
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(l2b.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        comm_id = bytes(idt.cpu().numpy().tobytes())
    device = int(os.environ.get("LOCAL_RANK", 0)) if world > 1 else 0
    if real and os.path.exists(real_path) and world == 1:
        ck = l2b.read_checkpoint(real_path, mmap=False)
        t = l2b.Transformer(ck)
        data_desc, forced = "stories15M.bin (real checkpoint, -t 0)", None
    elif args.in_process > 1:
        ck = shape_checkpoint(shape_key)
        t = l2b.Transformer(ck, synthetic_seed=SYNTH_SEED[workload], n_gpus=args.in_process)
        data_desc = SYNTH_DESC
        forced = teacher_tokens(positions + 1, ck.vocab_size)[1:]
    else:
        ck = shape_checkpoint(shape_key)
        t = l2b.Transformer(ck, synthetic_seed=SYNTH_SEED[workload], rank=rank, world_size=world,
                            device=device, comm_id=comm_id)
        data_desc = SYNTH_DESC
        forced = teacher_tokens(positions + 1, ck.vocab_size)[1:]

    last = {}

    def device_run():
        t.reset()
        out = t.generate_argmax(1, 0, positions, forced=forced, stop_on_bos=False)
        assert len(out) == positions
        last["tokens"] = out
        return t.last_timing()

    def overwrite_state():
        """The same positions from other tokens (untimed): the context keeps logits, x and the KV cache
        across calls, and every warm-up run leaves the values the next step should compute, so without
        this a step that skipped a kernel would still leave the expected values behind."""
        t.reset()
        other = (teacher_tokens(positions + 1, ck.vocab_size)[1:] + 1) % ck.vocab_size
        t.generate_argmax(2, 0, positions, forced=other, stop_on_bos=False)

    host_lib, GenOptions, GenResult = load_host_twin()
    opt = GenOptions(0.0, 0.9, positions, 0, 0, 0, 0)
    res = GenResult()
    prompt = None if forced is None else forced.ctypes.data_as(C.POINTER(C.c_int32))
    n_prompt = 0 if forced is None else positions

    def e2e_run():
        t.reset()
        rc = host_lib.l2h_generate(t.h, C.byref(t.cfg), C.byref(opt), prompt, n_prompt, None, None, 0, C.byref(res))
        assert rc == 0, rc
        return res.secs_total, res.h2d_bytes, res.d2h_bytes

    # ---- warm-up
    for _ in range(max(args.warmup, 3)):
        device_run()
    e2e_run()

    # ---- timed: K device-resident steps, each bracketed by barrier + synchronize, L2 flushed before
    step_s, dev_ms, launches = [], [], 0
    with ClockSampler(clock_index) as clocks:
        for i in range(args.steps):
            if args.dump_outputs and i == args.steps - 1:
                overwrite_state()
            flush()
            sync()
            t0 = time.perf_counter()
            ms, k = device_run()
            sync()
            step_s.append(time.perf_counter() - t0)
            dev_ms.append(ms)
            launches += k
        outputs = (step_outputs(t, positions, last["tokens"], world == 1 and args.in_process <= 1)
                   if args.dump_outputs and rank == 0 else None)
        # ---- e2e: same positions through l2b_forward with host buffers
        e2e_s, h2d, d2h = [], 0, 0
        for _ in range(max(1, min(args.steps, 5))):
            flush()
            sync()
            t0 = time.perf_counter()
            _, h2d, d2h = e2e_run()
            sync()
            e2e_s.append(time.perf_counter() - t0)
        # ---- same loop with the -t 0 fast path of the boundary (l2b_forward_argmax: the reference's argmax
        # fused into the classifier epilogue, 4 bytes D2H per token instead of vocab * 4)
        opt_am = GenOptions(0.0, 0.9, positions, 0, 1, 0, 0)
        am_s = []
        if forced is None:                       # free-running stream only (a forced prompt never takes the argmax path)
            for _ in range(max(1, min(args.steps, 5))):
                t.reset()
                flush()
                sync()
                t0 = time.perf_counter()
                rc = host_lib.l2h_generate(t.h, C.byref(t.cfg), C.byref(opt_am), None, 0, None, None, 0, C.byref(res))
                assert rc == 0, rc
                sync()
                am_s.append(time.perf_counter() - t0)
        # ---- per-kernel roofline inside real steps (CUDA events between kernels, eager launches)
        t.reset()
        acc = {}
        prof_positions = list(range(0, positions, max(1, positions // 16)))
        tok = 1
        for pos in range(positions):
            if pos in prof_positions:
                for name, layer, ms, nbytes in t.profile_step(tok, pos):
                    a = acc.setdefault(name, [0.0, 0, 0])
                    a[0] += ms; a[1] += nbytes; a[2] += 1
            nxt = t.forward_argmax(tok, pos)     # (re-running a position is idempotent)
            tok = int(forced[pos]) if forced is not None else nxt
    # max over ranks
    tot = float(np.sum(step_s))
    e2e_tot = float(np.mean(e2e_s))
    if world > 1:
        v = torch.tensor([tot, e2e_tot, float(np.sum(dev_ms))], device="cuda", dtype=torch.float64)
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        tot, e2e_tot, dev_tot = (float(x) for x in v.cpu())
    else:
        dev_tot = float(np.sum(dev_ms))
    wbytes, _ = t.step_bytes(0)
    kv_total = sum(t.step_bytes(p)[1] for p in range(positions))
    step_bytes_total = wbytes * positions + kv_total            # this rank's algorithmic bytes per run
    peak, peak_src = measured_peak()
    kernels = {n: {"ms": a[0] / a[2], "bytes": a[1] // a[2], "gbs": (a[1] / a[2]) / (a[0] / a[2] * 1e-3) / 1e9,
                   "launches_sampled": a[2]} for n, a in acc.items()}
    dom = max(kernels, key=lambda n: kernels[n]["bytes"] * kernels[n]["launches_sampled"])
    traffic, traffic_src = ncu_traffic(workload, dom) if world == 1 else (None, None)
    value = positions * args.steps / tot
    out = {
        "workload": workload, "positions": positions, "value": value,
        "ms_per_step": 1e3 * tot / args.steps, "device_ms_per_step": dev_tot / args.steps,
        "launches": launches,
        "e2e": {"value": positions / e2e_tot, "unit": "tokens/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h),
                "path": "C++ host loop (twin of src/main.zig:995-1042) -> l2b_forward(host logits) -> host argmax",
                "device_argmax_variant": (positions / float(np.mean(am_s))) if am_s else None},
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["gbs"], "peak": peak, "unit": "GB/s",
                     "frac": kernels[dom]["gbs"] / peak, "traffic": traffic, "traffic_source": traffic_src,
                     "frac_of_8TBps_nominal": kernels[dom]["gbs"] / 8000.0, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": kernels[dom]["bytes"],
                     "avg_launch_ms": kernels[dom]["ms"]},
        "whole_step": {"algorithmic_bytes_per_run_per_gpu": int(step_bytes_total),
                       "achieved_gbs_per_gpu": step_bytes_total * args.steps / (dev_tot * 1e-3) / 1e9,
                       "frac_of_peak": step_bytes_total * args.steps / (dev_tot * 1e-3) / 1e9 / peak,
                       "frac_of_8TBps_nominal": step_bytes_total * args.steps / (dev_tot * 1e-3) / 1e9 / 8000.0,
                       "note": "stories15M's 61 MB of weights stay in the 126 MB L2 after the first token"
                               if workload == "stories15M" else "weights exceed L2: HBM-served"},
        "kernels": kernels, "clocks": clocks.summary(), "data": data_desc,
        "weights_bytes_per_token_per_gpu": int(wbytes), "outputs": outputs,
    }
    if world > 1 and forced is not None:
        out["parity"] = tp_parity(t, ck, workload, rank, device)
    if world == 1 and forced is not None and args.in_process <= 1:
        # prompt prefill (SURVEY 8f.2): the same positions as one prompt, on the device, no logits
        t.reset()
        t.prefill(np.concatenate([[1], forced[:positions - 1]]).astype(np.int32), 0, want_logits=False)
        t.reset()
        flush()
        t.prefill(np.concatenate([[1], forced[:positions - 1]]).astype(np.int32), 0, want_logits=False)
        pms, _ = t.last_timing()
        out["prefill"] = {"tokens": positions, "tokens_per_s": positions / (pms * 1e-3), "device_ms": pms,
                          "note": "l2b_prefill: prompt positions on the device, classifier skipped; "
                                  "4 positions per weight pass on bandwidth-bound shapes"}
    t.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto"] + list(WORKLOADS))
    ap.add_argument("--also", default="auto", help="comma list of extra workloads reported under 'also' (N=1 only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--positions", type=int, default=0, help="override positions per step (profiling runs only)")
    ap.add_argument("--in-process", type=int, default=0, metavar="N",
                    help="ONE process drives N GPUs (l2b_create(.., n_gpus=N), what the Zig CLI's --gpus uses) "
                         "instead of one process per GPU; run without torchrun")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what each workload's last timed step computed "
                         "(logits, x, sampled key/value cache; tokens, the forced input under teacher "
                         "forcing) to DIR/<workload>_<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200: the reference arm times a sample whose length varies")

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the hot path")
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl")
    if args.in_process > 1:
        args.gpus = args.in_process
    assert world == args.gpus or args.in_process > 1, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N>1)"
    flush_buf = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")

    def flush():
        flush_buf.zero_()

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    workload = pick_workload(args)
    clock_index = int(os.environ.get("LOCAL_RANK", 0))
    main_res = run_workload(workload, args, rank, world, dist, sync, flush, clock_index)
    outputs = {workload: main_res["outputs"]}
    also = {}
    if world == 1 and args.also != "none" and args.in_process <= 1:
        extra = ["stories15M", "stories110M"] if args.also == "auto" else [w for w in args.also.split(",") if w]
        for w in extra:
            if w != workload:
                r = run_workload(w, args, rank, world, dist, sync, flush, clock_index)
                outputs[w] = r["outputs"]
                also[w] = {k: r[k] for k in ("value", "ms_per_step", "device_ms_per_step", "e2e", "roofline",
                                             "whole_step", "kernels", "positions", "data", "prefill") if k in r}
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        cpu = None
        if not args.no_cpu_baseline and world == 1 and args.in_process <= 1:
            cpu = cpu_port_run(workload, budget_s=12.0)
            cpu.pop("seconds", None)
            try:
                cpu["host"] = subprocess.run("nproc; grep -m1 'model name' /proc/cpuinfo", shell=True,
                                             capture_output=True, text=True).stdout.strip().replace("\n", "; ")
            except Exception:
                pass
        line = {
            "metric": "decode tokens/s", "value": main_res["value"], "unit": "tokens/s", "n_gpus": max(world, args.in_process),
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": main_res["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": main_res["data"],
            "config": bench_config(workload, main_res["positions"], max(world, args.in_process)),
            "device_ms_per_step": main_res["device_ms_per_step"],
            "e2e": main_res["e2e"], "gpu_launches": main_res["launches"],
            "roofline": main_res["roofline"], "whole_step": main_res["whole_step"],
            "kernels": main_res["kernels"], "clocks": main_res["clocks"],
            "cpu_baseline": cpu, "also": also,
        }
        if main_res.get("parity") is not None:
            line["parity"] = main_res["parity"]
        if main_res.get("prefill") is not None:
            line["prefill"] = main_res["prefill"]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
