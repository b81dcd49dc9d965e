#!/usr/bin/env python
"""bench_batch.py — aggregate decode tok/s of B streams over one copy of the llama2-7B weights.

  python scripts/bench_batch.py [--batches 1,2,4,8] [--steps K] [--warmup W] [--positions P]

llama2-7B synthetic (seed 7, as bench.py).  A step is one l2b_generate_argmax_batch run of B
streams over P positions (default 256) from empty KV caches, each stream teacher-forced with its
own token sequence; L2 is flushed before every timed step.  Time is taken with CUDA events
(l2b_last_timing) and with a host clock around a synchronise.  The single-stream figure is
l2b_generate_argmax of the same positions on one stream, measured in the same process.

Parity: after the timed runs of each B, every stream is replayed alone (same forced tokens, except
the last step, which is free-running so that the device argmax is compared too), and the batched
tokens and the logits of the last position (l2b_forward_batch vs l2b_forward) must be identical.
Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import L2_FLUSH_BYTES, ClockSampler, teacher_tokens  # noqa: E402


def stream_tokens(k, n, vocab):
    """Distinct teacher-forced sequence of stream k (k = 0 is bench.py's)."""
    return ((teacher_tokens(n, vocab).astype(np.int64) + 104729 * k) % vocab).astype(np.int32)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        name, power, sm, sm_max = [c.strip() for c in out.split(",")]
        return {"name": name, "power_limit_w": float(power), "sm_mhz": float(sm), "sm_max_mhz": float(sm_max)}
    except Exception as e:                     # noqa: BLE001
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,2,4,8")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--positions", type=int, default=256)
    args = ap.parse_args()
    batches = [int(b) for b in args.batches.split(",")]

    import torch
    import llama2_zig_b200 as l2b
    from llama2_zig_b200.checkpoint import shape_checkpoint

    flush_buf = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")

    def flush():
        flush_buf.zero_()
        torch.cuda.synchronize()

    P = args.positions
    ck = shape_checkpoint("llama2-7B")
    V = ck.vocab_size
    base = l2b.Transformer(ck, synthetic_seed=7)
    streams = [base] + [base.new_stream() for _ in range(max(batches) - 1)]
    # stream k: token 1 at position 0, then its own sequence forced
    forced = [stream_tokens(k, P + 1, V)[1:] for k in range(len(streams))]

    def timed(fn):
        secs, dev = [], []
        for _ in range(args.warmup):
            fn()
        for _ in range(args.steps):
            flush()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            secs.append(time.perf_counter() - t0)
            dev.append(streams[0].last_timing()[0])
        return float(np.median(secs)), float(np.median(dev)) / 1e3

    def single():
        base.reset()
        out = base.generate_argmax(1, 0, P, forced=forced[0], stop_on_bos=False)
        assert len(out) == P

    result = {"workload": "llama2-7B synthetic (seed 7)", "positions_per_run": P, "steps": args.steps,
              "warmup": args.warmup, "l2": "flushed (256 MiB) before every timed step", "batch": {}}
    with ClockSampler(0) as clocks:
        s_host, s_dev = timed(single)
        single_tps = P / s_dev
        result["single_stream"] = {"tok_s": round(single_tps, 2), "host_tok_s": round(P / s_host, 2),
                                   "ms_per_step": round(1e3 * s_dev / P, 4)}
        parity = True
        for B in batches:
            group = streams[:B]
            fb = np.stack([forced[k] for k in range(B)])

            def run():
                for t in group:
                    t.reset()
                outs = l2b.generate_argmax_batch(group, [1] * B, [0] * B, P, forced=fb, stop_on_bos=False)
                assert all(len(o) == P for o in outs)
                return outs

            b_host, b_dev = timed(run)
            _, launches = streams[0].last_timing()
            # parity: last step free-running; tokens and last-position logits against each stream alone
            fp = fb.copy()
            fp[:, -1] = -1
            for t in group:
                t.reset()
            outs = l2b.generate_argmax_batch(group, [1] * B, [0] * B, P, forced=fp, stop_on_bos=False)
            last_in = [int(fp[k, -2]) for k in range(B)]
            lg = l2b.forward_batch(group, last_in, [P - 1] * B)
            for k, t in enumerate(group):
                t.reset()
                alone = t.generate_argmax(1, 0, P, forced=fp[k], stop_on_bos=False)
                parity = parity and np.array_equal(alone, outs[k]) and np.array_equal(t.forward(last_in[k], P - 1), lg[k])
            agg = B * P / b_dev
            result["batch"][str(B)] = {
                "aggregate_tok_s": round(agg, 2), "per_stream_tok_s": round(agg / B, 2),
                "host_aggregate_tok_s": round(B * P / b_host, 2), "ms_per_step": round(1e3 * b_dev / P, 4),
                "kernel_launches_per_step": round(launches / P, 1), "ratio_to_single_stream": round(agg / single_tps, 3)}
        result["parity"] = bool(parity)
    result["gpu"] = gpu_info()
    result["clocks_during_run"] = clocks.summary()
    for t in reversed(streams):
        t.close()
    print(json.dumps(result), flush=True)


if __name__ == "__main__":
    main()
