"""Regenerates the committed golden fixtures from the CPU oracle (NOT from the Zig binary:
no Zig toolchain exists in this image, see oracle/llama2_oracle.h "Pinning status").

  stories15M_t0_tokens.json  token stream of `llama2 stories15M.bin -t 0` (no prompt) as the
                             oracle produces it; identical for W in {4,8,16}, strict/optimized
                             float mode; sha256 matches SURVEY.md Appendix B.
  stories15M_logits.npz      logits of selected positions along that stream (every 16th logit
                             + the top-32), oracle strict W=8.
  stories15M_header.bin      the checkpoint's 28-byte header (its size is in the tokens file).
  tokenizer.bin.xz           the shipped tokenizer.bin, xz-compressed.

Needs the real assets/stories15M.bin and assets/tokenizer.bin:  python tests/golden/make_golden.py
"""
import hashlib
import json
import lzma
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import oracle_lib as O  # noqa: E402

ASSETS = os.path.join(os.path.dirname(os.path.dirname(HERE)), "assets")
CKPT = os.path.join(ASSETS, "stories15M.bin")
POSITIONS = [0, 1, 2, 50, 98, 150, 220, 221]


def main():
    with open(CKPT, "rb") as f, open(os.path.join(HERE, "stories15M_header.bin"), "wb") as out:
        out.write(f.read(28))
    with open(os.path.join(ASSETS, "tokenizer.bin"), "rb") as f:
        packed = lzma.compress(f.read(), preset=9 | lzma.PRESET_EXTREME)
    with open(os.path.join(HERE, "tokenizer.bin.xz"), "wb") as out:
        out.write(packed)
    streams = {}
    for kind in ("strict", "fast"):
        cfg, shared, data = O.read_checkpoint(CKPT, kind)
        for W in (4, 8, 16):
            m = O.OracleModel(cfg, data, shared, W=W, kind=kind)
            calls, out, _ = m.generate(1, 256)
            streams[(kind, W)] = (calls, out[:calls].tolist())
            m.close()
    ref = streams[("strict", 8)]
    assert all(v == ref for v in streams.values()), "variants disagree"
    calls, nexts = ref
    assert nexts[-1] == 1, "expected BOS to end the stream"
    toks = np.array(nexts[:-1], dtype="<u4")
    sha = hashlib.sha256(toks.tobytes()).hexdigest()
    with open(os.path.join(HERE, "stories15M_t0_tokens.json"), "w") as f:
        json.dump({"checkpoint": "stories15M.bin", "checkpoint_bytes": os.path.getsize(CKPT),
                   "prompt": None, "temperature": 0, "first_token": 1, "forward_calls": calls,
                   "tokens": toks.tolist(), "terminator": 1, "sha256_le_u32": sha,
                   "produced_by": "oracle strict W=8 (== W 4/16, == optimized float mode)"}, f, indent=1)
    print("tokens", len(toks), sha)

    cfg, shared, data = O.read_checkpoint(CKPT, "strict")
    m = O.OracleModel(cfg, data, shared, W=8, kind="strict")
    token, keep = 1, {}
    for pos in range(calls):
        lg = m.forward(token, pos)
        if pos in POSITIONS:
            top = np.argsort(-lg, kind="stable")[:32].astype(np.int32)
            keep[f"p{pos}_strided"] = lg[::16].copy()
            keep[f"p{pos}_top_idx"] = top
            keep[f"p{pos}_top_val"] = lg[top].copy()
        token = nexts[pos]
    np.savez_compressed(os.path.join(HERE, "stories15M_logits.npz"), positions=np.array(POSITIONS), **keep)
    print("logits fixture written")


if __name__ == "__main__":
    main()
