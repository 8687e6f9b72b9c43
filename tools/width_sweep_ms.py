"""Cost of the transformer widths the engine runs (embed_dim, heads, ffn_hidden_dim), on the GPU.

    python tools/width_sweep_ms.py [--out FILE.json] [--reps N]

For the reference defaults (256 / 8 / 1024) and each width of tests/model_widths_support.py (a: 256 / 4 / 1024,
b: 256 / 16 / 512, c: 512 / 8 / 2048, d: 128 / 4 / 256, e: 192 / 6 / 768), at max_question_length 20 (every question 20
tokens long), bf16:
  - question side against cached images: ms per 256 questions, one CUDA-graph replay of ``answer`` (as
    tools/long_question_ms.py), top_k = 5;
  - whole forward: pairs/s of ``predict`` at B = 256 (fp32 NCHW images, top_k = 5).
Every shape is warmed up before it is timed.  The GPU's name and power limit are printed beside the numbers and stored
in the JSON.
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from long_question_ms import events_ms, gpu_info, inputs  # noqa: E402
from model_widths_support import CONFIGS  # noqa: E402
from vqa_b200.model import VQAModel  # noqa: E402

WIDTHS = {"default": (256, 8, 1024), **CONFIGS}


def per_width(name, reps, L=20):
    D, H, F = WIDTHS[name]
    torch.manual_seed(0)
    model = VQAModel(embed_dim=D, num_attention_heads=H, ffn_hidden_dim=F, max_question_length=L).eval().cuda()
    eng = model.engine()
    out = {"config": name, "embed_dim": D, "heads": H, "head_dim": D // H, "ffn_hidden_dim": F, "L": L}
    with torch.no_grad():
        img, ids, mask = inputs(256, L, 1234)
        cache = eng.encode_images(img)
        for _ in range(2):
            eng.answer(cache, ids, mask, top_k=5)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            eng.answer(cache, ids, mask, top_k=5)
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        out["question_side_ms_per_256"] = events_ms(g.replay, reps)
        del g
        for _ in range(3):
            model.predict(img, ids, mask, top_k=5)
        torch.cuda.synchronize()
        ms = events_ms(lambda: model.predict(img, ids, mask, top_k=5), reps)
        out["forward_ms_b256"] = ms
        out["forward_pairs_per_s_b256"] = 256 / ms * 1e3
        prog = eng.last_plan[0] if eng.last_plan is not None else None
        if prog is not None:
            out["chain"] = any(op.kind == "mlp_chain" for op in prog.ops)
    del eng, model
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    gpu = gpu_info()
    print(f"GPU: {gpu}", flush=True)
    res = {"gpu": gpu, "widths": []}
    for name in WIDTHS:
        r = per_width(name, args.reps)
        res["widths"].append(r)
        print(f"[{gpu}] {name:7s} D={r['embed_dim']:3d} H={r['heads']:2d} hd={r['head_dim']:2d} F={r['ffn_hidden_dim']:4d}: "
              f"question side {r['question_side_ms_per_256']:.3f} ms / 256 questions, forward "
              f"{r['forward_pairs_per_s_b256']:.0f} pairs/s at B=256 ({r['forward_ms_b256']:.2f} ms), "
              f"chain={r.get('chain')}", flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
