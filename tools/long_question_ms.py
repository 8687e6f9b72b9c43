"""Cost of long questions (max_question_length 20 ... 512) on the GPU, and where the two attention kernels meet.

    python tools/long_question_ms.py [--out FILE.json] [--reps N]

For L in {20, 64, 65, 128, 256, 512} (VQAModel(max_question_length=L), every question L tokens long):
  - question side against cached images: ms per 256 questions, one CUDA-graph replay of ``answer`` (as
    tools/question_side_ms.py), top_k = 5;
  - whole forward: pairs/s of ``predict`` at B = 256 (fp32 NCHW images, top_k = 5);
  - batch-1 ``predict`` latency (host clock around the call and a device synchronise);
  - plan workspace per pair.
Then the attention op alone at 256 pairs: attn_mma_kernel (self_attn) at L = 64 against attn_chunked_kernel at L = 64 and
L = 65, timed alternately in rounds with CUDA events.  Every shape is warmed up before it is timed.  The GPU's name and
power limit are printed beside the numbers and stored in the JSON.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vqa_b200 import program as P  # noqa: E402
from vqa_b200.model import VQAModel  # noqa: E402
from vqa_b200.runtime import Plan  # noqa: E402
from vqa_b200.synth import synth_batch  # noqa: E402

LENGTHS = (20, 64, 65, 128, 256, 512)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def events_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def inputs(B, L, seed):
    _, img, ids, mask = synth_batch(B, seed, max_len=L, full_length=True)
    return img.cuda(), ids.cuda(), mask.cuda()


def per_length(L, reps):
    torch.manual_seed(0)
    model = VQAModel(max_question_length=L).eval().cuda()
    eng = model.engine()
    out = {"L": L}
    with torch.no_grad():
        img, ids, mask = inputs(256, L, 1234)
        # question side against cached images, graph replay
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
        # whole forward at B = 256
        for _ in range(3):
            model.predict(img, ids, mask, top_k=5)
        torch.cuda.synchronize()
        ms = events_ms(lambda: model.predict(img, ids, mask, top_k=5), reps)
        out["forward_ms_b256"] = ms
        out["forward_pairs_per_s_b256"] = 256 / ms * 1e3
        prog = eng.last_plan[0] if eng.last_plan is not None else None
        if prog is not None:
            out["workspace_mb_per_pair"] = prog.ws.size / prog.B / 2 ** 20
            out["attention_kernels"] = sorted({op.kind for op in prog.ops if "attn" in op.kind})
        # batch-1 predict latency
        i1, d1, m1 = img[:1].contiguous(), ids[:1].contiguous(), mask[:1].contiguous()
        for _ in range(5):
            model.predict(i1, d1, m1, top_k=5)
        torch.cuda.synchronize()
        t = []
        for _ in range(reps):
            t0 = time.perf_counter()
            model.predict(i1, d1, m1, top_k=5)
            torch.cuda.synchronize()
            t.append((time.perf_counter() - t0) * 1e3)
        t.sort()
        out["predict_b1_ms_median"] = t[len(t) // 2]
    del eng, model
    torch.cuda.empty_cache()
    return out


def attention_alone(rounds, n):
    """The self-attention op of 256 pairs: attn_mma_kernel at L = 64, attn_chunked_kernel at L = 64 and 65."""
    B, H, D = 256, 8, 256
    plans = {}
    for name, kind, L in (("self_attn L64", "self_attn", 64), ("attn_chunked L64", "attn_chunked", 64),
                          ("attn_chunked L65", "attn_chunked", 65)):
        W = P.Weights("cuda")
        W.add("dummy", torch.zeros(8), torch.float32)
        W.finalize()
        ol = P.OpList(W, "cuda")
        qkv = ol._buf("qkv", torch.float32, B * L, 3 * D)
        m = ol._buf("mask", torch.int32, B, L)
        out = ol._buf("out", torch.float32, B * L, D)
        if kind == "self_attn":
            ol._op(kind, "attn", dict(B=B, L=L, H=H, hd=32, ld_qkv=3 * D, no_round=0), dict(qkv=qkv, mask=m, out=out))
        else:
            ol._op(kind, "attn", dict(B=B, L=L, H=H, hd=32, T=L, ld_q=3 * D, ld_kv=3 * D, k_off=D, v_off=2 * D, no_round=0,
                                      q_per_kv=1), dict(q=qkv, kv=qkv, mask=m, out=out, weights=None))
        ol.commit()
        ol.named["qkv"][0].view(torch.float32).normal_()
        ol.named["mask"][0].view(torch.int32).fill_(1)
        plans[name] = (ol, Plan(ol.ops, 0))
    stream = torch.cuda.current_stream().cuda_stream
    run = {k: (lambda p=p: p.run([0] * 6, stream)) for k, (_, p) in plans.items()}
    for f in run.values():
        for _ in range(20):
            f()
    torch.cuda.synchronize()
    times = {k: [] for k in run}
    for _ in range(rounds):
        for k, f in run.items():
            times[k].append(events_ms(f, n) * 1e3)
    return {k: {"us_median": sorted(v)[len(v) // 2], "us_all": [round(x, 2) for x in v]} for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    gpu = gpu_info()
    print(f"GPU: {gpu}", flush=True)
    res = {"gpu": gpu, "lengths": []}
    for L in LENGTHS:
        r = per_length(L, args.reps)
        res["lengths"].append(r)
        print(f"[{gpu}] L={L:3d}: question side {r['question_side_ms_per_256']:.3f} ms / 256 questions, forward "
              f"{r['forward_pairs_per_s_b256']:.0f} pairs/s at B=256 ({r['forward_ms_b256']:.2f} ms), batch-1 predict "
              f"{r['predict_b1_ms_median']:.2f} ms, workspace {r.get('workspace_mb_per_pair', 0):.2f} MB/pair, "
              f"{r.get('attention_kernels')}", flush=True)
    res["attention_op_b256"] = attention_alone(rounds=7, n=50)
    for k, v in res["attention_op_b256"].items():
        print(f"[{gpu}] {k}: {v['us_median']:.2f} us per launch (median of 7 alternating rounds of 50)", flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
