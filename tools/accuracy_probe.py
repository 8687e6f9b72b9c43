"""Achieved HBM bandwidth of the accuracy kernel (csrc/metrics.cu), with the GPU's name and power limit.

    python tools/accuracy_probe.py                          # logits larger than the 126 MB L2, CUDA events
    python tools/accuracy_probe.py --compare path/to/other/libvqa_b200.so

``--compare`` times ``vqa_accuracy_update`` of another build of the library (same ABI) against this tree's, the two
alternating launch block by launch block on the same inputs, so that a change to the kernel is measured under the same
clocks and neighbours.  Both must count the same on these finite logits.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vqa_b200.runtime import check, lib  # noqa: E402

SHAPES = ((65536, 1000), (32768, 3129), (256, 1000))
ROUNDS, LAUNCHES, WARMUP = 10, 20, 5


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(", ")
    return {"name": name or torch.cuda.get_device_name(), "power_limit": power or "unknown"}


def load(path):
    L = C.CDLL(path)
    L.vqa_accuracy_update.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.vqa_last_error.restype = C.c_char_p
    return L


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--compare", help="another libvqa_b200.so whose accuracy kernel is timed alternately with this one")
    args = ap.parse_args()
    libs = {"this": lib()}
    if args.compare:
        libs["compare"] = load(os.path.abspath(args.compare))
    stream = torch.cuda.current_stream()
    out = {}
    for B, N in SHAPES:
        logits = torch.randn(B, N, device="cuda")
        targets = torch.randint(0, N, (B,), device="cuda")
        counters = {k: torch.zeros(3, dtype=torch.int64, device="cuda") for k in libs}

        def launch(name):
            check(libs[name].vqa_accuracy_update(logits.data_ptr(), N, N, None, targets.data_ptr(), B, 5,
                                                 counters[name].data_ptr(), None, None, stream.cuda_stream), libs[name])

        for name in libs:
            for _ in range(WARMUP):
                launch(name)
        torch.cuda.synchronize()
        ms = {name: 0.0 for name in libs}
        for _ in range(ROUNDS):
            for name in libs:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(LAUNCHES):
                    launch(name)
                b.record()
                torch.cuda.synchronize()
                ms[name] += a.elapsed_time(b)
        nbytes = B * N * 4 + B * 8
        want = int((logits.argmax(-1) == targets).sum()) * (WARMUP + ROUNDS * LAUNCHES)
        res = {}
        for name in libs:
            assert counters[name].tolist()[0] == want and counters[name].tolist()[2] == B * (WARMUP + ROUNDS * LAUNCHES)
            us = ms[name] / (ROUNDS * LAUNCHES) * 1e3
            res[name] = {"us_per_launch": round(us, 3), "achieved_gbps": round(nbytes / us / 1e3, 1)}
        out[f"{B}x{N}"] = {"algorithmic_bytes": nbytes, **res}
    print(json.dumps({"kernel": "accuracy_kernel", "bound": "hbm", "gpu": gpu_identity(), "shapes": out}))


if __name__ == "__main__":
    main()
