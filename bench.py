#!/usr/bin/env python
"""Headline benchmark: VQA pairs/sec of the fused eval-mode VQAModel.forward on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch 256] [--impl reference] [--dump-outputs DIR]

One process per GPU (torchrun sets RANK/LOCAL_RANK/WORLD_SIZE).  Workload = BASELINE.json
configs[1]: batch 256 per GPU, 224x224 images, 20-token questions, 1000 answers, bf16 engine,
seeded random-init weights, synthetic inputs.  The batch is sharded across ranks with no
data-path collective (weak scaling); rank 0 broadcasts the packed weight arena once at load.

Prints ONE JSON line (rank 0).  ``value`` times K forwards with inputs resident in HBM (fp32 NCHW,
154 MB per batch > 126 MB L2, so no L2 flush is needed); ``e2e`` times the same through the predict
path from pinned HOST buffers (uint8 HWC images + ids + mask H2D, top-5 D2H inside the timed
region).  ``--impl reference`` times the reference's own CPU implementation on the host cores for the
same metric: the UNMODIFIED reference when it is staged (oracle/_ref/reference.zip, written by
tools/stage_reference.sh in the build container; ``kind: "reference"``), else the oracle port
(``kind: "port"``).

``--dump-outputs DIR`` writes the logits of the last timed step of ``value`` as DIR/logits.npy; inputs and weights
are seeded, so two builds of the project can be compared output for output.  With several GPUs the file holds rank
0's shard of the batch.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

CONV_FLOP_PER_PAIR = 3.6273e9   # SURVEY 8(d): stem + stages 1-4 incl. shortcuts
STEM_FLOP_PER_PAIR = 2 * 147 * 64 * 112 * 112   # conv 7x7/2, 3 -> 64 channels, 112 x 112 outputs
FLOP_PER_PAIR = 3.849e9          # SURVEY.md section 8d: FlopCounterMode on the reference, L=20 (2*MAC)
METRIC = "vqa_pairs_per_sec"
WORKLOAD = "VQAModel.forward eval, 224x224 images, 20-token questions, 1000 answers (BASELINE configs[1])"


def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


DUMP_MAX_BYTES = 60 * 10**6     # below 64 MB with room for the .npy header


def dump_logits(out_dir: str, logits) -> None:
    """Write fp32 ``logits`` [B, N] as ``out_dir/logits.npy``.  A batch too large for DUMP_MAX_BYTES keeps a fixed,
    seeded sample of its rows (sorted), the same rows on every run with the same arguments."""
    import numpy as np
    a = logits.float().cpu().numpy()
    cap = DUMP_MAX_BYTES // a[0].nbytes
    if a.shape[0] > cap:
        a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], cap, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logits.npy"), a)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled by ONE long-running ``nvidia-smi -lms`` process.

    The process is started before the warm-up (nothing is forked inside the timed region); ``mark()``
    brackets the timed region and ``summary()`` reports the samples that fall inside it (or, for a
    region shorter than the sampling period, the samples nearest to it, flagged ``"nearest"``).
    """
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    PERIOD_MS = 20

    def __init__(self, index: int):
        self.index = index
        self.rows = []          # (host time, fields)
        self.t0 = self.t1 = None
        self._p = None
        self._t = None

    def _loop(self):
        try:
            for line in self._p.stdout:
                parts = [x.strip() for x in line.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append((time.time(), parts))
        except Exception:
            pass

    def start(self):
        try:
            self._p = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                        "--format=csv,noheader,nounits", "-lms", str(self.PERIOD_MS)],
                                       stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()
        except Exception:
            self._p = None
        return self

    def __enter__(self):        # the timed region
        self.t0 = time.time()
        return self

    def __exit__(self, *a):
        self.t1 = time.time()

    def stop(self):
        if self._p is not None:
            time.sleep(2.5 * self.PERIOD_MS / 1e3)     # let the sample that covers the end of the region arrive
            self._p.terminate()
            try:
                self._p.wait(timeout=5)
            except Exception:
                self._p.kill()
            self._t.join(timeout=5)

    def summary(self):
        if not self.rows or self.t0 is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        inside = [r for t, r in self.rows if self.t0 <= t <= self.t1 + self.PERIOD_MS / 1e3]
        how = "during"
        if not inside:          # region shorter than the sampling period: the two samples around it
            mid = 0.5 * (self.t0 + self.t1)
            inside = [r for _, r in sorted(self.rows, key=lambda tr: abs(tr[0] - mid))[:2]]
            how = "nearest"
        num = lambda x: x.replace(".", "").isdigit()
        sm = [float(r[0]) for r in inside if num(r[0])]
        mx = [float(r[1]) for r in inside if num(r[1])]
        pw = [float(r[2]) for r in inside if num(r[2])]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in inside)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w": statistics.median(pw) if pw else None, "reasons": reasons, "samples": len(inside),
                "sampled": how, "period_ms": self.PERIOD_MS}


# ----------------------------------------------------------------------------- reference arm
def cpu_reference_run(steps: int, warmup: int, batch: int = 32):
    """The reference's eval-mode forward on the host cores: pairs/s.  The UNMODIFIED reference
    (models/vqa_model.py:243-311) when it is present / staged, else the oracle port of the same algorithm."""
    import torch
    from oracle import vqa_oracle as O
    from oracle.ref_loader import load_reference
    from vqa_b200.model import VQAModel
    from vqa_b200.synth import synth_batch
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    _, img, ids, mask = synth_batch(batch, 1234, full_length=True)
    ref_mod, where = load_reference()
    torch.manual_seed(0)
    if ref_mod is not None:
        ref = ref_mod.VQAModel().eval()          # same seed + construction order = the same weights as vqa_b200.VQAModel()
        kind = "reference"

        def fwd():
            with torch.no_grad():
                return ref(img, ids, mask)[0]
    else:
        sd = VQAModel().eval().state_dict()
        kind = "port"

        def fwd():
            return O.vqa_forward(sd, img, ids, mask)[0]
    for _ in range(warmup):
        fwd()
    times = []
    logits = None
    for _ in range(steps):
        t0 = time.perf_counter()
        logits = fwd()
        times.append(time.perf_counter() - t0)
    total = sum(times)
    return {"value": batch * steps / total, "ms_per_step": 1e3 * total / steps, "cores": torch.get_num_threads(),
            "best": batch / min(times), "batch": batch, "inputs": (img, ids, mask), "logits": logits, "kind": kind,
            "source": where}


def library_bar(batch: int, dev):
    """Informational (SURVEY 2.1 / 8d): the UNMODIFIED reference on the same B200 through PyTorch's own kernels
    (cuDNN / cuBLAS), eager fp32 with the library defaults and eager autocast(bf16) + channels_last -- the kernel
    set a user of the reference gets on this GPU today.  None when the reference is not staged."""
    import torch
    from oracle.ref_loader import load_reference
    from vqa_b200.synth import synth_batch
    ref_mod, where = load_reference()
    if ref_mod is None:
        return {"unavailable": where}
    torch.manual_seed(0)
    ref = ref_mod.VQAModel().eval().to(dev)
    _, img, ids, mask = synth_batch(batch, 1234, full_length=True)
    img, ids, mask = img.to(dev), ids.to(dev), mask.to(dev)
    out = {"source": where, "batch": batch, "allow_tf32_cudnn": bool(torch.backends.cudnn.allow_tf32),
           "allow_tf32_matmul": bool(torch.backends.cuda.matmul.allow_tf32)}

    def timed(fn, n=5):
        with torch.no_grad():
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    ms = timed(lambda: ref(img, ids, mask))
    out["eager_fp32"] = {"ms_per_step": ms, "pairs_per_sec": batch / (ms * 1e-3)}
    ref_cl = ref.to(memory_format=torch.channels_last)
    img_cl = img.contiguous(memory_format=torch.channels_last)

    def amp():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return ref_cl(img_cl, ids, mask)
    ms = timed(amp)
    out["eager_autocast_bf16_channels_last"] = {"ms_per_step": ms, "pairs_per_sec": batch / (ms * 1e-3)}
    del ref, ref_cl
    torch.cuda.empty_cache()
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, max(args.warmup, 1)
    r = cpu_reference_run(steps, min(warmup, 2))
    sample = (f"{steps} timed fp32 forwards of batch {r['batch']} (BASELINE configs[0]) on the host CPU, "
              + ("the unmodified reference VQAModel" if r["kind"] == "reference" else "oracle port of the reference forward"))
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "pairs/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": min(warmup, 2), "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_step": r["batch"], "device": "host CPU"},
            "cpu_baseline": {"value": r["value"], "unit": "pairs/s", "cores": r["cores"], "kind": r["kind"],
                             "sample": sample},
            "e2e": {"value": r["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    from vqa_b200 import program as P
    from vqa_b200.engine import Engine
    from vqa_b200.model import VQAModel
    from vqa_b200.runtime import launch_count
    from vqa_b200.synth import synth_batch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    B, L, K, Wm = args.batch, 20, args.steps, args.warmup
    torch.manual_seed(0)
    model = VQAModel().eval().to(dev)
    # weights: rank 0 packs, everyone receives the arena over NCCL/NVLink (one collective, at load only)
    weights = P.build_weights(model.state_dict(), model.config, dev)
    if world > 1:
        if rank != 0:
            weights.arena.tensor.zero_()
        dist.broadcast(weights.arena.tensor, src=0)
    engine = Engine(model, weights)
    model._engine = engine

    u8, img, ids, mask = synth_batch(B, 1234 + rank, full_length=True)
    d_img, d_ids, d_mask = img.to(dev), ids.to(dev), mask.to(dev)
    h_u8, h_ids, h_mask = u8.pin_memory(), ids.pin_memory(), mask.pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput.  One forward (every kernel of the plan, both lanes) is captured into a CUDA graph
    # per compute lane; a lane = its own stream + its own plan workspace (Engine.run(slot=lane)).  Step k is replayed on
    # lane k % LANES, so consecutive steps overlap on the GPU: the launch-latency-bound text / fusion / head kernels of
    # one step and the partially filled last wave of each persistent convolution leave SMs idle that the next step's
    # kernels fill.  Every step is a complete forward of its own batch; inputs resident in HBM.  The single-stream
    # figure (steps strictly one after another) is measured first and reported beside it.
    LANES = max(1, int(os.environ.get("VQA_BENCH_LANES", "3")))
    clocks = ClockSampler(local).start()
    eng = model.engine()
    with torch.no_grad():
        for _ in range(2):
            model(d_img, d_ids, d_mask)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        n0 = launch_count()
        with torch.cuda.graph(graph):
            logits, _ = model(d_img, d_ids, d_mask)
        launches_per_step = launch_count() - n0
        for _ in range(max(Wm, 3)):
            graph.replay()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            graph.replay()
        e1.record()
        barrier()
        ms_single = reduce_max(e0.elapsed_time(e1))
        # lanes: lane 0 reuses the graph above (plan slot 0)
        lane_streams = [torch.cuda.Stream(dev) for _ in range(LANES)]
        lane_graphs, lane_out = [graph], [logits]
        for l in range(1, LANES):
            with torch.cuda.stream(lane_streams[l]):
                for _ in range(2):
                    eng.run(d_img, d_ids, d_mask, slot=l)
            torch.cuda.synchronize()
            g_l = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_l, stream=lane_streams[l]):
                out_l = eng.run(d_img, d_ids, d_mask, slot=l)[0]
            lane_graphs.append(g_l)
            lane_out.append(out_l)
        cur = torch.cuda.current_stream()

        def lanes_run(n):
            fork = torch.cuda.Event()
            fork.record(cur)
            for st in lane_streams:
                st.wait_event(fork)
            for k in range(n):
                with torch.cuda.stream(lane_streams[k % LANES]):
                    lane_graphs[k % LANES].replay()
            for st in lane_streams:
                j = torch.cuda.Event()
                j.record(st)
                cur.wait_event(j)

        lanes_run(max(Wm, 3) * LANES)
        barrier()
        assert all(torch.equal(o, lane_out[0]) for o in lane_out[1:]), "lanes disagree"
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with clocks:
            e0.record(cur)
            lanes_run(K)
            e1.record(cur)
            barrier()
        launches = launches_per_step * K
        ms = reduce_max(e0.elapsed_time(e1))
        if args.dump_outputs and rank == 0:     # step K-1 ran on lane (K-1) % LANES, into that lane's own buffer
            dump_logits(args.dump_outputs, lane_out[(K - 1) % LANES])
    clocks.stop()
    if args.quick:    # A/B experiments: device-resident throughput only (not a bench line)
        if rank == 0:
            print(json.dumps({"quick": True, "lanes": LANES, "value": world * B * K / (ms * 1e-3), "ms_per_step": ms / K,
                              "single_stream": world * B * K / (ms_single * 1e-3), "single_ms_per_step": ms_single / K,
                              "launches_per_step": launches_per_step}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    value = world * B * K / (ms * 1e-3)
    value_single = world * B * K / (ms_single * 1e-3)
    # ---- sustained leg (N = 1): the same lanes replayed back to back for >= 3 s with their own clock samples, so the
    # question "burst or sustained peak as the denominator" is answered by data (the headline's K steps last ~30 ms)
    sustained = None
    if world == 1 and rank == 0:
        with torch.no_grad():
            n_sus = max(K, int(3.2 / (ms / K * 1e-3)))
            n_sus = (n_sus + LANES - 1) // LANES * LANES
            clocks_s = ClockSampler(local).start()
            time.sleep(0.1)
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with clocks_s:
                s0.record(cur)
                lanes_run(n_sus)
                s1.record(cur)
                torch.cuda.synchronize()
            clocks_s.stop()
            ms_sus = s0.elapsed_time(s1)
        sustained = {"seconds": ms_sus * 1e-3, "steps": n_sus, "value": B * n_sus / (ms_sus * 1e-3),
                     "ms_per_step": ms_sus / n_sus, "clocks": clocks_s.summary(),
                     "frac_of_sustained_peak": FLOP_PER_PAIR * B * n_sus / (ms_sus * 1e-3) / 1e12 / measured_peaks()["bf16_tflops_sustained"],
                     "frac_of_burst_peak": FLOP_PER_PAIR * B * n_sus / (ms_sus * 1e-3) / 1e12 / measured_peaks()["bf16_tflops"]}
    del lane_graphs[1:], lane_out[1:]

    # ---- BASELINE configs[2]: 8192 uint8 images + questions per step over 8 GPUs = 1024 per GPU per step, the GPU
    # preprocessing (uint8 HWC -> normalised, phase-packed bf16) inside the step; device-resident inputs, graph replay
    B3 = 1024
    u8_3, _, ids_3, mask_3 = synth_batch(B3, 4321 + rank, full_length=True)
    u8_3, ids_3, mask_3 = u8_3.to(dev), ids_3.to(dev), mask_3.to(dev)
    with torch.no_grad():
        k3 = max(3 * LANES, K // 4)
        g3s = []
        for l in range(LANES):
            with torch.cuda.stream(lane_streams[l]):
                for _ in range(2):
                    eng.run(u8_3, ids_3, mask_3, slot=l)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=lane_streams[l]):
                eng.run(u8_3, ids_3, mask_3, slot=l)
            g3s.append(g)

        def lanes3(n, nl):
            fork = torch.cuda.Event()
            fork.record(cur)
            for st in lane_streams[:nl]:
                st.wait_event(fork)
            for k in range(n):
                with torch.cuda.stream(lane_streams[k % nl]):
                    g3s[k % nl].replay()
            for st in lane_streams[:nl]:
                j = torch.cuda.Event()
                j.record(st)
                cur.wait_event(j)

        ms3_by = {}
        for nl in sorted({1, LANES}):
            lanes3(nl, nl)
            barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(cur)
            lanes3(k3, nl)
            c1.record(cur)
            barrier()
            ms3_by[nl] = reduce_max(c0.elapsed_time(c1))
        best3 = min(ms3_by, key=ms3_by.get)     # at 1024 pairs per step the small kernels are no longer latency-bound:
        ms3 = ms3_by[best3]                       # one stream is usually as fast as several lanes here
    config3 = {"workload": "BASELINE configs[2]: uint8 HWC images + questions, 1024 pairs per GPU per step, GPU preprocessing included",
               "global_batch": world * B3, "steps": k3, "ms_per_step": ms3 / k3, "compute_lanes": best3,
               "pairs_per_sec": world * B3 * k3 / (ms3 * 1e-3),
               "pairs_per_sec_by_lanes": {str(nl): world * B3 * k3 / (t * 1e-3) for nl, t in ms3_by.items()},
               "frac_of_peak": FLOP_PER_PAIR * B3 * k3 / (ms3 * 1e-3) / 1e12 / measured_peaks()["bf16_tflops_sustained"]}
    g3 = g3s
    del g3, g3s, u8_3, ids_3, mask_3
    for key in [k_ for k_ in eng._plans if k_[0] == B3 and k_[-1] > 0]:     # drop the extra lanes' 1024-pair workspaces
        del eng._plans[key]
    torch.cuda.empty_cache()

    # ---- SURVEY 8f row f2: the image side cached (encode_images once), only the question side per step
    cached_leg = None
    if world == 1:
        with torch.no_grad():
            eng = model.engine()
            cache = eng.encode_images(d_img)
            for _ in range(2):
                eng.answer(cache, d_ids, d_mask, top_k=5)
            torch.cuda.synchronize()
            gq = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gq):
                q_out = eng.answer(cache, d_ids, d_mask, top_k=5)
            for _ in range(3):
                gq.replay()
            torch.cuda.synchronize()
            same = bool(torch.equal(q_out[0], model(d_img, d_ids, d_mask)[0]))
            kq = max(5, K)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(kq):
                gq.replay()
            c1.record()
            torch.cuda.synchronize()
            msq = c0.elapsed_time(c1) / kq
        cached_leg = {"workload": "question side only against cached images (VQAModel.encode_images once, then answer): "
                                  "text encoder + cross-attention + gate + head + top-5, 256 questions per step",
                      "ms_per_step": msq, "questions_per_sec": B / (msq * 1e-3), "cache_bytes_per_image": cache.nbytes // B,
                      "logits_bit_identical_to_forward": same}
        del gq, cache, q_out
        torch.cuda.empty_cache()

    # ---- BASELINE configs[4]: one image, 16 questions of 64 tokens (VQAModel(max_question_length=64)); the backbone,
    # projector and K/V projections run once per image.  Three forms, each one CUDA-graph replay: the image repeated 16
    # times (what the reference does), the in-call form (1 image + 16 questions), and the question side alone against the
    # cached image
    config5 = None
    if world == 1:
        with torch.no_grad():
            torch.manual_seed(0)
            m64 = VQAModel(max_question_length=64).eval().to(dev)
            _, img5, ids5, mask5 = synth_batch(16, 77, max_len=64)
            img5, ids5, mask5 = img5.to(dev), ids5.to(dev), mask5.to(dev)
            one5, rep5 = img5[:1].contiguous(), img5[:1].repeat(16, 1, 1, 1).contiguous()
            e5 = m64.engine()
            cache5 = e5.encode_images(one5)

            def timed_graph(fn, reps=50):
                for _ in range(2):
                    fn()
                torch.cuda.synchronize()
                g5 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g5):
                    out5 = fn()
                for _ in range(3):
                    g5.replay()
                t0_, t1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0_.record()
                for _ in range(reps):
                    g5.replay()
                t1_.record()
                torch.cuda.synchronize()
                return t0_.elapsed_time(t1_) / reps, out5

            ms_rep, o_rep = timed_graph(lambda: m64(rep5, ids5, mask5)[0])
            ms_one, o_one = timed_graph(lambda: m64(one5, ids5, mask5)[0])
            ms_q, o_q = timed_graph(lambda: e5.answer(cache5, ids5, mask5)[0])
            config5 = {"workload": "BASELINE configs[4]: one image, 16 questions of 64 tokens, backbone once per image",
                       "ms_image_repeated_16x": ms_rep, "ms_one_image_in_call": ms_one, "ms_question_side_cached_image": ms_q,
                       "bit_identical": bool(torch.equal(o_rep, o_one) and torch.equal(o_one, o_q))}
            del m64, e5, cache5, o_rep, o_one, o_q
            torch.cuda.empty_cache()

    # ---- end to end from host buffers through the predict API's batch path (uint8 HWC -> top-5):
    # pinned host buffers -> H2D -> GPU normalise + forward + softmax/top-k -> D2H, all inside the timed region
    from vqa_b200.inference import VQAInference
    inf = VQAInference(device=str(dev))
    inf.model, inf._is_loaded = model, True      # same weights as the device-resident leg
    # raw pinned H2D bandwidth of this box (explains the e2e number: 38.6 MB of uint8 pixels per 256-pair step)
    d_probe = torch.empty_like(h_u8, device=dev)
    d_probe.copy_(h_u8, non_blocking=True)
    torch.cuda.synchronize()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(5):
        d_probe.copy_(h_u8, non_blocking=True)
    c1.record()
    torch.cuda.synchronize()
    h2d_gbps = 5 * h_u8.numel() / (c0.elapsed_time(c1) * 1e-3) / 1e9
    # the same copies with every rank copying AT THE SAME TIME: the box's aggregate pinned H2D ceiling (host DRAM / PCIe
    # root complexes shared by the GPUs), which bounds the end-to-end number at N > 1
    barrier()
    c0.record()
    for _ in range(10):
        d_probe.copy_(h_u8, non_blocking=True)
    c1.record()
    torch.cuda.synchronize()
    ms_conc = reduce_max(c0.elapsed_time(c1))
    barrier()
    h2d_conc_gbps = 10 * h_u8.numel() / (ms_conc * 1e-3) / 1e9          # per rank, slowest rank
    del d_probe
    def e2e_run(lanes, idle_s=0.0):
        inf.pipeline_lanes = lanes
        inf.pipeline_slots = int(os.environ.get("VQA_PIPE_SLOTS", "0"))
        with torch.no_grad():
            for _ in inf.predict_tensors_pipelined([(h_u8, h_ids, h_mask)] * (4 * lanes + 4), 5):   # captures every slot's graph
                pass
            barrier()
            if idle_s > 0:                            # informational leg: start from an idle GPU (see e2e.from_idle_value)
                time.sleep(idle_s)
                barrier()
            t0 = time.perf_counter()                  # host clock: copies and compute run on the API's own streams
            n_out = 0
            for top_idx, top_probs in inf.predict_tensors_pipelined([(h_u8, h_ids, h_mask)] * K, 5):
                n_out += top_idx.shape[0]
            torch.cuda.synchronize()
            ms_local = (time.perf_counter() - t0) * 1e3
            barrier()
            assert n_out == B * K
            return reduce_max(ms_local), top_idx.clone()

    ms_e2e_1, idx_1 = e2e_run(1)                      # A/B: one compute lane (forwards strictly one after another)
    ms_e2e_2, idx_2 = e2e_run(2)                     # A/B: two lanes
    assert torch.equal(idx_1, idx_2)
    ms_e2e, idx_3 = e2e_run(3)                       # the API's default: three lanes, like the device-resident leg
    assert torch.equal(idx_1, idx_3)
    ms_e2e_idle, _ = e2e_run(3, idle_s=0.5)           # the same K steps started from an idle GPU
    inf.pipeline_lanes = 3
    e2e_value = world * B * K / (ms_e2e * 1e-3)
    h2d = h_u8.numel() + h_ids.numel() * 8 + h_mask.numel() * 8
    d2h = B * 5 * (8 + 4)

    # ---- batch-1 latency through VQAInference.predict (BASELINE configs[3]): PIL image + question string in,
    # answer dict out; wall clock per call (includes PIL -> uint8, tokenisation, H2D, graph replay, D2H, decode)
    latency = None
    if rank == 0 and world == 1:
        from PIL import Image
        from vqa_b200.synth import synth_images_u8
        from vqa_b200.text import Tokenizer, AnswerVocabulary
        inf.tokenizer = Tokenizer(max_length=20)
        inf.tokenizer.build_vocab(["what is this", "what color", "how many", "is there", "where is", "what type"], min_freq=1)
        inf.answer_vocab = AnswerVocabulary(num_answers=1000)
        for i in range(1000):
            inf.answer_vocab.idx2answer[i] = f"answer_{i}"
        pil = Image.fromarray(synth_images_u8(1, 99)[0].numpy(), "RGB")
        for _ in range(20):
            inf.predict(pil, "What color is this?")
        lat = []
        for _ in range(300):
            t0 = time.perf_counter()
            inf.predict(pil, "What color is this?")
            lat.append((time.perf_counter() - t0) * 1e3)
        lat.sort()
        latency = {"p50_ms": lat[len(lat) // 2], "p99_ms": lat[int(len(lat) * 0.99) - 1], "calls": len(lat),
                   "path": "VQAInference.predict(PIL 224x224, str), CUDA-graph replay"}
        # the same call with the image LRU on (SURVEY 8f row f2): a repeated image costs its content hash + the question side
        inf.image_cache_size = 8
        for _ in range(20):
            inf.predict(pil, "What color is this?")
        lat = []
        for _ in range(300):
            t0 = time.perf_counter()
            inf.predict(pil, "What color is this?")
            lat.append((time.perf_counter() - t0) * 1e3)
        lat.sort()
        inf.image_cache_size = 0
        latency["cached_image"] = {"p50_ms": lat[len(lat) // 2], "p99_ms": lat[int(len(lat) * 0.99) - 1], "calls": len(lat),
                                   "path": "VQAInference(image_cache_size=8).predict on an image seen before: SHA-1 of the "
                                           "pixels, then the question side only (CUDA-graph replay)", **inf.cache_info()}

    # ---- per-kernel timing pass (CUDA events around every op of the plan) for the roofline line
    peaks = measured_peaks()
    roof = None
    per_kernel = {}
    if rank == 0:
        prog, plan = engine.plan_for(B, L, "nchw_f32", P.MASK_I64, False, 0)
        logits = torch.empty(B, model.config["num_answers"], device=dev)
        ext = [d_img.data_ptr(), d_ids.data_ptr(), d_mask.data_ptr(), logits.data_ptr(), 0, 0]
        stream = torch.cuda.current_stream().cuda_stream
        reps = 3
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(plan.n_ops + 1)] for _ in range(reps)]
        for r_ in range(reps):
            evs[r_][0].record()
            for k in range(plan.n_ops):
                plan.run(ext, stream, k, k + 1)
                evs[r_][k + 1].record()
        torch.cuda.synchronize()
        op_ms = [statistics.median(evs[r_][k].elapsed_time(evs[r_][k + 1]) for r_ in range(reps))
                 for k in range(plan.n_ops)]
        gemm_ms_ev = sum(t for k, t in enumerate(op_ms) if prog.ops[k].kind == "gemm")
        total_ms = sum(op_ms)
        # the dominant kernel's launches back to back (no events in between, so no per-op event overhead):
        # all 48 gemm_tap_kernel launches of one forward, and the 17 convolution launches alone
        def b2b(sel):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            best = None
            for _ in range(4):
                torch.cuda.synchronize()
                a.record()
                for k in sel:
                    plan.run(ext, stream, k, k + 1)
                b.record()
                torch.cuda.synchronize()
                t = a.elapsed_time(b)
                best = t if best is None else min(best, t)
            return best
        # every tensor-core kernel of the forward: gemm_tap_kernel (convolutions + Linears), stem_pool_kernel (fused stem)
        # and mlp_chain_kernel (fused W_o / FFN / next projection chains) -- together they execute all GEMM-shaped FLOPs
        TENSOR_KINDS = ("gemm", "stem_pool", "mlp_chain")
        gemm_ops = [k for k in range(plan.n_ops) if prog.ops[k].kind in TENSOR_KINDS]
        conv_ops = [k for k in gemm_ops if prog.ops[k].kind == "stem_pool" or
                    (prog.ops[k].kind == "gemm" and prog.ops[k].i["dtype"] == P.DT_BF16 and prog.ops[k].i["out_dtype"] == P.OUT_BF16)]
        n_by_kind = {kd: sum(1 for k in gemm_ops if prog.ops[k].kind == kd) for kd in TENSOR_KINDS}
        block_conv_ops = [k for k in conv_ops if prog.ops[k].kind == "gemm"]     # the dominant kernel's launches
        gemm_ms = b2b(gemm_ops)
        conv_ms = b2b(conv_ops)
        block_ms = b2b(block_conv_ops)
        traffic = traffic_note = None
        try:
            import glob
            src = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles",
                                                "*_ncu_*_summary.json")))[-1]      # newest capture (names sort by round / stage)
            with open(src) as f:
                nc = json.load(f)
            traffic = (nc["dram_read_mb"] + nc["dram_write_mb"]) * 1e6     # bytes per 256-pair forward
            traffic_note = {"launches": "sum over the 17 convolution launches of one 256-pair forward",
                            "algorithmic_bytes": 9.07e6 * B,
                            "source": "profiles/" + os.path.basename(src).replace(".json", ".md")
                                      + " (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum)"}
        except Exception:
            pass
        for k, t in enumerate(op_ms):
            nm = plan.kernel_name(k)
            per_kernel[nm] = per_kernel.get(nm, 0.0) + t
        # the dominant kernel: gemm_tap_kernel's ResBlock convolution launches (88 % of the forward's 3.849 GFLOP per pair;
        # the stem has its own kernel, the text / fusion / head path is ~6 %); algorithmic FLOPs per launch = BLOCK_CONV / 16
        block_flop = (CONV_FLOP_PER_PAIR - STEM_FLOP_PER_PAIR) * B
        achieved = block_flop / (block_ms * 1e-3) / 1e12
        peak = peaks["bf16_tflops_sustained"]
        roof = {"bound": "tensor",
                "kernel": f"gemm_tap_kernel: the {len(block_conv_ops)} ResBlock convolution launches of one forward",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
                "peak_source": peaks["source"] + " (sustained cuBLAS bf16)",
                "flop_per_launch": block_flop / max(1, len(block_conv_ops)), "us_per_launch": block_ms * 1e3 / max(1, len(block_conv_ops)),
                "launches_per_step": len(block_conv_ops),
                "timing": f"CUDA events around these {len(block_conv_ops)} launches issued back to back on one stream (best of 4); "
                          "achieved = 3.391 GFLOP per pair (stages 1-4 incl. shortcuts, SURVEY 8d) x batch / that time",
                "conv_only": {"ms_per_step": conv_ms, "launches": len(conv_ops),
                              "what": "fused stem (stem_pool_kernel) + the 16 ResBlock convolutions, 3.627 GFLOP per pair",
                              "achieved": CONV_FLOP_PER_PAIR * B / (conv_ms * 1e-3) / 1e12,
                              "frac": CONV_FLOP_PER_PAIR * B / (conv_ms * 1e-3) / 1e12 / peak},
                "all_tensor_kernels": {"ms_per_step": gemm_ms, "launches": len(gemm_ops),
                                       "what": f"{n_by_kind['gemm']} gemm_tap_kernel (convolutions + Linears), {n_by_kind['stem_pool']} "
                                               f"stem_pool_kernel, {n_by_kind['mlp_chain']} mlp_chain_kernel launches, 3.849 GFLOP per pair; the "
                                               "small Linears are bound by their launch latency when issued one by one",
                                       "achieved": FLOP_PER_PAIR * B / (gemm_ms * 1e-3) / 1e12,
                                       "frac": FLOP_PER_PAIR * B / (gemm_ms * 1e-3) / 1e12 / peak},
                "all_kernels_ms_per_step": total_ms, "gemm_share_of_step": gemm_ms_ev / total_ms,
                "share_of_step": sum(op_ms[k] for k in block_conv_ops) / total_ms,   # compare: profiles/*_ncu_full_summary.md (s1-s4 convolutions)
                "whole_forward_frac": (FLOP_PER_PAIR * B * K / (ms * 1e-3) / 1e12) / peak}
        if args.dump_ops:
            os.makedirs(os.path.dirname(args.dump_ops) or ".", exist_ok=True)
            with open(args.dump_ops, "w") as f:
                json.dump({"batch": B, "ops": [{"op": k, "name": prog.ops[k].name, "kernel": plan.kernel_name(k),
                                                "ms": op_ms[k]} for k in range(plan.n_ops)],
                           "per_kernel_ms": per_kernel}, f, indent=1)

    # ---- parity on EVERY rank (after the NCCL weight broadcast): 32 pairs of this rank's own seed against the fp32 oracle
    # on this rank's host cores, max over ranks in the line (a rank whose weights arrived damaged cannot hide)
    rank_parity = None
    if not args.no_cpu_baseline or world > 1:
        from oracle import vqa_oracle as _O
        torch.set_num_threads(max(1, (os.cpu_count() or 1) // max(1, world)))
        _, pi, pd, pm = synth_batch(32, 9000 + rank)
        sd_cpu = {k_: v_.detach().cpu() for k_, v_ in model.state_dict().items()}
        want_r, _ = _O.vqa_forward(sd_cpu, pi, pd, pm)
        with torch.no_grad():
            got_r = model(pi.to(dev), pd.to(dev), pm.to(dev))[0].float().cpu()
        err_r = float((got_r - want_r).abs().max() / want_r.abs().max())
        agree_r = float((got_r.argmax(1) == want_r.argmax(1)).float().mean())
        t = torch.tensor([err_r, -agree_r], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rank_parity = {"pairs_per_rank": 32, "ranks": world, "max_over_ranks": float(t[0].item()),
                       "min_top1_agree_over_ranks": -float(t[1].item()), "gate": 2e-2,
                       "oracle": "oracle/vqa_oracle.py (fp32, this rank's host cores), inputs seeded 9000 + rank"}

    # ---- host CPU baseline (rank 0, N=1 only): bounded sample of the same workload
    cpu = None
    parity = None
    lib_bar = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(steps=4, warmup=1)
        cpu = {"value": r["value"], "unit": "pairs/s", "cores": r["cores"], "kind": r["kind"],
               "sample": "4 timed fp32 forwards of batch 32 (BASELINE configs[0]) on the host CPU: "
                         + ("the unmodified reference VQAModel (oracle/_ref)" if r["kind"] == "reference"
                            else "the oracle port (reference not staged)")}
        try:
            lib_bar = library_bar(B, dev)
        except Exception as e:       # informational leg: never fail the bench line
            lib_bar = {"unavailable": f"{type(e).__name__}: {e}"}
        # parity on this box, same 32 pairs: both precision modes of the CUDA path against the oracle's fp32 logits
        # (the model of the timed legs has the same seed-0 weights as the oracle run)
        from vqa_b200.model import VQAModel as _VM
        i32, d32, m32 = (t.to(dev) for t in r["inputs"])
        want = r["logits"]
        with torch.no_grad():
            got_bf16 = model(i32, d32, m32)[0].float().cpu()
            torch.manual_seed(0)
            m_tf32 = _VM(precision="tf32").eval().to(dev)
            got_tf32 = m_tf32(i32, d32, m32)[0].float().cpu()
            # throughput of the tolerance mode, same batch-256 workload, CUDA-graph replay
            for _ in range(2):
                m_tf32(d_img, d_ids, d_mask)
            torch.cuda.synchronize()
            g2 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g2):
                m_tf32(d_img, d_ids, d_mask)
            for _ in range(3):
                g2.replay()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(5):
                g2.replay()
            b.record()
            torch.cuda.synchronize()
        rel = lambda x: float((x - want).abs().max() / want.abs().max())
        parity = {"pairs": int(want.shape[0]),
                  "oracle": ("the unmodified reference VQAModel, fp32 on the host (oracle/_ref)" if r["kind"] == "reference"
                             else "fp32 CPU restatement of the reference (oracle/vqa_oracle.py)"),
                  "bf16_mode_max_abs_rel_err": rel(got_bf16), "bf16_gate": 2e-2,
                  "bf16_top1_agree": float((got_bf16.argmax(1) == want.argmax(1)).float().mean()),
                  "tf32_mode_max_abs_rel_err": rel(got_tf32), "tf32_gate": 1e-3,
                  "tf32_top1_agree": float((got_tf32.argmax(1) == want.argmax(1)).float().mean()),
                  "tf32_mode_pairs_per_sec": B * 5 / (a.elapsed_time(b) * 1e-3)}
        del m_tf32, g2
    if rank_parity is not None:
        parity = dict(parity or {}, **rank_parity)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": max(Wm, 3),
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16", "data": "synthetic",
                "config": {"workload": WORKLOAD, "batch_per_gpu": B, "global_batch": B * world, "seq_len": L,
                           "precision": "bf16 backbone operands / fp16 text+fusion+head operands, fp32 accumulate",
                           "parallelism": f"batch-sharded x{world}, weights broadcast once",
                           "l2": "inputs 154 MB/GPU (fp32 NCHW) exceed the 126 MB L2; no flush needed",
                           "launch": f"one forward captured in a CUDA graph ({launches_per_step} kernels, programmatic dependent launch) per compute lane; "
                                     f"step k replays on lane k % {LANES} (own stream + own workspace), so consecutive steps overlap",
                           "compute_lanes": LANES},
                "single_stream": {"value": value_single, "ms_per_step": ms_single / K,
                                  "note": "the same K steps replayed strictly one after another on one stream"},
                "sustained": sustained, "library_bar": lib_bar,
                "roofline": roof, "cpu_baseline": cpu, "parity": parity, "config3_batch1024_u8": config3,
                "cached_image_side": cached_leg, "config5_one_image_16_questions": config5,
                "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms_e2e / K, "h2d_pinned_copy_gbps": h2d_gbps,
                        "h2d_ceiling": {
                            "per_rank_gbps_all_ranks_copying": h2d_conc_gbps, "aggregate_gbps": world * h2d_conc_gbps,
                            "pairs_per_sec": world * h2d_conc_gbps * 1e9 / (h2d / B),
                            "e2e_fraction": e2e_value / (world * h2d_conc_gbps * 1e9 / (h2d / B)),
                            "note": "copies only, every rank at once (barrier on both sides, slowest rank): what the "
                                    "host side of this box delivers when all GPUs pull their pixels; the e2e step also "
                                    "has to compute"},
                        "single_lane_value": world * B * K / (ms_e2e_1 * 1e-3), "compute_lanes": 3,
                        "two_lane_value": world * B * K / (ms_e2e_2 * 1e-3),
                        "from_idle_value": world * B * K / (ms_e2e_idle * 1e-3),
                        "from_idle_note": "the same K steps after 0.5 s of idle: `value` above is taken right after ~150 ms of "
                                          "continuous load (the one- and two-lane A/B runs and this leg's own warm-up), i.e. in the "
                                          "power-capped regime the `sustained` leg reports, while the device-resident `value` of "
                                          "this line starts from an idle GPU; the captured graphs themselves run at the same speed "
                                          "(tools/lane_probe.py)",
                        "path": "VQAInference.predict_tensors_pipelined: pinned uint8 HWC + ids + mask -> H2D (copy "
                                "stream, 6 device slots) -> normalise+forward+top-5 (three compute lanes: the forwards of "
                                "consecutive batches overlap on the GPU) -> D2H; every step copies its own "
                                "inputs and results; timed on the host clock around all K steps"},
                "latency_batch1": latency,
                "gpu_launches": int(launches), "clocks": clocks.summary()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_agreement(args):
    """Top-1 agreement of the engine with the fp32 oracle over N pairs (BASELINE: >= 99 % over 10k)."""
    import torch
    from oracle import vqa_oracle as O
    from vqa_b200.model import VQAModel
    from vqa_b200.synth import synth_batch
    torch.manual_seed(0)
    model = VQAModel().eval()
    sd = model.state_dict()
    model = model.cuda()
    n = agree = 0
    worst = 0.0
    b = 0
    while n < args.agreement:
        _, img, ids, mask = synth_batch(250, 1234 + b)
        with torch.no_grad():
            got, _ = model(img.cuda(), ids.cuda(), mask.cuda())
        want, _ = O.vqa_forward(sd, img, ids, mask)
        got = got.cpu()
        agree += int((got.argmax(1) == want.argmax(1)).sum())
        worst = max(worst, float((got - want).abs().max() / want.abs().max()))
        n += 250
        b += 1
    print(json.dumps({"pairs": n, "top1_agreement": agree / n, "max_abs_rel_logit_err": worst}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-ops", default="")
    ap.add_argument("--agreement", type=int, default=0)
    ap.add_argument("--quick", action="store_true", help="device-resident throughput only (A/B experiments)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the logits of the last timed step as DIR/logits.npy (rank 0's shard with several GPUs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.agreement):
        ap.error("--dump-outputs writes the B200 timed path's logits; --impl reference and --agreement do not run it")
    if args.impl == "reference":
        return run_reference(args)
    if args.agreement:
        return run_agreement(args)
    run_b200(args)


if __name__ == "__main__":
    main()
