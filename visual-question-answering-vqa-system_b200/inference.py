"""``VQAInference``: the reference's predict API on the sm_100a engine.

Boundary #2 of SURVEY.md section 8b.  Same constructor, lazy ``load()`` with the same
fall-backs (random default model / 13-word default tokenizer / ``answer_{i}`` vocabulary when
the files do not exist), same method names and result schema as ``api/inference.py:36-358``:

    predict(image, question, top_k=5) -> {'question', 'answers': [{'answer','probability','index'}],
                                          'top_answer', 'confidence'}

What changes underneath: the image stays uint8 after PIL decode/resize and is normalised by
the ingest kernel on the GPU (one 150 KB host-to-device copy instead of a 602 KB fp32 one); the
forward, softmax and top-k run as one plan launch; the result comes back in a single
device-to-host copy instead of 2*k ``.item()`` synchronisations.  For a fixed batch size the
whole launch sequence is captured once in a CUDA graph and replayed (batch-1 latency path).
"""
from __future__ import annotations

import hashlib
import os
from collections import OrderedDict
from io import BytesIO
from typing import Dict, List, Optional, Tuple, Union

import torch
from PIL import Image

from .model import VQAModel, load_vqa_model
from .synth import IMAGENET_MEAN, IMAGENET_STD
from .text import AnswerVocabulary, Tokenizer

# Defaults of the reference's config singletons (utils/config.py:73-134,225) that the predict
# path reads; the reference's PathConfig (which creates directories on import) is not mirrored.
DEFAULT_QUESTION_VOCAB_SIZE = 10000
DEFAULT_NUM_ANSWERS = 1000
DEFAULT_MAX_QUESTION_LENGTH = 20
DEFAULT_IMAGE_SIZE = 224
DEFAULT_TOP_K = 5
_REF_BASE = "d:/cnn"   # the reference hard-codes Windows paths under this prefix (utils/config.py:27-44)
DEFAULT_CHECKPOINT = _REF_BASE + "/checkpoints/best_model.pt"
DEFAULT_QUESTION_VOCAB = _REF_BASE + "/data/question_vocab.json"
DEFAULT_ANSWER_VOCAB = _REF_BASE + "/data/vocab.json"

ImageLike = Union[str, bytes, Image.Image]


def get_device() -> str:
    """The engine has no CPU path: CUDA or a loud failure at load()."""
    return "cuda"


class VQAInference:
    def __init__(self, checkpoint_path: Optional[str] = None, device: Optional[str] = None,
                 question_vocab_path: Optional[str] = None, answer_vocab_path: Optional[str] = None,
                 use_cuda_graph: bool = True, image_cache_size: int = 0, max_graphs: int = 16):
        self.device = device or get_device()
        self.checkpoint_path = checkpoint_path or DEFAULT_CHECKPOINT
        self.question_vocab_path = question_vocab_path or DEFAULT_QUESTION_VOCAB
        self.answer_vocab_path = answer_vocab_path or DEFAULT_ANSWER_VOCAB
        self.model: Optional[VQAModel] = None
        self.tokenizer: Optional[Tokenizer] = None
        self.answer_vocab: Optional[AnswerVocabulary] = None
        self.transform = None
        self.use_cuda_graph = use_cuda_graph
        self.pipeline_lanes = 3     # concurrent forwards in predict_tensors_pipelined (each lane: own stream + plan workspace)
        self.gpu_resize = True      # PIL-exact resize of non-224x224 inputs on the device (SURVEY 8f, f1)
        # captured CUDA graphs (static pinned / device buffers + the plan they replay), one per (batch, length, k) shape:
        # an LRU, because every entry pins a plan workspace (7.4 MB per pair)
        self.max_graphs = max(1, int(max_graphs))
        self._graphs: "OrderedDict[tuple, dict]" = OrderedDict()
        self._is_loaded = False
        # SURVEY 8f row f2: LRU of per-image K/V entries (200 KB each) keyed by image content; 0 = off (reference behaviour:
        # every call recomputes the image side)
        self.image_cache_size = int(image_cache_size)
        self._image_cache: "OrderedDict[tuple, object]" = OrderedDict()
        self.cache_hits = self.cache_misses = 0

    # ------------------------------------------------------------------ loading
    def load(self):
        if self._is_loaded:
            return
        if not str(self.device).startswith("cuda"):
            raise RuntimeError("vqa_b200.VQAInference needs a CUDA device (sm_100a); there is no CPU path")
        if os.path.exists(self.checkpoint_path):
            self.model = load_vqa_model(self.checkpoint_path, self.device)
        else:
            self.model = VQAModel(vocab_size=DEFAULT_QUESTION_VOCAB_SIZE,
                                  num_answers=DEFAULT_NUM_ANSWERS).to(self.device)
        self.model.eval()
        if self.image_cache_size > 0:
            from .engine import check_cacheable
            check_cacheable(self.model.config)
        if os.path.exists(self.question_vocab_path):
            self.tokenizer = Tokenizer()
            self.tokenizer.load(self.question_vocab_path)
        else:
            self.tokenizer = Tokenizer(max_length=DEFAULT_MAX_QUESTION_LENGTH)
            self.tokenizer.build_vocab(["what is this", "what color", "how many", "is there", "where is",
                                        "what type"], min_freq=1)
        if os.path.exists(self.answer_vocab_path):
            self.answer_vocab = AnswerVocabulary()
            self.answer_vocab.load(self.answer_vocab_path)
        else:
            self.answer_vocab = AnswerVocabulary(num_answers=DEFAULT_NUM_ANSWERS)
            for i in range(DEFAULT_NUM_ANSWERS):
                self.answer_vocab.idx2answer[i] = f"answer_{i}"
        self.transform = self.preprocess_image
        self._is_loaded = True

    # ------------------------------------------------------------------ preprocessing
    @staticmethod
    def _open(image: ImageLike) -> Image.Image:
        if isinstance(image, str):
            pil = Image.open(image)
        elif isinstance(image, (bytes, bytearray)):
            pil = Image.open(BytesIO(image))
        else:
            pil = image
        if pil.mode != "RGB":
            pil = pil.convert("RGB")
        return pil

    def preprocess_image_u8(self, image: ImageLike, device_resize: Optional[bool] = None) -> torch.Tensor:
        """Decode + resize to 224x224 exactly like the reference's transform does for PIL inputs
        (torchvision Resize -> PIL antialiased bilinear, data/preprocess.py:117-121), but stop at
        uint8 HWC [224,224,3]: /255 and mean/std normalisation happen in the GPU ingest kernel.

        ``device_resize`` (default: on when the engine device is CUDA): images that are not 224x224 are uploaded
        at their native size and resized by the PIL-exact CUDA kernels (``vqa_resize_bilinear_u8``); the result
        is then a uint8 CUDA tensor, bit-identical to ``PIL.Image.resize`` (tested).  Off: PIL on the host."""
        pil = self._open(image)
        size = DEFAULT_IMAGE_SIZE
        if device_resize is None:
            device_resize = self.gpu_resize and str(self.device).startswith("cuda") and torch.cuda.is_available()
        if pil.size != (size, size):
            if device_resize:
                from .runtime import resize_bilinear_u8
                w, h = pil.size
                raw = torch.frombuffer(bytearray(pil.tobytes()), dtype=torch.uint8).view(h, w, 3)
                return resize_bilinear_u8(raw.to(self.device, non_blocking=True), size, size)
            pil = pil.resize((size, size), Image.BILINEAR)
        return torch.frombuffer(bytearray(pil.tobytes()), dtype=torch.uint8).view(size, size, 3)

    def preprocess_image(self, image: ImageLike) -> torch.Tensor:
        """Reference-compatible output: normalised float32 [1,3,224,224] on the CPU."""
        u8 = self.preprocess_image_u8(image, device_resize=False)
        x = u8.to(torch.float32).div(255.0).permute(2, 0, 1)
        mean = torch.tensor(IMAGENET_MEAN, dtype=torch.float32).view(3, 1, 1)
        std = torch.tensor(IMAGENET_STD, dtype=torch.float32).view(3, 1, 1)
        return ((x - mean) / std).unsqueeze(0)

    def preprocess_question(self, question: str) -> Tuple[torch.Tensor, torch.Tensor]:
        ids, mask = self.tokenizer.encode(question, add_special_tokens=True, padding=True, truncation=True)
        if self.model is not None and ids and max(ids) >= self.model.config["vocab_size"]:
            # the reference's nn.Embedding raises here (tokenizer vocabulary larger than the checkpoint's); the CUDA embed
            # kernel cannot raise, so the range is checked on the host where the ids still are
            raise IndexError(f"token id {max(ids)} is out of range for the model's vocab_size "
                             f"{self.model.config['vocab_size']} (index out of range in self)")
        return torch.tensor([ids], dtype=torch.long), torch.tensor([mask], dtype=torch.long)

    # ------------------------------------------------------------------ execution
    def _run(self, u8: torch.Tensor, ids: torch.Tensor, mask: torch.Tensor, top_k: int):
        """u8 [B,224,224,3], ids/mask [B,L] on the host -> (top_idx [B,k], top_probs [B,k]) on the host."""
        B, L = ids.shape
        if top_k < 1:
            raise ValueError("top_k must be at least 1")
        k = min(top_k, self.model.num_answers)
        if not self.use_cuda_graph:
            with torch.no_grad():
                idx, probs = self.model.predict(u8.to(self.device, non_blocking=True),
                                                ids.to(self.device, non_blocking=True),
                                                mask.to(self.device, non_blocking=True), top_k=k)
            return idx.cpu(), probs.cpu()
        key = (B, L, k)
        g = self._graph_get(key)
        if g is None:
            g = self._graph_put(key, self._capture(B, L, k))
        if u8.is_cuda:                      # resized on the device already
            g["d_u8"].copy_(u8, non_blocking=True)
        else:
            g["h_u8"].copy_(u8)
            g["d_u8"].copy_(g["h_u8"], non_blocking=True)
        g["h_ids"].copy_(ids)
        g["h_mask"].copy_(mask)
        g["graph"].replay()
        torch.cuda.current_stream().synchronize()
        return g["h_idx"].clone(), g["h_probs"].clone()

    def _graph_get(self, key):
        g = self._graphs.get(key)
        if g is not None:
            self._graphs.move_to_end(key)
        return g

    def _graph_put(self, key, g):
        self._graphs[key] = g
        while len(self._graphs) > self.max_graphs:
            self._graphs.popitem(last=False)      # drops the graph, its buffers and its reference to the plan
        return g

    def _capture(self, B: int, L: int, k: int) -> dict:
        """Static pinned/device buffers + one CUDA graph: H2D copies, the plan's launches, D2H copies."""
        dev = torch.device(self.device)
        g = {
            "h_u8": torch.empty(B, 224, 224, 3, dtype=torch.uint8).pin_memory(),
            "h_ids": torch.empty(B, L, dtype=torch.long).pin_memory(),
            "h_mask": torch.empty(B, L, dtype=torch.long).pin_memory(),
            "h_idx": torch.empty(B, k, dtype=torch.long).pin_memory(),
            "h_probs": torch.empty(B, k, dtype=torch.float32).pin_memory(),
            "d_u8": torch.zeros(B, 224, 224, 3, dtype=torch.uint8, device=dev),
            "d_ids": torch.zeros(B, L, dtype=torch.long, device=dev),
            "d_mask": torch.ones(B, L, dtype=torch.long, device=dev),
        }
        engine = self.model.engine()
        with torch.no_grad():
            for _ in range(2):   # warm up: builds the plan, loads kernels
                engine.predict(g["d_u8"], g["d_ids"], g["d_mask"], k)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):       # the image copy stays outside: it may come from the device-side resize
                g["d_ids"].copy_(g["h_ids"], non_blocking=True)
                g["d_mask"].copy_(g["h_mask"], non_blocking=True)
                idx, probs = engine.predict(g["d_u8"], g["d_ids"], g["d_mask"], k)
                g["h_idx"].copy_(idx, non_blocking=True)
                g["h_probs"].copy_(probs, non_blocking=True)
        g["graph"] = graph
        g["keep"] = (idx, probs, engine.last_plan)   # the graph replays this plan's workspace: keep it alive
        return g

    @torch.no_grad()
    def predict_tensors_pipelined(self, batches, top_k: int = DEFAULT_TOP_K):
        """Throughput path: iterate over host batches ``(u8 [B,224,224,3], ids [B,L], mask [B,L])`` (ideally
        pinned) and yield ``(top_idx, top_probs)`` host tensors in order.

        ``pipeline_lanes`` compute lanes (default 3) run on their own streams with their own plan workspace, so the
        forward of batch i+1 overlaps the forward of batch i on the GPU: the small launch-latency-bound kernels of one
        batch's text / fusion / head path and the last, partially filled wave of each persistent convolution leave SMs
        idle that the other batch's kernels fill.  Inputs go through ``2 * lanes`` device slots filled by a copy stream
        (the host-to-device copy of a later batch runs while earlier ones compute); each slot's forward is captured in
        its own CUDA graph; each result comes back in one small device-to-host copy."""
        if not self._is_loaded:
            self.load()
        dev = torch.device(self.device)
        lanes = max(1, int(getattr(self, "pipeline_lanes", 3)))
        n_slots = max(lanes, int(getattr(self, "pipeline_slots", 0) or 2 * lanes))
        if not hasattr(self, "_pipe_streams") or len(self._pipe_streams[1]) != lanes or self._pipe_nslots != n_slots:
            self._pipe_streams = (torch.cuda.Stream(dev), [torch.cuda.Stream(dev) for _ in range(lanes)])
            self._pipe_nslots = n_slots
            self._pipe_slots = {}       # (B, L, k) -> input/output slots with their captured graphs (kept across calls)
        copy_s, comp = self._pipe_streams
        k = min(top_k, self.model.num_answers)
        engine = self.model.engine()
        pending = []   # (done_event, h_idx, h_probs)

        def drain(n_keep):
            while len(pending) > n_keep:
                ev, hi, hp = pending.pop(0)
                ev.synchronize()
                yield hi.clone(), hp.clone()

        for i, (u8, ids, mask) in enumerate(batches):
            B, L = ids.shape
            slots = self._pipe_slots.get((B, L, k))
            if slots is None:
                slots = self._pipe_slots[(B, L, k)] = [None] * n_slots
                while len(self._pipe_slots) > 4:        # shapes are few in practice; never keep more than four sets
                    self._pipe_slots.pop(next(iter(self._pipe_slots)))
            j = i % n_slots
            lane = j % lanes
            comp_s = comp[lane]
            sl = slots[j]
            if sl is None:
                sl = {"shape": (B, L),
                      "d_u8": torch.empty(B, 224, 224, 3, dtype=torch.uint8, device=dev),
                      "d_ids": torch.empty(B, L, dtype=torch.long, device=dev),
                      "d_mask": torch.empty(B, L, dtype=torch.long, device=dev),
                      "h_idx": torch.empty(B, k, dtype=torch.long).pin_memory(),
                      "h_probs": torch.empty(B, k, dtype=torch.float32).pin_memory(),
                      "copied": torch.cuda.Event(), "free": None}
                slots[j] = sl
            with torch.cuda.stream(copy_s):
                if sl["free"] is not None:
                    copy_s.wait_event(sl["free"])          # the forward that last read this slot has finished
                sl["d_u8"].copy_(u8, non_blocking=True)
                sl["d_ids"].copy_(ids, non_blocking=True)
                sl["d_mask"].copy_(mask, non_blocking=True)
                sl["copied"].record(copy_s)
            with torch.cuda.stream(comp_s):
                comp_s.wait_event(sl["copied"])
                if self.use_cuda_graph:
                    if sl.get("graph") is None:             # capture this slot's forward once (static buffers)
                        engine.predict(sl["d_u8"], sl["d_ids"], sl["d_mask"], k, slot=lane)   # builds the plan, loads kernels
                        torch.cuda.synchronize(dev)
                        gr = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(gr, stream=comp_s):
                            sl["idx"], sl["probs"] = engine.predict(sl["d_u8"], sl["d_ids"], sl["d_mask"], k, slot=lane)
                        sl["graph"], sl["plan"] = gr, engine.last_plan   # keep the replayed plan's workspace alive
                    sl["graph"].replay()
                    idx, probs = sl["idx"], sl["probs"]
                else:
                    idx, probs = engine.predict(sl["d_u8"], sl["d_ids"], sl["d_mask"], k, slot=lane)
                sl["free"] = torch.cuda.Event()
                sl["free"].record(comp_s)
                sl["h_idx"].copy_(idx, non_blocking=True)
                sl["h_probs"].copy_(probs, non_blocking=True)
                done = torch.cuda.Event()
                done.record(comp_s)
            pending.append((done, sl["h_idx"], sl["h_probs"]))
            yield from drain(n_slots - 1)                   # a slot's host buffers are read before the slot is refilled
        yield from drain(0)

    def _format(self, question: str, idx_row, prob_row) -> Dict:
        answers = []
        for i, p in zip(idx_row, prob_row):
            i = int(i)
            answers.append({"answer": self.answer_vocab.decode(i), "probability": float(p), "index": i})
        return {"question": question, "answers": answers, "top_answer": answers[0]["answer"],
                "confidence": answers[0]["probability"]}

    # ------------------------------------------------------------------ image cache (SURVEY 8f row f2)
    @staticmethod
    def image_key(image: ImageLike) -> tuple:
        """Content key of an input image: file identity for paths, SHA-1 of the bytes / pixels otherwise."""
        if isinstance(image, str):
            st = os.stat(image)
            return ("path", os.path.abspath(image), st.st_mtime_ns, st.st_size)
        if isinstance(image, (bytes, bytearray)):
            return ("bytes", hashlib.sha1(image).hexdigest())
        h = hashlib.sha1(f"{image.mode}|{image.size}".encode())
        h.update(image.tobytes())
        return ("pil", h.hexdigest())

    @torch.no_grad()
    def encode_image(self, image: ImageLike):
        """Backbone + projector + cross-attention K/V of one image (an ``engine.ImageCache`` of one entry).  With
        ``image_cache_size > 0`` entries are kept in an LRU keyed by ``image_key`` and reused across calls."""
        if not self._is_loaded:
            self.load()
        key = self.image_key(image) if self.image_cache_size > 0 else None
        if key is not None and key in self._image_cache:
            self._image_cache.move_to_end(key)
            self.cache_hits += 1
            return self._image_cache[key]
        u8 = self.preprocess_image_u8(image).unsqueeze(0).to(self.device, non_blocking=True)
        entry = self.model.encode_images(u8)
        if key is not None:
            self.cache_misses += 1
            self._image_cache[key] = entry
            while len(self._image_cache) > self.image_cache_size:
                self._image_cache.popitem(last=False)
        return entry

    @torch.no_grad()
    def answer(self, cache, questions: List[str], top_k: int = DEFAULT_TOP_K) -> List[Dict]:
        """Questions against encoded images: ``cache`` is what ``encode_image`` returned (or an ``ImageCache`` of n
        entries with ``len(questions) % n == 0``: entry i answers the next len(questions) / n questions).  Only the text
        encoder, the cross-attention, the gate and the head run; results equal ``predict`` on the same image."""
        if not self._is_loaded:
            self.load()
        if not questions:
            return []
        pairs = [self.preprocess_question(q) for q in questions]
        ids = torch.cat([p[0] for p in pairs], dim=0)
        mask = torch.cat([p[1] for p in pairs], dim=0)
        k = min(top_k, self.model.num_answers)
        if self.use_cuda_graph:
            idx, probs = self._answer_graph(cache, ids, mask, k)
        else:
            _, idx, probs = self.model.engine().answer(cache, ids.to(self.device, non_blocking=True),
                                                       mask.to(self.device, non_blocking=True), top_k=k)
            idx, probs = idx.cpu(), probs.cpu()
        return [self._format(q, idx[i].tolist(), probs[i].tolist()) for i, q in enumerate(questions)]

    def _answer_graph(self, cache, ids: torch.Tensor, mask: torch.Tensor, k: int):
        """Question side as one CUDA-graph replay per (questions, length, k, images) shape: static K/V buffers (the cache
        entry is copied in, 200 KB per image), H2D of ids / mask, the question-side plan, D2H of the top-k."""
        B, L = ids.shape
        key = ("answer", B, L, k, cache.n_images, len(cache.kv))
        g = self._graph_get(key)
        dev = torch.device(self.device)
        if g is None:
            from .engine import ImageCache
            g = {"kv": [torch.zeros_like(t, device=dev) for t in cache.kv],
                 "h_ids": torch.zeros(B, L, dtype=torch.long).pin_memory(),
                 "h_mask": torch.ones(B, L, dtype=torch.long).pin_memory(),
                 "h_idx": torch.empty(B, k, dtype=torch.long).pin_memory(),
                 "h_probs": torch.empty(B, k, dtype=torch.float32).pin_memory(),
                 "d_ids": torch.zeros(B, L, dtype=torch.long, device=dev),
                 "d_mask": torch.ones(B, L, dtype=torch.long, device=dev)}
            static = ImageCache(g["kv"], cache.n_images)
            engine = self.model.engine()
            for _ in range(2):       # warm up: builds the plan, loads kernels
                engine.answer(static, g["d_ids"], g["d_mask"], top_k=k)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                g["d_ids"].copy_(g["h_ids"], non_blocking=True)
                g["d_mask"].copy_(g["h_mask"], non_blocking=True)
                _, idx, probs = engine.answer(static, g["d_ids"], g["d_mask"], top_k=k)
                g["h_idx"].copy_(idx, non_blocking=True)
                g["h_probs"].copy_(probs, non_blocking=True)
            g["graph"], g["keep"] = graph, (idx, probs, engine.last_plan)
            self._graph_put(key, g)
        for dst, src in zip(g["kv"], cache.kv):
            dst.copy_(src, non_blocking=True)
        g["h_ids"].copy_(ids)
        g["h_mask"].copy_(mask)
        g["graph"].replay()
        torch.cuda.current_stream().synchronize()
        return g["h_idx"].clone(), g["h_probs"].clone()

    def cache_info(self) -> Dict:
        return {"size": len(self._image_cache), "capacity": self.image_cache_size, "hits": self.cache_hits,
                "misses": self.cache_misses,
                "bytes": sum(e.nbytes for e in self._image_cache.values())}

    @torch.no_grad()
    def predict(self, image: ImageLike, question: str, top_k: int = DEFAULT_TOP_K) -> Dict:
        if not self._is_loaded:
            self.load()
        if self.image_cache_size > 0:       # image side from the LRU (computed on a miss), question side per call
            return self.answer(self.encode_image(image), [question], top_k)[0]
        u8 = self.preprocess_image_u8(image).unsqueeze(0)
        ids, mask = self.preprocess_question(question)
        idx, probs = self._run(u8, ids, mask, top_k)
        return self._format(question, idx[0].tolist(), probs[0].tolist())

    @torch.no_grad()
    def predict_questions(self, image: ImageLike, questions: List[str], top_k: int = DEFAULT_TOP_K) -> List[Dict]:
        """One image, many questions (SURVEY 8f row f2; not in the reference API): the backbone, the projector and
        the K/V projections of the cross-attention layers run once, every question cross-attends the same 49-token
        feature map.  Same result dicts as ``predict`` called per question."""
        if not self._is_loaded:
            self.load()
        if not questions:
            return []
        if self.image_cache_size > 0:       # image side from the LRU, question side only
            return self.answer(self.encode_image(image), questions, top_k)
        u8 = self.preprocess_image_u8(image).unsqueeze(0).to(self.device, non_blocking=True)
        pairs = [self.preprocess_question(q) for q in questions]
        ids = torch.cat([p[0] for p in pairs], dim=0).to(self.device, non_blocking=True)
        mask = torch.cat([p[1] for p in pairs], dim=0).to(self.device, non_blocking=True)
        k = min(top_k, self.model.num_answers)
        idx, probs = self.model.predict(u8, ids, mask, top_k=k)
        idx, probs = idx.cpu(), probs.cpu()
        return [self._format(q, idx[i].tolist(), probs[i].tolist()) for i, q in enumerate(questions)]

    @torch.no_grad()
    def predict_batch(self, images: List[ImageLike], questions: List[str], top_k: int = DEFAULT_TOP_K) -> List[Dict]:
        if len(images) != len(questions):
            raise ValueError("Number of images must match number of questions")
        if not self._is_loaded:
            self.load()
        tensors = [self.preprocess_image_u8(im) for im in images]
        if any(t.is_cuda for t in tensors):
            tensors = [t.to(self.device, non_blocking=True) for t in tensors]
        u8 = torch.stack(tensors, dim=0)
        pairs = [self.preprocess_question(q) for q in questions]
        ids = torch.cat([p[0] for p in pairs], dim=0)
        mask = torch.cat([p[1] for p in pairs], dim=0)
        idx, probs = self._run(u8, ids, mask, top_k)
        return [self._format(q, idx[b].tolist(), probs[b].tolist()) for b, q in enumerate(questions)]

    def get_model_info(self) -> Dict:
        if not self._is_loaded:
            self.load()
        return {"device": str(self.device), "vocab_size": self.tokenizer.vocab_size,
                "num_answers": self.answer_vocab.num_answers, "parameters": self.model.get_num_parameters(),
                "config": self.model.config}


_inference_instance: Optional[VQAInference] = None


def get_inference_engine() -> VQAInference:
    global _inference_instance
    if _inference_instance is None:
        _inference_instance = VQAInference()
        _inference_instance.load()
    return _inference_instance
