"""Static model of a program's schedule (TEST INFRASTRUCTURE): what every op reads and writes, and which op pairs the
two-lane run of ``vqa_plan_run_range`` (csrc/plan.cu) orders.

``ACCESS`` says, per op kind and pointer field (``program.FIELDS``), whether the op reads the memory behind the field,
writes it, or both.  An access covers the bytes of the ``Buf`` the field points at (the whole allocation for every buffer
``OpList._buf`` makes; ``stem_in.data`` covers the data rows of ``stem_in`` only) and is charged to the allocation the
pointer falls in (``ws._bufs``).  Pointers into the weight arena are read-only constants and take no part; the external
slots (``ExtRef``) do: ``images``, ``ids``, ``mask`` and ``kv*`` are read, ``logits``, ``top_idx`` and ``top_probs``
written.  ``tests/test_schedule_cpu.py`` checks the table against the CPU emulator op by op.

``happens_before`` restates the stream / event logic of ``vqa_plan_run_range`` for consecutive whole-plan runs on one
caller stream: caller-stream order and side-stream order, the fork at the first lane-1 op, ``VQA_LANE_JOIN`` edges (a
side op waits for the main ops issued so far, a main op for the side ops issued so far), the final join, and the next run
issued after that join.  ``hazards`` lists every pair of ops with overlapping extents, at least one writing, that this
order leaves unordered; ``unwritten_reads`` lists every workspace byte an op reads that no op ordered before it in the
same run wrote, apart from ``ALLOW``.
"""
from __future__ import annotations

import bisect
from collections import defaultdict
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

from vqa_b200 import program as P

R, W, RW, SCRATCH, CONST, UNUSED = "r", "w", "rw", "scratch", "const", "-"
# R: reads what was there before the op; W: overwrites; RW: reads the old contents and writes (in place / counters);
# SCRATCH: the op writes it before it reads it back (no dependency on earlier contents); CONST: weight-arena pointer;
# UNUSED: the op ignores the field in this form even when it is set.

_PGL = dict(wg=CONST, bg=CONST, gamma=CONST, beta=CONST)
ACCESS: Dict[str, dict] = {
    "ingest": dict(src=R, dst=W),
    "gemm": dict(a0=R, a1=R, b=CONST, out=W, bias=CONST, res=R, dbg=W, sums=W, topk_idx=W, topk_probs=W,
                 topk_part=SCRATCH,      # per-tile partial winners, written by every tile and merged by the last one
                 topk_cnt=RW),           # arrival counter: incremented per tile, reset to 0 by the merging CTA
    "maxpool": dict(src=R, dst=W),
    "se_squeeze": dict(src=R, sums=W),
    "se_excite": dict(sums=R, w1=CONST, w2=CONST, scale=W),
    "spatial_map": dict(src=R, scale=R, wconv=CONST, att=W),
    "scale_relayout": dict(src=R, scale=R, att=R, dst=W),
    "embed": dict(ids=R, table=CONST, pe=CONST, dst=W, gamma=CONST, beta=CONST, ln_dst=W, mask_src=R, mask_dst=W,
                  mask_dstf=W),
    "layernorm": dict(src=R, gamma=CONST, beta=CONST, dst=W, pos=CONST, gamma2=CONST, beta2=CONST, dst2=W,
                      gamma3=CONST, beta3=CONST, dst3=W),
    "self_attn": dict(qkv=R, mask=R, out=W),
    "cross_attn": dict(q=R, kv=R, out=W, weights=W),
    # by ``phase``: 0 = pools + sum + LayerNorm, 1 = pools + [att; txt] for the gate GEMM, 2 = gate mix + LayerNorm of
    # the pools phase 1 stored (xatt / text / mask are set in every phase and read in phases 0 and 1 only)
    "pool_gate_ln": {
        0: dict(_PGL, xatt=R, text=R, mask=R, fused=W, att_pooled=W, txt_pooled=W, cat=W, pre=UNUSED),
        1: dict(_PGL, xatt=R, text=R, mask=R, fused=UNUSED, att_pooled=W, txt_pooled=W, cat=W, pre=UNUSED),
        2: dict(_PGL, xatt=UNUSED, text=UNUSED, mask=UNUSED, fused=W, att_pooled=R, txt_pooled=R, cat=W, pre=R),
    },
    "softmax_topk": dict(logits=R, idx=W, probs=W),
    "mask_prep": dict(src=R, dst=W, dstf=W),
    "grid_to_nchw": dict(src=R, dst=W),
    "copy_rows": dict(src=R, dst=W),
    "split_tf32": dict(src=R, dst=W),
    "stage_tail": dict(src=R, w1=CONST, w2=CONST, wconv=CONST, dst=W, scale=W, att=W,
                       sums=R),          # per-slab channel sums from the stage's last convolution (VQA_SE_EPILOGUE=1)
    "stem_pool": dict(a=R, w=CONST, out=W, dbg=W),
    "mlp_chain": dict(ctx=R, xres=R, xout=W, wo=CONST, w1=CONST, b1=CONST, w2=CONST, b2=CONST, ln_g=CONST, ln_b=CONST,
                      n_g=CONST, n_b=CONST, wn=CONST, y=W),
}


def field_modes(op: P.Op) -> Dict[str, str]:
    t = ACCESS[op.kind]
    return t[op.i.get("phase", 0)] if op.kind == "pool_gate_ln" else t


@dataclass
class Access:
    field: str
    mode: str
    key: str                    # allocation name, or "ext:<slot>"
    lo: Optional[int] = None    # workspace byte range [lo, hi) (None for external slots)
    hi: Optional[int] = None

    @property
    def reads(self):
        return self.mode in (R, RW)

    @property
    def writes(self):
        return self.mode in (W, RW, SCRATCH)


_EXT_NAME = {v: k for k, v in P.EXT.items()}


class Layout:
    """Byte extents of a program's workspace allocations."""

    def __init__(self, prog: P.OpList):
        self.prog = prog
        self.bufs = sorted(prog.ws._bufs, key=lambda b: b.offset)
        self._offs = [b.offset for b in self.bufs]

    def alloc_of(self, buf: P.Buf) -> P.Buf:
        k = bisect.bisect_right(self._offs, buf.offset) - 1
        while k >= 0 and not (self.bufs[k].offset <= buf.offset < self.bufs[k].offset + max(self.bufs[k].nbytes, 1)):
            k -= 1
        assert k >= 0, f"pointer at workspace offset {buf.offset} lies in no allocation"
        return self.bufs[k]

    def accesses(self, op: P.Op) -> List[Access]:
        modes = field_modes(op)
        assert set(modes) == set(P.FIELDS[op.kind]["p"]), (op.kind, sorted(set(modes) ^ set(P.FIELDS[op.kind]["p"])))
        out = []
        for f, ref in op.p.items():
            if ref is None or modes[f] == UNUSED:
                continue
            if isinstance(ref, P.ExtRef):
                assert modes[f] != CONST, (op.name, f)
                out.append(Access(f, modes[f], "ext:" + _EXT_NAME[ref.slot]))
                continue
            if ref.arena is not self.prog.ws:
                assert ref.arena is self.prog.W.arena, (op.name, f)
                continue                                    # weights: read-only constants
            assert modes[f] != CONST, f"{op.name}.{f} is a weight field but points into the workspace"
            a = self.alloc_of(ref)
            assert ref.offset + ref.nbytes <= a.offset + a.nbytes, (op.name, f, a.name)
            out.append(Access(f, modes[f], a.name, ref.offset, ref.offset + ref.nbytes))
        return out


# ----------------------------------------------------------------------------- zero-at-commit regions
def _stem_guard(prog, lay):
    """The 32 phase-pixel rows in front of the ingest data and the one row behind it.  The overlapping-row tensor maps of
    the tf32 stem (and of the bf16 stem with window=False) address an A row by its first phase-pixel, so rows that start
    left of or above the image must be in-range coordinates; they read these rows, which only ``Arena.commit(zero=True)``
    ever writes: they must hold zeros."""
    ing = [op for op in prog.ops if op.kind == "ingest"]
    if not ing:
        return []
    data = ing[0].p["dst"]
    a = lay.alloc_of(data)
    return [(a.offset, data.offset), (data.offset + data.nbytes, a.offset + a.nbytes)]


def _topk_counters(prog, lay):
    """The fused top-k epilogue's per-M-tile arrival counters: the CTA that finishes a tile's last N tile merges the
    partial winners and resets the counter to 0, so a run leaves it as the commit found it."""
    return [(b.offset, b.offset + b.nbytes) for b in lay.bufs if b.name.endswith(".topk_cnt")]


# (name, byte ranges of a program, reason): workspace bytes a run reads without writing them first
ALLOW = [
    ("stem_in guard rows", _stem_guard,
     "the overlapping-row stem tensor maps read them as the zero pixels left of / above the image"),
    ("*.topk_cnt", _topk_counters,
     "fused top-k arrival counter: zero at commit, reset to zero by the CTA that merges a tile's winners"),
]


def allowed_ranges(prog, allow=None) -> List[Tuple[int, int]]:
    lay = Layout(prog)
    return [r for _, fn, _ in (ALLOW if allow is None else allow) for r in fn(prog, lay) if r[1] > r[0]]


# ----------------------------------------------------------------------------- happens-before
def happens_before(ops: List[P.Op], runs: int = 2):
    """Bitset per op instance (run * n + op) of the instances ordered before it; and the stream (0 caller, 1 side) of
    each op.  Mirrors vqa_plan_run_range over the whole plan, ``runs`` times on one caller stream."""
    n = len(ops)
    two = any(op.lane & 1 for op in ops)
    front = [0, 0]                  # everything each stream has been made to wait for, itself included
    hb, stream = [], []
    for r in range(runs):
        side_used = False
        for k, op in enumerate(ops):
            s = 0
            if two:
                side, join = bool(op.lane & 1), bool(op.lane & P.LANE_JOIN)
                if side and not side_used:
                    front[1] |= front[0]                # fork
                    side_used = True
                elif join and side_used:
                    if side:
                        front[1] |= front[0]
                    else:
                        front[0] |= front[1]
                s = int(side)
            u = r * n + k
            hb.append(front[s])
            front[s] |= 1 << u
            stream.append(s)
        if side_used:
            front[0] |= front[1]                        # final join: the caller's stream sees the side lane's work
    return hb, stream


@dataclass
class Hazard:
    first: str
    second: str
    buffer: str
    lanes: Tuple[int, int]
    modes: Tuple[str, str]
    cross_run: bool

    def __str__(self):
        lane = ("main", "side")
        how = ("the next run is not ordered after this run's final join" if self.cross_run else
               f"no edge {lane[self.lanes[0]]} -> {lane[self.lanes[1]]}: a JOIN is missing on {self.second} "
               f"(or on a {lane[self.lanes[1]]}-lane op issued between the two)")
        return (f"{self.first} [{lane[self.lanes[0]]}, {self.modes[0]}] and {self.second} [{lane[self.lanes[1]]}, "
                f"{self.modes[1]}] both touch {self.buffer} unordered{' (consecutive runs)' if self.cross_run else ''}: "
                f"{how}")


def hazards(prog: P.OpList) -> List[Hazard]:
    ops = prog.ops
    n = len(ops)
    lay = Layout(prog)
    acc = [lay.accesses(op) for op in ops]
    hb, stream = happens_before(ops, 2)
    by_key = defaultdict(list)
    for u in range(2 * n):
        for a in acc[u % n]:
            by_key[a.key].append((u, a))
    out, seen = [], set()
    for key, lst in by_key.items():
        for i in range(len(lst)):
            u, a = lst[i]
            for v, b in lst[i + 1:]:
                if u == v or not (a.writes or b.writes) or (hb[v] >> u) & 1:
                    continue
                h = Hazard(ops[u % n].name, ops[v % n].name, key, (stream[u], stream[v]), (a.mode, b.mode),
                           u // n != v // n)
                tag = (h.first, h.second, key, h.cross_run)
                if tag not in seen:
                    seen.add(tag)
                    out.append(h)
    return out


def _merge(iv):
    out = []
    for lo, hi in sorted(iv):
        if out and lo <= out[-1][1]:
            out[-1][1] = max(out[-1][1], hi)
        else:
            out.append([lo, hi])
    return out


def _subtract(lo, hi, merged):
    """Parts of [lo, hi) not covered by the sorted, merged ranges."""
    out, cur = [], lo
    for a, b in merged:
        if b <= cur:
            continue
        if a >= hi:
            break
        if a > cur:
            out.append((cur, min(a, hi)))
        cur = max(cur, b)
        if cur >= hi:
            break
    if cur < hi:
        out.append((cur, hi))
    return out


def unwritten_reads(prog: P.OpList, allow=None) -> List[str]:
    """Reads of workspace bytes that no op ordered before the reader (in the same run) wrote and ``allow`` does not
    cover.  Each entry names the op, the field, the buffer and the byte range within the buffer."""
    ops = prog.ops
    lay = Layout(prog)
    acc = [lay.accesses(op) for op in ops]
    hb, _ = happens_before(ops, 1)
    allowed = allowed_ranges(prog, allow)
    out = []
    for k, op in enumerate(ops):
        reads = [a for a in acc[k] if a.reads and a.lo is not None]
        if not reads:
            continue
        cover = list(allowed)
        for j in range(k):
            if (hb[k] >> j) & 1:
                cover += [(a.lo, a.hi) for a in acc[j] if a.writes and a.lo is not None]
        cover = _merge(cover)
        for a in reads:
            base = lay.alloc_of(P.Buf(prog.ws, a.lo, 0))
            for lo, hi in _subtract(a.lo, a.hi, cover):
                out.append(f"{op.name}.{a.field} reads bytes [{lo - base.offset}, {hi - base.offset}) of {a.key} "
                           f"({base.nbytes} B) that no earlier op writes")
    return out


def untouched_buffers(prog: P.OpList) -> List[str]:
    lay = Layout(prog)
    used = {a.key for op in prog.ops for a in lay.accesses(op)}
    return [b.name for b in lay.bufs if b.name not in used]


def overlap_table(prog: P.OpList) -> str:
    """For each op, the ops of the other lane it may run alongside within one run (neither is ordered before the other)."""
    ops = prog.ops
    n = len(ops)
    hb, stream = happens_before(ops, 1)
    lines = []
    for k, op in enumerate(ops):
        other = [j for j in range(n) if stream[j] != stream[k] and not (hb[k] >> j) & 1 and not (hb[j] >> k) & 1]
        desc = "-" if not other else (f"{ops[other[0]].name} .. {ops[other[-1]].name} ({len(other)} ops)"
                                      if len(other) > 2 else ", ".join(ops[j].name for j in other))
        lines.append(f"{k:4d} {'side' if stream[k] else 'main'} {op.name:<24} {desc}")
    return "\n".join(lines)
