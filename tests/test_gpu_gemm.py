"""tcgen05 tap-shifted GEMM (VQA_OP_GEMM) through the C ABI against the CPU emulator.

Ordered from the plainest configuration to the ones that rely on less-documented hardware
behaviour (row-shifted UMMA descriptors inside a SWIZZLE_128B window, overlapping-row tensor
maps), so that a failure in the latter does not hide the former.
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

from vqa_b200 import program as P  # noqa: E402
import gpu_util as G  # noqa: E402


def _weights(device, name, n, k, dtype, seed, npad=None):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(n, k, generator=g) * (1.0 / k ** 0.5)
    if dtype == torch.float32:
        w = P.round_tf32(w)
    if npad:
        w = P._pad_rows(w, npad)
    W = P.Weights(device)
    W.add(name + ".w", w, dtype)
    W.add(name + ".b", P._pad_rows(torch.randn(n, generator=g), npad or 1), torch.float32)
    return W


def _fill(ol, name, seed, scale=1.0):
    b, dtype, shape = ol.named[name]
    g = torch.Generator().manual_seed(seed)
    t = (torch.randn(*shape, generator=g) * scale)
    if dtype == torch.float32:
        t = P.round_tf32(t)
    return t.to(dtype)


@pytest.mark.parametrize("M,K,N", [(128, 64, 64), (300, 128, 64), (1000, 192, 128), (517, 256, 256), (130, 512, 512)])
@pytest.mark.parametrize("out_dtype", [P.OUT_BF16, P.OUT_F32])
def test_plain_bf16_gemm(M, K, N, out_dtype):
    def build(device):
        W = _weights(device, "w", N, K, torch.bfloat16, 1).finalize()
        ol = P.OpList(W, device)
        a = ol._buf("a", torch.bfloat16, M, K)
        o = ol._buf("o", torch.bfloat16 if out_dtype == P.OUT_BF16 else torch.float32, M, N)
        ol.gemm("g", dtype=P.DT_BF16, M=M, N=N, a0=a, a0_shape=(M, K, K), groups=[(0, 0, 0, K // 64, [0])],
                w="w.w", bias="w.b", out=o, ldo=N, out_dtype=out_dtype, relu=True)
        ol.commit()
        G.named(ol, "a").copy_(_fill(ol, "a", 2))
        return ol
    cpu, gpu, _, _ = G.run_pair(build)
    tol = 2e-2 if out_dtype == P.OUT_BF16 else 2e-3
    G.report(f"plain bf16 M{M} K{K} N{N}", G.named(gpu, "o"), G.named(cpu, "o"), atol=tol, rtol=1e-2)


@pytest.mark.parametrize("M,K,N,ldo", [(256, 256, 256, 256), (100, 256, 768, 768), (77, 1024, 256, 256),
                                      (256, 256, 1000, 1000), (5, 512, 36, 40), (1500, 256, 256, 256),
                                      (64, 256, 3000, 3000)])   # N beyond the 2048-entry bias table
@pytest.mark.parametrize("max_ctas", [0, 2])
def test_tf32_linear_with_residual(M, K, N, ldo, max_ctas):
    def build(device):
        W = _weights(device, "w", N, K, torch.float32, 3, npad=256).finalize()
        ol = P.OpList(W, device)
        a = ol._buf("a", torch.float32, M, K)
        o = ol._buf("o", torch.float32, M, ldo)
        ol.linear("lin", a, M, K, "w.w", "w.b", o, N, ldo=ldo, res=o)
        ol.ops[-1].i["max_ctas"] = max_ctas
        ol.commit()
        G.named(ol, "a").copy_(_fill(ol, "a", 4))
        G.named(ol, "o").copy_(_fill(ol, "o", 5))
        return ol
    cpu, gpu, _, _ = G.run_pair(build)
    G.report(f"tf32 M{M} K{K} N{N}", G.named(gpu, "o"), G.named(cpu, "o"), atol=2e-3, rtol=2e-3)


def _conv_case(device, window, B, H, Wd, cin, cout, residual, mt=None, max_ctas=0, extra_ds=False, sums=False, tail=None):
    g = P.Grid(B, H, Wd)
    gen = torch.Generator().manual_seed(7)
    k = 9 * cin + (cin if extra_ds else 0)
    W = P.Weights(device)
    W.add("c.w", torch.randn(cout, k, generator=gen) * (1.0 / k ** 0.5), torch.bfloat16)
    W.add("c.b", torch.randn(cout, generator=gen), torch.float32)
    W.finalize()
    ol = P.OpList(W, device, window=window)
    x = ol._buf("x", torch.bfloat16, g.rows, cin)
    x1 = ol._buf("x1", torch.bfloat16, g.rows, cin)
    o = ol._buf("o", torch.bfloat16, g.rows, cout)
    groups, halo, mt_auto = ol._conv3x3_groups(g, cin // 64, cout)
    if extra_ds:
        groups = groups + [(1, 0, 0, cin // 64, [halo])]
    ol.gemm("conv", dtype=P.DT_BF16, M=g.rows, N=cout, a0=x, a0_shape=(g.rows, cin, cin), groups=groups,
            a1=x1 if extra_ds else None, a1_shape=(g.rows, cin, cin) if extra_ds else None,
            w="c.w", bias="c.b", out=o, ldo=cout, out_dtype=P.OUT_BF16, relu=True,
            res=x if residual else None, res_dtype=P.OUT_BF16 if residual else -1, ldr=cin, grid=g,
            halo=halo, MT=mt or mt_auto, sums=ol._buf("sums", torch.float32, (g.rows + 31) // 32, cout) if sums else None)
    ol.ops[-1].i["max_ctas"] = max_ctas
    if tail is not None:   # SE (+ spatial attention) stage tail fed by the slab sums: "stream" | "staged"
        r = max(cout // 16, 1)
        gen2 = torch.Generator().manual_seed(8)
        W2 = P.Weights(device)
        W2.add("se.w1", torch.randn(r, cout, generator=gen2) * 0.2, torch.float32)
        W2.add("se.w2", torch.randn(r, cout, generator=gen2) * 0.5, torch.float32)
        W2.add("sp.w", torch.randn(2, 49, generator=gen2) * 0.1, torch.float32)
        W2.finalize()
        ol._w2 = W2
        mode = 1 if tail == "stream" else 0
        gn = P.Grid(B, H // 2, Wd // 2) if mode else g
        dst = ol._buf("dst", torch.bfloat16, (4 if mode else 1) * gn.rows, cout)
        sc = ol._buf("scale", torch.float32, B, cout)
        att = ol._buf("att", torch.float32, B, H * Wd) if tail == "staged" else None
        split = 0
        if tail == "stream":
            split = 2 if H % 4 == 0 else 1
        ol._op("stage_tail", "tail",
               dict(B=B, C=cout, H=H, W=Wd, P=g.P, RPI=g.rpi, R=r, ks=7 if tail == "staged" else 0, mode=mode, Po=gn.P,
                    RPIo=gn.rpi, phase_rows=gn.rows if mode else g.rows, CS=1, f32=0, split=split),
               dict(src=o, w1=W2.buf("se.w1"), w2=W2.buf("se.w2"), wconv=W2.buf("sp.w") if tail == "staged" else None,
                    dst=dst, scale=sc, att=att, sums=ol.named["sums"][0]))
    ol.commit()
    # valid pixels random, shared pads zero (the layout invariant every producer keeps)
    xv = torch.randn(g.rows, cin, generator=gen)
    r = torch.arange(g.rows) % g.rpi
    valid = ((r // g.P) < g.H) & ((r % g.P) < g.W)
    xv[~valid] = 0
    G.named(ol, "x").copy_(xv.to(torch.bfloat16))
    x1v = torch.randn(g.rows, cin, generator=gen)
    x1v[~valid] = 0
    G.named(ol, "x1").copy_(x1v.to(torch.bfloat16))
    return ol


@pytest.mark.parametrize("B,H,W,cin,cout,residual", [(2, 8, 8, 64, 64, False), (3, 14, 14, 128, 128, True),
                                                    (2, 7, 7, 256, 512, False)])
@pytest.mark.parametrize("max_ctas", [0, 2])
def test_conv3x3_per_tap_loads(B, H, W, cin, cout, residual, max_ctas):
    """window=False: every tap TMA-loads its own row-shifted A tile (negative / out-of-range rows zero-fill)."""
    cpu, gpu, _, _ = G.run_pair(lambda d: _conv_case(d, False, B, H, W, cin, cout, residual and cin == cout,
                                                     max_ctas=max_ctas))
    G.report(f"conv per-tap {B}x{H}x{W} {cin}->{cout}", G.named(gpu, "o"), G.named(cpu, "o"), atol=3e-2, rtol=2e-2)


def test_conv3x3_matches_torch_conv2d():
    """The padded-flat shift-GEMM is a real 3x3 convolution: compare with F.conv2d on the valid pixels."""
    B, H, Wd, cin, cout = 2, 9, 11, 64, 64
    cpu, gpu, _, _ = G.run_pair(lambda d: _conv_case(d, False, B, H, Wd, cin, cout, False))
    g = P.Grid(B, H, Wd)
    import emulator as E
    idx = E._grid_index(B, H, Wd, g.P, g.rpi)
    x = G.named(cpu, "x")[idx].float().view(B, H, Wd, cin).permute(0, 3, 1, 2)
    w = cpu.W.tensor("c.w").float().view(cout, 3, 3, cin).permute(0, 3, 1, 2)
    want = torch.relu(torch.nn.functional.conv2d(x, w, cpu.W.tensor("c.b"), padding=1))
    got = G.named(gpu, "o").cpu()[idx].float().view(B, H, Wd, cout).permute(0, 3, 1, 2)
    G.report("conv vs F.conv2d", got, want, atol=3e-2, rtol=2e-2)
    pads = torch.ones(g.rows, dtype=torch.bool)
    pads[idx] = False
    assert G.named(gpu, "o").cpu()[pads].abs().max() == 0  # shared zero padding is preserved


@pytest.mark.parametrize("max_ctas", [0, 1])
def test_stem_overlapping_row_tensor_map(max_ctas):
    """Stem trick: rows of 64 bf16 that start every 16 elements (overlapping global strides)."""
    rows, guard = 3000, 32
    def build(device):
        W = _weights(device, "w", 64, 256, torch.bfloat16, 11).finalize()
        ol = P.OpList(W, device)
        a = ol._buf("a", torch.bfloat16, rows + guard, 16)
        o = ol._buf("o", torch.float32, rows, 64)
        taps = [(0, (ia - 2) * 30 - 2 + guard, 0, 1, [0]) for ia in range(4)]
        ol.gemm("stem", dtype=P.DT_BF16, M=rows, N=64, a0=a, a0_shape=(rows + guard, 64, 16), groups=taps,
                w="w.w", bias="w.b", out=o, ldo=64, out_dtype=P.OUT_F32)
        ol.ops[-1].i["max_ctas"] = max_ctas
        ol.commit()
        G.named(ol, "a").copy_(_fill(ol, "a", 12))
        return ol
    cpu, gpu, _, _ = G.run_pair(build)
    G.report("stem overlapped map", G.named(gpu, "o"), G.named(cpu, "o"), atol=2e-2, rtol=1e-2)


@pytest.mark.parametrize("B,H,W,cin,cout,mt", [(2, 8, 8, 64, 64, 1), (2, 56, 56, 64, 64, 1), (3, 14, 14, 128, 128, 2),
                                              (4, 28, 28, 128, 128, 2), (2, 7, 7, 512, 512, 2)])
@pytest.mark.parametrize("max_ctas", [0, 3])
def test_conv3x3_window(B, H, W, cin, cout, mt, max_ctas):
    """window=True: one A window per K chunk, taps are row-shifted UMMA descriptors into it.

    max_ctas=3 forces many tiles per persistent CTA (ring wrap-around, both MMA issuers, TMEM double
    buffering).  Measured on B200 (round 1): with the descriptor base_offset field left 0 the row-shifted start
    address reads the TMA-written SWIZZLE_128B window correctly (the swizzle is a function of the
    absolute shared-memory address); setting base_offset=(addr>>7)&7 gives wrong results."""
    cpu, gpu, _, _ = G.run_pair(lambda d: _conv_case(d, True, B, H, W, cin, cout, cin == cout, mt=mt,
                                                     max_ctas=max_ctas))
    G.report(f"conv window max_ctas={max_ctas} {B}x{H}x{W} {cin}->{cout} MT{mt}", G.named(gpu, "o"),
             G.named(cpu, "o"), atol=3e-2, rtol=2e-2)


@pytest.mark.parametrize("B,H,W,c,mt,tail", [(3, 56, 56, 64, 1, "stream"), (2, 28, 28, 128, 2, "stream"), (5, 14, 14, 256, 2, "staged"),
                                            (4, 7, 7, 512, 2, "staged"), (3, 8, 12, 64, 1, "stream")])
@pytest.mark.parametrize("max_ctas", [0, 3])
def test_conv3x3_slab_sums_feed_the_stage_tail(B, H, W, c, mt, tail, max_ctas):
    """The last convolution of a stage also writes the column sums of every 32-row slab of its output (SE squeeze
    partial sums); the stage tail derives the SE scale from them -- streaming form without spatial attention, staged
    form with it.  The emulator computes the mean from the stored bf16 data instead: both must agree."""
    cpu, gpu, _, _ = G.run_pair(lambda d: _conv_case(d, True, B, H, W, c, c, True, mt=mt, max_ctas=max_ctas, sums=True, tail=tail))
    G.report("conv out", G.named(gpu, "o"), G.named(cpu, "o"), atol=3e-2, rtol=2e-2)
    g = P.Grid(B, H, W)
    full = slice((g.rpi + 31) // 32, (g.rows // 32))     # slabs of the middle images (never partial at the end of the tensor)
    G.report("slab sums", G.named(gpu, "sums")[full], G.named(cpu, "sums")[full], atol=2e-2, rtol=1e-3)
    G.report("SE scale", G.named(gpu, "scale"), G.named(cpu, "scale"), atol=2e-3, rtol=2e-3)
    if tail == "staged":
        G.report("spatial attention", G.named(gpu, "att"), G.named(cpu, "att"), atol=2e-3, rtol=2e-3)
    G.report("tail dst", G.named(gpu, "dst"), G.named(cpu, "dst"), atol=2e-2, rtol=1.6e-2)


def test_conv3x3_window_with_shortcut_group():
    cpu, gpu, _, _ = G.run_pair(lambda d: _conv_case(d, True, 3, 14, 14, 128, 128, False, mt=2, extra_ds=True))
    G.report("conv window + shortcut K group", G.named(gpu, "o"), G.named(cpu, "o"), atol=3e-2, rtol=2e-2)


@pytest.mark.parametrize("max_ctas", [0, 2])
@pytest.mark.parametrize("mt", [1, 2])
def test_stem_window_32_byte_rows(mt, max_ctas):
    """Stem form: 32-byte rows (SWIZZLE_32B), one asymmetric window per tile, 16 row-shifted K=16 taps."""
    Pw, rows = 30, 4000
    def build(device):
        W = _weights(device, "w", 64, 256, torch.bfloat16, 21).finalize()
        ol = P.OpList(W, device)
        a = ol._buf("a", torch.bfloat16, rows, 16)
        o = ol._buf("o", torch.float32 if mt == 2 else torch.bfloat16, rows, 64)
        lo, hi = 2 * Pw + 2, Pw + 1
        rels = [lo + (ia - 2) * Pw + (ib - 2) for ia in range(4) for ib in range(4)]
        ol.gemm("stem", dtype=P.DT_BF16, M=rows, N=64, a0=a, a0_shape=(rows, 16, 16), groups=[(0, 0, 0, 1, rels)],
                w="w.w", bias="w.b", out=o, ldo=64, out_dtype=P.OUT_F32 if mt == 2 else P.OUT_BF16, relu=True,
                halo=lo, halo_hi=hi, MT=mt, row_bytes=32)
        ol.ops[-1].i["max_ctas"] = max_ctas
        ol.commit()
        G.named(ol, "a").copy_(_fill(ol, "a", 22))
        return ol
    cpu, gpu, _, _ = G.run_pair(build)
    G.report(f"stem window row32 MT{mt} max_ctas={max_ctas}", G.named(gpu, "o"), G.named(cpu, "o"), atol=2e-2, rtol=1e-2)


@pytest.mark.parametrize("max_ctas", [0, 3])
@pytest.mark.parametrize("B,HW", [(2, 20), (3, 112)])
def test_stem_window_fused_maxpool(B, HW, max_ctas):
    """Stem conv + ReLU + 3x3/2 max-pool in one kernel: a tile is 3 conv rows of one image (strided M tiling,
    MT=3), pooled in shared memory into one row of the pooled padded grid."""
    g0, g1 = P.Grid(B, HW, HW, pad=2), P.Grid(B, HW // 2, HW // 2)
    def build(device):
        W = _weights(device, "w", 64, 256, torch.bfloat16, 31).finalize()
        ol = P.OpList(W, device)
        a = ol._buf("a", torch.bfloat16, g0.rows, 16)
        o = ol._buf("o", torch.bfloat16, g1.rows, 64)
        lo, hi = 2 * g0.P + 2, g0.P + 1
        rels = [lo + (ia - 2) * g0.P + (ib - 2) for ia in range(4) for ib in range(4)]
        ol.gemm("stem", dtype=P.DT_BF16, M=g0.rows, N=64, a0=a, a0_shape=(g0.rows, 16, 16), groups=[(0, 0, 0, 1, rels)],
                w="w.w", bias="w.b", out=o, ldo=64, out_dtype=P.OUT_BF16, relu=True, grid=g0,
                halo=lo, halo_hi=hi, MT=3, row_bytes=32, pool_to=g1)
        ol.ops[-1].i["max_ctas"] = max_ctas
        ol.commit()
        G.named(ol, "a").copy_(_fill(ol, "a", 32))
        G.named(ol, "o").fill_(7.0)      # pad rows/columns must be overwritten with zeros
        return ol
    cpu, gpu, _, _ = G.run_pair(build)
    G.report(f"stem + fused max-pool B{B} {HW}x{HW} max_ctas={max_ctas}", G.named(gpu, "o"), G.named(cpu, "o"),
             atol=2e-2, rtol=1e-2)


@pytest.mark.parametrize("max_ctas", [0, 3])
@pytest.mark.parametrize("B,HW,run_len", [(2, 20, 5), (2, 20, 1), (3, 112, 14), (1, 112, 2), (2, 56, None)])
def test_stem_two_row_fused_maxpool(B, HW, run_len, max_ctas):
    """stem_pool op: one N = 128 MMA set per conv-row pair (block 1 = the same window one vertical tap lower), vertical
    max carried in registers along runs of pooled rows, horizontal max through shared memory."""
    g0, g1 = P.Grid(B, HW, HW, pad=2), P.Grid(B, HW // 2, HW // 2)
    def build(device):
        g = torch.Generator().manual_seed(41)
        w = torch.randn(64, 256, generator=g) * (1.0 / 147 ** 0.5)
        W = P.Weights(device)
        W.add("w2", P._stem_two_row_matrix(w), torch.bfloat16)
        W.finalize()
        ol = P.OpList(W, device)
        a = ol._buf("a", torch.bfloat16, g0.rows, 16)
        o = ol._buf("o", torch.bfloat16, g1.rows, 64)
        ol.stem_pool("stem", a, g0, "w2", o, g1, run_len=run_len, max_ctas=max_ctas)
        ol.commit()
        G.named(ol, "a").copy_(_fill(ol, "a", 42))
        G.named(ol, "o").fill_(7.0)      # pad rows/columns must be overwritten with zeros
        return ol
    cpu, gpu, _, _ = G.run_pair(build)
    G.report(f"two-row stem + max-pool B{B} {HW}x{HW} run_len={run_len} max_ctas={max_ctas}", G.named(gpu, "o"),
             G.named(cpu, "o"), atol=2e-2, rtol=1e-2)


def _conv_sf_case(device, B, H, Wd, residual, max_ctas, pair):
    """Shift-fused 64 -> 64 3x3 convolution (N = 192 MMAs, horizontal taps added in the epilogue)."""
    g = P.Grid(B, H, Wd)
    gen = torch.Generator().manual_seed(17)
    w4 = torch.randn(64, 64, 3, 3, generator=gen) * (1.0 / 576 ** 0.5)
    W = P.Weights(device)
    W.add("c.wsf", P._ohwi_shift_fused(w4), torch.bfloat16)
    W.add("c.w4", w4.to(torch.bfloat16).float(), torch.float32)     # the same (bf16-rounded) weights for F.conv2d
    W.add("c.b", torch.randn(64, generator=gen), torch.float32)
    W.finalize()
    ol = P.OpList(W, device)
    x = ol._buf("x", torch.bfloat16, g.rows, 64)
    o = ol._buf("o", torch.bfloat16, g.rows, 64)
    groups, halo, halo_hi = ol._conv3x3_sf(g, 1)
    ol.gemm("conv", dtype=P.DT_BF16, M=g.rows, N=64, a0=x, a0_shape=(g.rows, 64, 64), groups=groups, w="c.wsf", bias="c.b",
            out=o, ldo=64, out_dtype=P.OUT_BF16, relu=True, res=x if residual else None,
            res_dtype=P.OUT_BF16 if residual else -1, ldr=64, grid=g, halo=halo, halo_hi=halo_hi, MT=1, sf=3, pair=pair)
    ol.ops[-1].i["max_ctas"] = max_ctas
    ol.commit()
    xv = torch.randn(g.rows, 64, generator=gen)
    r = torch.arange(g.rows) % g.rpi
    xv[~(((r // g.P) < g.H) & ((r % g.P) < g.W))] = 0
    G.named(ol, "x").copy_(xv.to(torch.bfloat16))
    G.named(ol, "o").fill_(3.0)            # every row, pads included, must be written
    return ol


@pytest.mark.parametrize("pair", [False, True])
@pytest.mark.parametrize("max_ctas", [0, 3])
@pytest.mark.parametrize("B,H,W,residual", [(2, 8, 8, False), (1, 56, 56, True), (3, 20, 13, True), (5, 56, 56, False)])
def test_conv3x3_shift_fused(B, H, W, residual, max_ctas, pair):
    """sf = 3: one 192-column MMA per vertical tap; the epilogue adds the three horizontal taps with row shifts
    0 / 1 / 2 (warp shuffles + the exchange between 32-row slabs), tiles advance by 126 rows and the last slab of
    every tile is stored through a 30-row box.  Checked against the emulator and against F.conv2d itself."""
    cpu, gpu, _, _ = G.run_pair(lambda d: _conv_sf_case(d, B, H, W, residual, max_ctas, pair))
    G.report(f"conv sf3 {B}x{H}x{W} res={residual} max_ctas={max_ctas} pair={pair}", G.named(gpu, "o"), G.named(cpu, "o"),
             atol=3e-2, rtol=2e-2)
    g = P.Grid(B, H, W)
    import emulator as E
    idx = E._grid_index(B, H, W, g.P, g.rpi)
    x = G.named(cpu, "x")[idx].float().view(B, H, W, 64).permute(0, 3, 1, 2)
    want = torch.nn.functional.conv2d(x, cpu.W.tensor("c.w4"), cpu.W.tensor("c.b"), padding=1)
    want = torch.relu(want + x if residual else want)
    got = G.named(gpu, "o").cpu()[idx].float().view(B, H, W, 64).permute(0, 3, 1, 2)
    G.report("conv sf3 vs F.conv2d", got, want, atol=3e-2, rtol=2e-2)
    pads = torch.ones(g.rows, dtype=torch.bool)
    pads[idx] = False
    assert G.named(gpu, "o").cpu()[pads].abs().max() == 0   # shared zero padding is rewritten as zeros


@pytest.mark.parametrize("T,F,Nn,max_ctas,cs", [(128, 1024, 0, 0, 0), (300, 1024, 768, 0, 0), (1000, 1024, 256, 3, 1), (700, 256, 768, 2, 2),
                                                (5120, 1024, 768, 0, 0), (1100, 1024, 768, 4, 4), (2000, 512, 256, 0, 1)])
def test_mlp_chain(T, F, Nn, max_ctas, cs):
    """Fused post-attention chain (W_o + residual, LayerNorm, FFN in 128-column hidden chunks, residual, the next block's
    LayerNorm + projection) against the emulator; max_ctas forces several 128-row tiles per CTA (barrier phases, TMEM and
    operand-buffer reuse across tiles), T = 300 / 700 / 1000 a ragged last tile, cs the cluster size that shares the
    multicast weight stream (0 = automatic; phantom tiles pad the last cluster)."""
    D = 256
    def build(device):
        g = torch.Generator().manual_seed(61)
        W = P.Weights(device)
        rnd = lambda *s: torch.randn(*s, generator=g)
        W.add("l.o.w.h", rnd(D, D) / 16, torch.float16)
        W.add("l.fc1.w.h", rnd(F, D) / 16, torch.float16)
        W.add("l.fc1.b", rnd(F) * 0.1, torch.float32)
        W.add("l.fc2.w.h", rnd(D, F) / F ** 0.5, torch.float16)
        W.add("l.fc2.b", rnd(D) * 0.1, torch.float32)
        W.add("l.ln.g", 1 + 0.1 * rnd(D), torch.float32)
        W.add("l.ln.b", 0.1 * rnd(D), torch.float32)
        W.add("n.ln.g", 1 + 0.1 * rnd(D), torch.float32)
        W.add("n.ln.b", 0.1 * rnd(D), torch.float32)
        W.add("n.w.h", rnd(max(Nn, 128), D) / 16, torch.float16)
        W.finalize()
        ol = P.OpList(W, device)
        ctx = ol._buf("ctx", torch.float16, T, D)
        x = ol._buf("x", torch.float32, T, D)
        xo = ol._buf("xo", torch.float32, T, D)
        y = ol._buf("y", torch.float32, T, max(Nn, 4))
        ol.mlp_chain("chain", ctx=ctx, xres=x, xout=xo, T=T, prefix="l", ln="l.ln",
                     nxt=("n.ln", "n.w.h", y, Nn) if Nn else None, max_ctas=max_ctas, cs=cs)
        ol.commit()
        G.named(ol, "ctx").copy_(_fill(ol, "ctx", 62))
        G.named(ol, "x").copy_(_fill(ol, "x", 63, scale=2.0))
        return ol
    cpu, gpu, _, _ = G.run_pair(build)
    G.report(f"chain xout T{T} F{F}", G.named(gpu, "xo"), G.named(cpu, "xo"), atol=4e-3, rtol=2e-3)
    if Nn:
        G.report(f"chain y T{T} Nn{Nn}", G.named(gpu, "y"), G.named(cpu, "y"), atol=6e-3, rtol=4e-3)


@pytest.mark.parametrize("M,N,k", [(256, 1000, 5), (1, 1000, 5), (300, 1000, 8), (130, 136, 1), (1024, 1000, 5), (64, 3128, 3),
                                   (5, 4, 4), (3, 8, 8)])
def test_linear_with_fused_softmax_topk(M, N, k):
    """The answer head's last Linear with softmax + top-k in its epilogue (models/vqa_model.py:336-337,
    api/inference.py:231-234) against the stable rank order (tests/topk_ref.py: NaN > +inf > finite > -inf, ties to the
    lower index) and the fp64 softmax of the SAME logits; rows with -inf, duplicated maxima, all NaN, one NaN and +inf;
    k = N; the launch is repeated so the arrival counters must have been reset by the merging CTA."""
    import gpu_util as G
    from topk_ref import ref_order, ref_softmax
    K = 256
    special = M > 4 and N > 40

    def build(device):
        gen = torch.Generator().manual_seed(11)
        W = P.Weights(device)
        npad = (N + 127) // 128 * 128
        w = torch.zeros(npad, K)
        w[:N] = torch.randn(N, K, generator=gen) * 0.2
        if N > 40:
            w[7] = w[3]                       # two identical logit columns: a tie in every row
            w[N - 1] = w[N - 2]
        bias = torch.zeros(npad)
        bias[:N] = torch.randn(N, generator=gen)
        if N > 40:
            bias[7], bias[N - 1] = bias[3], bias[N - 2]
            bias[11] = float("-inf")          # a column nobody may pick before the finite ones
        if special:
            # +inf weights in columns 13 and 17 meet inputs of one sign per row: -inf there in every row, except
            # row 3, where +inf meets column 13's -inf bias (one NaN), and row 4, which gets +inf in column 17
            w[13, 5] = w[17, 9] = float("inf")
            bias[13] = float("-inf")
        W.add("w.h", w, torch.float16)
        W.add("b", bias, torch.float32)
        W.finalize()
        ol = P.OpList(W, device)
        ol.half_tail, ol.tf32 = True, False
        a = ol._buf("a", torch.float16, M, K)
        ol.linear("head2", a, M, K, "w", "b", P.ExtRef(P.EXT["logits"]), N, ldo=N,
                  topk=(k, P.ExtRef(P.EXT["top_idx"]), P.ExtRef(P.EXT["top_probs"])))
        ol.commit()
        av = torch.randn(M, K, generator=gen)
        if special:
            av[:, [5, 9]] = -(av[:, [5, 9]].abs() + 0.1)
            av[3, 5], av[4, 9] = 1.0, 1.0
        if M > 2:
            av[2] = float("nan")              # an all-NaN row (a fully masked question in the reference)
        G.named(ol, "a").copy_(av.to(torch.float16))
        return ol

    ext = [None, None, None, torch.zeros(M, N), torch.zeros(M, k, dtype=torch.int64), torch.zeros(M, k)]
    cpu, gpu, ext_c, ext_g = G.run_pair(build, ext)
    logits = ext_g[3].cpu()
    G.report("logits", logits, ext_c[3], atol=2e-3, rtol=2e-3) if M <= 2 else None
    rows = [r for r in range(M) if r != 2] if M > 2 else list(range(M))
    got_i, got_p = ext_g[4].cpu(), ext_g[5].cpu()
    if os.environ.get("VQA_DRY"):
        # the emulator's topk of the probabilities promises no order among equal values or NaN: there only the values
        # picked in rows with a finite softmax are compared
        rows = [r for r in rows if not bool(torch.isnan(ref_softmax(logits[r])).any())]
    order = ref_order(logits[rows], k)
    torch.testing.assert_close(torch.gather(logits[rows], 1, got_i[rows]), torch.gather(logits[rows], 1, order),
                               rtol=0, atol=0, equal_nan=True)
    want_p = torch.gather(ref_softmax(logits[rows]), 1, order).float()
    torch.testing.assert_close(got_p[rows], want_p, rtol=2e-5, atol=1e-9, equal_nan=True)
    if os.environ.get("VQA_DRY"):
        return
    assert torch.equal(got_i[rows], order)
    if M > 2:                                 # the NaN row: first k indices, NaN probabilities, no fault
        assert torch.equal(got_i[2], torch.arange(k)) and bool(torch.isnan(got_p[2]).all())
    if special:
        assert int(torch.isnan(logits[3]).sum()) == 1 and bool(torch.isnan(logits[3, 13]))
        assert float(logits[4, 17]) == float("inf") and int(torch.isinf(logits[4]).sum()) == 3   # +inf; -inf at 11, 13
        assert int(got_i[3, 0]) == 13 and int(got_i[4, 0]) == 17
    # replay on the same plan: counters were reset
    from vqa_b200.runtime import Plan
    plan = Plan(gpu.ops, 0)
    ext_g[4].fill_(-1)
    ptrs = [0 if t is None else t.data_ptr() for t in ext_g]
    for _ in range(3):
        plan.run(ptrs, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert torch.equal(ext_g[4].cpu()[rows], order)
