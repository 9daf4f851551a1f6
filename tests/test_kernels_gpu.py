"""Op-level parity of every CUDA kernel (through the C-ABI) against plain torch fp32 math on the
same fp16-rounded inputs.  Tolerances: fp16 output rounding (rel 2^-11) plus fp32 accumulation
order; stated per test."""
import math

import numpy as np
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# spatial-attention kernels under test: 3 (short sequences) and 7 (long sequences), each on every shape
ATTN_IMPLS = [int(v) for v in os.environ.get("VISTA_B200_TEST_ATTN_IMPLS", "3,7").split(",")]


@pytest.fixture(scope="module")
def ops():
    from vista_b200 import lib, ops as _ops
    lib.load()
    return _ops


def dev():
    return torch.device("cuda:0")


def rnd(*shape, seed=0, scale=1.0, dtype=torch.float16):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(dtype).to(dev())


def check(out, ref, rtol=2e-3, atol=2e-3, name=""):
    out = out.float()
    ref = ref.float()
    err = (out - ref).abs()
    tol = atol + rtol * ref.abs()
    bad = (err > tol)
    rel = float((out - ref).norm() / (ref.norm() + 1e-20))
    assert not bool(bad.any()), (f"{name}: {int(bad.sum())}/{bad.numel()} mismatches, max err {float(err.max()):.4g}, "
                                 f"rel-L2 {rel:.3g}, first bad idx {bad.nonzero()[:4].tolist()}")
    return rel


# ------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,K,N,tile_n", [(128, 64, 64, 64), (300, 128, 96, 96), (1000, 320, 320, 160),
                                          (4096, 1280, 640, 256), (7200, 2560, 1280, 256), (50, 768, 1280, 256)])
def test_gemm_linear_plain(ops, M, K, N, tile_n):
    a, w = rnd(M, K, seed=1), rnd(N, K, seed=2, scale=K ** -0.5)
    out = torch.empty(M, N, dtype=torch.float16, device=dev())
    ops.gemm(a, w, out, tile_n=tile_n)
    torch.cuda.synchronize()
    check(out, a.float() @ w.float().t(), name=f"gemm {M}x{K}x{N}")


def test_gemm_epilogue_full(ops):
    M, K, N = 2 * 25 * 24, 320, 640      # 2 clips x 25 frames x 24 tokens
    a, w = rnd(M, K, seed=3), rnd(N, K, seed=4, scale=K ** -0.5)
    bias = rnd(N, seed=5, dtype=torch.float32)
    rowvec = rnd(25, N, seed=6, dtype=torch.float32)          # indexed by frame-in-clip
    res1, res2 = rnd(M, N, seed=7), rnd(M, N, seed=8)
    out = torch.empty(M, N, dtype=torch.float16, device=dev())
    ops.gemm(a, w, out, bias=bias, rowvec=rowvec, rv_div=24, rv_mod=25, res1=res1, s_res1=0.25, res2=res2, s_res2=0.75,
             s_acc=0.6, act=0)
    torch.cuda.synchronize()
    frame = (torch.arange(M, device=dev()) // 24) % 25
    ref = 0.6 * (a.float() @ w.float().t() + bias) + rowvec[frame] + 0.25 * res1.float() + 0.75 * res2.float()
    check(out, ref, name="gemm epilogue")


def test_gemm_silu_f32_out_and_strided(ops):
    M, K, N = 50, 320, 1280
    abuf = rnd(M, K + 64, seed=9)
    a = abuf[:, 64:]                                      # strided A view (lda = K + 64)
    w = rnd(N, K, seed=10, scale=K ** -0.5)
    bias = rnd(N, seed=11, dtype=torch.float32)
    obuf = torch.zeros(M, N + 8, dtype=torch.float32, device=dev())
    ops.gemm(a, w, obuf[:, 8:], bias=bias, act=1)
    torch.cuda.synchronize()
    check(obuf[:, 8:], F.silu(a.float() @ w.float().t() + bias), name="gemm silu f32")
    assert float(obuf[:, :8].abs().max()) == 0.0


def test_gemm_geglu(ops):
    from vista_b200.weights import permute_geglu
    M, Cc = 900, 320
    a = rnd(M, Cc, seed=12)
    w = rnd(8 * Cc, Cc, seed=13, scale=Cc ** -0.5)
    b = rnd(8 * Cc, seed=14, dtype=torch.float32)
    tile_n = 256
    wp, bp = permute_geglu(w, b, tile_n)
    out = torch.empty(M, 4 * Cc, dtype=torch.float16, device=dev())
    ops.gemm(a, wp, out, bias=bp, act=2, tile_n=tile_n)
    torch.cuda.synchronize()
    val, gate = (a.float() @ w.float().t() + b).chunk(2, dim=-1)
    check(out, val * F.gelu(gate), name="geglu")


@pytest.mark.parametrize("NB,H,W,Cin,Cout", [(3, 8, 16, 64, 64), (4, 9, 16, 128, 96), (2, 18, 32, 192, 128),
                                             (2, 36, 64, 320, 320), (1, 72, 128, 64, 160)])
def test_gemm_conv3x3(ops, NB, H, W, Cin, Cout):
    x = rnd(NB, H, W, Cin, seed=15)                       # NHWC
    wt = rnd(Cout, Cin, 3, 3, seed=16, scale=(9 * Cin) ** -0.5)
    bias = rnd(Cout, seed=17, dtype=torch.float32)
    emb = rnd(NB, Cout, seed=18, dtype=torch.float32)     # per-frame vector (emb_out)
    w2 = wt.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous()   # tap-major K
    out = torch.empty(NB * H * W, Cout, dtype=torch.float16, device=dev())
    ops.gemm(x.reshape(-1, Cin), w2, out, taps=ops.TAPS_3X3, geom=(W, H, NB), bias=bias, rowvec=emb, rv_div=H * W,
             rv_mod=NB)
    torch.cuda.synchronize()
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, padding=1) + emb[:, :, None, None]
    check(out.reshape(NB, H, W, Cout), ref.permute(0, 2, 3, 1), name="conv3x3")


@pytest.mark.parametrize("kind,NB,H,W,Cin,Cout,fps", [("conv_rv", 4, 8, 128, 64, 320, 1), ("conv_res", 4, 36, 64, 128, 640, 1),
                                                      ("lin_res", 3, 4, 128, 320, 320, 1), ("tconv_res", 2, 1, 256, 128, 128, 5),
                                                      ("conv_plain", 2, 16, 256, 64, 128, 2)])
def test_gemm_fused_groupnorm_statistics(ops, kind, NB, H, W, Cin, Cout, fps):
    """The STATS epilogue: column partials of the stored output -> b200v_groupnorm_from_partials must give the (mean, rstd)
    torch computes on the same output tensor, for every epilogue variant that has a fused-statistics instantiation,
    per-frame and clip-wide (frames_per_stat) statistics, and a partial matrix shared by two producers (column slices)."""
    tokens = NB * H * W
    frames = NB if kind != "tconv_res" else NB * fps
    tpf = tokens // frames if kind != "tconv_res" else W
    x = rnd(tokens if kind != "tconv_res" else frames * tpf, Cin, seed=61)
    tokens = x.shape[0]
    bias = rnd(Cout, seed=63, dtype=torch.float32)
    res = rnd(tokens, Cout, seed=64)
    out = torch.empty(tokens, 2 * Cout, dtype=torch.float16, device=dev())[:, Cout:]     # a column slice (skip-concat)
    part_full = torch.zeros(tokens // 128 * 4, 2 * Cout, 2, dtype=torch.float32, device=dev())
    part = part_full[:, Cout:]
    if kind in ("conv_rv", "conv_res", "conv_plain"):
        w2 = rnd(Cout, 9 * Cin, seed=62, scale=(9 * Cin) ** -0.5)
        kw = dict(taps=ops.TAPS_3X3, geom=(W, H, NB))
        if kind == "conv_rv":
            kw.update(rowvec=rnd(NB, Cout, seed=65, dtype=torch.float32), rv_div=H * W, rv_mod=NB)
        elif kind == "conv_res":
            kw.update(res1=res)
    elif kind == "lin_res":
        w2 = rnd(Cout, Cin, seed=62, scale=Cin ** -0.5)
        kw = dict(res1=res)
    else:
        w2 = rnd(Cout, 3 * Cin, seed=62, scale=(3 * Cin) ** -0.5)
        kw = dict(taps=ops.TAPS_T3, geom=(tpf, fps, NB), res1=res, s_acc=0.4)
    ops.gemm(x, w2, out, bias=bias, stats=part, **kw)
    ref_out = torch.empty(tokens, Cout, dtype=torch.float16, device=dev())
    ops.gemm(x, w2, ref_out, bias=bias, **kw)                                          # same launch without statistics
    st = torch.zeros(frames // fps, 32, 2, dtype=torch.float32, device=dev())
    ops.groupnorm_from_partials(part, frames, tpf, Cout, 1e-5, st, frames_per_stat=fps)
    torch.cuda.synchronize()
    assert torch.equal(out, ref_out)
    o = out.float().reshape(frames // fps, fps * tpf, 32, Cout // 32)
    mean = o.mean(dim=(1, 3))
    rstd = torch.rsqrt(o.var(dim=(1, 3), unbiased=False) + 1e-5)
    # the partials hold the fp32 values BEFORE the fp16 rounding of the store: agreement to fp16-rounding noise / sqrt(n)
    assert float((st[..., 0] - mean).abs().max()) < 2e-4 * float(o.abs().max())
    assert float((st[..., 1] / rstd - 1).abs().max()) < 2e-4
    assert float(part_full[:, :Cout].abs().max()) == 0.0                                # the other producer's columns untouched


def test_gemm_conv3x3_thin_output_f32(ops):
    """out[2] / decoder conv_out path: Cout padded to 8, fp32 output, tile_n 32."""
    NB, H, W, Cin = 2, 9, 16, 320
    x = rnd(NB, H, W, Cin, seed=51)
    wt = torch.zeros(8, Cin, 3, 3, dtype=torch.float16, device=dev())
    wt[:4] = rnd(4, Cin, 3, 3, seed=52, scale=(9 * Cin) ** -0.5)
    bias = torch.zeros(8, device=dev())
    bias[:4] = rnd(4, seed=53, dtype=torch.float32)
    out = torch.full((NB * H * W, 8), 7.0, dtype=torch.float32, device=dev())
    ops.gemm(x.reshape(-1, Cin), wt.permute(0, 2, 3, 1).reshape(8, 9 * Cin).contiguous(), out, taps=ops.TAPS_3X3,
             geom=(W, H, NB), bias=bias, tile_n=32)
    torch.cuda.synchronize()
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, padding=1).permute(0, 2, 3, 1)
    check(out.reshape(NB, H, W, 8), ref, rtol=1e-3, atol=1e-3, name="thin conv")


@pytest.mark.parametrize("nb,T,S,Cc", [(2, 25, 128, 64), (2, 25, 144, 128), (1, 14, 512, 64)])
def test_gemm_temporal_conv(ops, nb, T, S, Cc):
    x = rnd(nb, T, S, Cc, seed=19)                        # tokens (b t) s
    wt = rnd(Cc, Cc, 3, 1, 1, seed=20, scale=(3 * Cc) ** -0.5)
    bias = rnd(Cc, seed=21, dtype=torch.float32)
    res = rnd(nb * T * S, Cc, seed=22)
    w2 = wt[:, :, :, 0, 0].permute(0, 2, 1).reshape(Cc, 3 * Cc).contiguous()
    out = torch.empty(nb * T * S, Cc, dtype=torch.float16, device=dev())
    ops.gemm(x.reshape(-1, Cc), w2, out, taps=ops.TAPS_T3, geom=(S, T, nb), bias=bias, res1=res, s_res1=1.0, s_acc=0.4)
    torch.cuda.synchronize()
    x5 = x.float().permute(0, 3, 1, 2)[..., None]         # b c t s 1
    ref = F.conv3d(x5, wt.float(), bias, padding=(1, 0, 0))[..., 0].permute(0, 2, 3, 1).reshape(-1, Cc)
    check(out, 0.4 * ref + res.float(), name="tconv")


@pytest.mark.parametrize("nb,T,S,Cc", [(1, 7, 128, 64), (1, 6, 144, 128), (2, 5, 256, 64)])
def test_gemm_temporal_conv_with_halo_frames(ops, nb, T, S, Cc):
    """h_pad = 1: the (3,1,1) convolution of a frame shard reads its neighbours' boundary frames from the halo slots of the
    extended tensor [prev | T local | next] in ONE launch — equal to the same frames cut out of the convolution of the
    longer clip (and to zero padding where a halo slot holds zeros: the clip ends)."""
    full = rnd(nb, T + 2, S, Cc, seed=33)                 # the T local frames with one real neighbour frame on each side
    wt = rnd(Cc, Cc, 3, 1, 1, seed=34, scale=(3 * Cc) ** -0.5)
    bias = rnd(Cc, seed=35, dtype=torch.float32)
    w2 = wt[:, :, :, 0, 0].permute(0, 2, 1).reshape(Cc, 3 * Cc).contiguous()
    out = torch.empty(nb * T * S, Cc, dtype=torch.float16, device=dev())
    stats = torch.zeros(-(-nb * T * S // 128) * 4, Cc, 2, dtype=torch.float32, device=dev()) if S % 128 == 0 else None
    ops.gemm(full.reshape(-1, Cc), w2, out, taps=ops.TAPS_T3, geom=(S, T, nb), bias=bias, h_pad=1, stats=stats)
    torch.cuda.synchronize()
    x5 = full.float().permute(0, 3, 1, 2)[..., None]      # b c (T+2) s 1
    ref = F.conv3d(x5, wt.float(), bias, padding=(1, 0, 0))[..., 0][:, :, 1:T + 1].permute(0, 2, 3, 1).reshape(-1, Cc)
    check(out, ref, name="tconv+halo")
    if stats is not None:                                  # fused statistics see the halo contributions
        got = stats[..., 0].sum(0)
        assert torch.allclose(got, out.float().sum(0), rtol=2e-3, atol=2e-2)
    # zero halos == zero padding of the plain launch
    full[:, 0] = 0
    full[:, T + 1] = 0
    out2 = torch.empty_like(out)
    ops.gemm(full.reshape(-1, Cc), w2, out, taps=ops.TAPS_T3, geom=(S, T, nb), bias=bias, h_pad=1)
    ops.gemm(full[:, 1:T + 1].reshape(-1, Cc), w2, out2, taps=ops.TAPS_T3, geom=(S, T, nb), bias=bias)
    torch.cuda.synchronize()
    assert torch.equal(out, out2)


# ------------------------------------------------------------------------------------------ attention
@pytest.mark.parametrize("impl", ATTN_IMPLS)
@pytest.mark.parametrize("frames,seq,heads", [(2, 128, 1), (3, 144, 2), (2, 576, 4), (1, 2304, 2), (2, 200, 1), (1, 256, 1),
                                              (2, 300, 1),
                                              # more work items than SMs (persistent loop of v5: 200 / 200 items), with and
                                              # without a skipped second query tile in the last block of a (frame, head)
                                              (10, 1280, 4), (20, 320, 5),
                                              # level 0 of the full-size network (72 x 128 tokens) and the inner levels
                                              # of the tiny / small networks (sequences below one 128-row tile)
                                              (2, 9216, 5), (2, 32, 2), (3, 8, 1)])
def test_attention_spatial(ops, frames, seq, heads, impl):
    Cc = heads * 64
    qkv = rnd(frames * seq, 3 * Cc, seed=23)
    out = torch.zeros(frames * seq, Cc, dtype=torch.float16, device=dev())
    ops.attention_spatial(qkv[:, :Cc], qkv[:, Cc:2 * Cc], qkv[:, 2 * Cc:], out, frames, seq, heads, impl=impl)
    torch.cuda.synchronize()
    q, k, v = (t.float().reshape(frames, seq, heads, 64).permute(0, 2, 1, 3) for t in qkv.chunk(3, dim=-1))
    if seq <= 4096:
        ref = F.scaled_dot_product_attention(q, k, v).permute(0, 2, 1, 3).reshape(frames * seq, Cc)
        check(out, ref, rtol=4e-3, atol=2e-3, name="attn spatial")
        return
    # long sequences: fp64 reference of a fixed random subset of 512 query rows (the same rows in every frame and head)
    rows = torch.randperm(seq, generator=torch.Generator().manual_seed(5))[:512].to(dev())
    ref = F.scaled_dot_product_attention(q[:, :, rows].double(), k.double(), v.double())     # frames, heads, 512, 64
    got = out.reshape(frames, seq, heads, 64)[:, rows].permute(0, 2, 1, 3)
    check(got, ref, rtol=4e-3, atol=2e-3, name="attn spatial (row subset)")


@pytest.mark.parametrize("impl", ATTN_IMPLS)
def test_attention_spatial_strided_out(ops, impl):
    """out is a column slice of a wider buffer (ld_o > C); the columns around it stay untouched."""
    frames, seq, heads = 2, 300, 2
    Cc = heads * 64
    qkv = rnd(frames * seq, 3 * Cc, seed=27)
    obuf = torch.full((frames * seq, Cc + 64), 7.0, dtype=torch.float16, device=dev())
    ops.attention_spatial(qkv[:, :Cc], qkv[:, Cc:2 * Cc], qkv[:, 2 * Cc:], obuf[:, 32:32 + Cc], frames, seq, heads, impl=impl)
    torch.cuda.synchronize()
    q, k, v = (t.double().reshape(frames, seq, heads, 64).permute(0, 2, 1, 3) for t in qkv.chunk(3, dim=-1))
    ref = F.scaled_dot_product_attention(q, k, v).permute(0, 2, 1, 3).reshape(frames * seq, Cc)
    check(obuf[:, 32:32 + Cc], ref, rtol=4e-3, atol=2e-3, name="attn spatial strided out")
    assert bool((obuf[:, :32] == 7.0).all()) and bool((obuf[:, 32 + Cc:] == 7.0).all())


@pytest.mark.parametrize("impl", ATTN_IMPLS)
def test_attention_spatial_peaky(ops, impl):
    """Large logits: the running max / (lazy) rescale path must hold (scores ~ +-40)."""
    frames, seq, heads = 1, 640, 1
    qkv = rnd(frames * seq, 192, seed=24, scale=2.5)
    out = torch.zeros(frames * seq, 64, dtype=torch.float16, device=dev())
    ops.attention_spatial(qkv[:, :64], qkv[:, 64:128], qkv[:, 128:], out, frames, seq, heads, impl=impl)
    torch.cuda.synchronize()
    q, k, v = (t.float().reshape(1, seq, 1, 64).permute(0, 2, 1, 3) for t in qkv.chunk(3, dim=-1))
    ref = F.scaled_dot_product_attention(q, k, v).permute(0, 2, 1, 3).reshape(seq, 64)
    check(out, ref, rtol=1e-2, atol=1e-2, name="attn peaky")


@pytest.mark.parametrize("impl", [i for i in ATTN_IMPLS if i >= 2])
def test_attention_spatial_increasing_max(ops, impl):
    """Keys ordered so that the row maximum keeps growing block after block: exercises every lazy-rescale branch."""
    seq = 1024
    g = torch.Generator().manual_seed(3)
    q = torch.randn(seq, 64, generator=g)
    k = torch.randn(seq, 64, generator=g) * torch.linspace(0.2, 6.0, seq)[:, None]
    v = torch.randn(seq, 64, generator=g)
    qkv = torch.cat([q, k, v], 1).half().to(dev())
    out = torch.zeros(seq, 64, dtype=torch.float16, device=dev())
    ops.attention_spatial(qkv[:, :64], qkv[:, 64:128], qkv[:, 128:], out, 1, seq, 1, impl=impl)
    torch.cuda.synchronize()
    qq, kk, vv = (t.float().reshape(1, seq, 1, 64).permute(0, 2, 1, 3) for t in qkv.chunk(3, dim=-1))
    ref = F.scaled_dot_product_attention(qq, kk, vv).permute(0, 2, 1, 3).reshape(seq, 64)
    check(out, ref, rtol=1e-2, atol=1e-2, name="attn increasing max")


@pytest.mark.parametrize("nb,T,S,heads", [(2, 25, 32, 1), (2, 25, 20, 5), (1, 14, 16, 2), (2, 25, 8, 20),
                                          # 23040 (clip, pixel, head) items: every warp walks several (the Q tile of
                                          # each holds the previous item's O in its padding rows)
                                          (2, 25, 2304, 5),
                                          (1, 32, 64, 2), (2, 1, 40, 1), (1, 17, 96, 3)])  # no key padding, one frame, odd T
def test_attention_temporal(ops, nb, T, S, heads):
    Cc = heads * 64
    qkv = rnd(nb * T * S, 3 * Cc, seed=25)
    out = torch.zeros(nb * T * S, Cc, dtype=torch.float16, device=dev())
    ops.attention_temporal(qkv[:, :Cc], qkv[:, Cc:2 * Cc], qkv[:, 2 * Cc:], out, nb, T, S, heads)
    torch.cuda.synchronize()
    q, k, v = (t.float().reshape(nb, T, S, heads, 64).permute(0, 2, 3, 1, 4) for t in qkv.chunk(3, dim=-1))
    ref = F.scaled_dot_product_attention(q, k, v)          # (nb, S, heads, T, 64)
    ref = ref.permute(0, 3, 1, 2, 4).reshape(nb * T * S, Cc)
    check(out, ref, name="attn temporal")


def test_attention_temporal_peaky_strided_out(ops):
    """Large logits (inputs x 2.5) and out as a column slice of a wider buffer."""
    nb, T, S, heads = 2, 25, 40, 2
    Cc = heads * 64
    qkv = rnd(nb * T * S, 3 * Cc, seed=26, scale=2.5)
    obuf = torch.full((nb * T * S, Cc + 64), 7.0, dtype=torch.float16, device=dev())
    ops.attention_temporal(qkv[:, :Cc], qkv[:, Cc:2 * Cc], qkv[:, 2 * Cc:], obuf[:, 64:], nb, T, S, heads)
    torch.cuda.synchronize()
    q, k, v = (t.double().reshape(nb, T, S, heads, 64).permute(0, 2, 3, 1, 4) for t in qkv.chunk(3, dim=-1))
    ref = F.scaled_dot_product_attention(q, k, v).permute(0, 3, 1, 2, 4).reshape(nb * T * S, Cc)
    # P is rounded to fp16 before P V; with peaked rows and |v| ~ 2.5 that costs more than the 2e-3 of the plain test
    check(obuf[:, 64:], ref, rtol=1e-2, atol=1e-2, name="attn temporal peaky")
    assert bool((obuf[:, :64] == 7.0).all())


# ------------------------------------------------------------------------------------------ norms
@pytest.mark.parametrize("frames,tpf,Cc,fps", [(4, 128, 64, 1), (6, 300, 320, 1), (50, 144, 2560, 25), (4, 100, 960, 2),
                                               (2, 2304, 1920, 1)])
@pytest.mark.parametrize("silu", [False, True])
def test_groupnorm(ops, frames, tpf, Cc, fps, silu):
    x = rnd(frames * tpf, Cc, seed=26, scale=2.0) + 0.7
    gamma = rnd(Cc, seed=27, dtype=torch.float32) * 0.1 + 1
    beta = rnd(Cc, seed=28, dtype=torch.float32) * 0.1
    y = torch.empty_like(x)
    ops.groupnorm(x, y, frames, tpf, gamma, beta, 1e-5, silu, frames_per_stat=fps)
    y1 = y.clone()
    ops.groupnorm(x, y, frames, tpf, gamma, beta, 1e-5, silu, frames_per_stat=fps)
    torch.cuda.synchronize()
    assert torch.equal(y, y1), "GroupNorm must be bit-reproducible"
    xr = x.float().reshape(frames // fps, fps * tpf, Cc).permute(0, 2, 1)     # (stat, C, L)
    ref = F.group_norm(xr, 32, gamma, beta, 1e-5)
    if silu:
        ref = F.silu(ref)
    check(y, ref.permute(0, 2, 1).reshape(frames * tpf, Cc), name="groupnorm")


@pytest.mark.parametrize("tokens,Cc", [(100, 64), (1000, 320), (333, 1280), (77, 2560), (517, 640)])
def test_layernorm(ops, tokens, Cc):
    x = rnd(tokens, Cc, seed=29, scale=1.5) - 0.3
    gamma = rnd(Cc, seed=30, dtype=torch.float32) * 0.1 + 1
    beta = rnd(Cc, seed=31, dtype=torch.float32) * 0.1
    add = rnd(5, Cc, seed=32, dtype=torch.float32)
    y = torch.empty_like(x)
    ops.layernorm(x, y, gamma, beta, 1e-5)
    torch.cuda.synchronize()
    check(y, F.layer_norm(x.float(), (Cc,), gamma, beta, 1e-5), name="layernorm")
    ops.layernorm(x, y, gamma, beta, 1e-5, addvec=add, av_div=7, av_mod=5)
    torch.cuda.synchronize()
    idx = (torch.arange(tokens, device=dev()) // 7) % 5
    check(y, F.layer_norm(x.float() + add[idx], (Cc,), gamma, beta, 1e-5), name="layernorm+add")


@pytest.mark.parametrize("Cc", [96, 320, 640, 1280])
def test_layernorm_strided(ops, Cc):
    """x and y are column slices of wider buffers (ldx, ldy > C); y's neighbouring columns stay untouched."""
    tokens = 389
    xbuf = rnd(tokens, Cc + 40, seed=29, scale=1.5)
    x = xbuf[:, 24:24 + Cc]
    gamma = rnd(Cc, seed=30, dtype=torch.float32) * 0.1 + 1
    beta = rnd(Cc, seed=31, dtype=torch.float32) * 0.1
    ybuf = torch.full((tokens, Cc + 16), 7.0, dtype=torch.float16, device=dev())
    ops.layernorm(x, ybuf[:, 8:8 + Cc], gamma, beta, 1e-5)
    torch.cuda.synchronize()
    check(ybuf[:, 8:8 + Cc], F.layer_norm(x.double(), (Cc,), gamma.double(), beta.double(), 1e-5), name="layernorm strided")
    assert bool((ybuf[:, :8] == 7.0).all()) and bool((ybuf[:, 8 + Cc:] == 7.0).all())


# ------------------------------------------------------------------------------------------ small ops
@pytest.mark.parametrize("cin,cout", [(8, 320), (4, 64), (8, 100)])
def test_conv3x3_small_cin(ops, cin, cout):
    NB, H, W = 3, 9, 16
    x = rnd(NB, H, W, 8, seed=33)
    wt = rnd(cout, cin, 3, 3, seed=34, dtype=torch.float32, scale=0.2)
    bias = rnd(cout, seed=35, dtype=torch.float32)
    out = torch.empty(NB * H * W, cout, dtype=torch.float16, device=dev())
    ops.conv3x3_small_cin(x.reshape(-1, 8), cin, wt, bias, out, NB, H, W)
    torch.cuda.synchronize()
    ref = F.conv2d(x.float()[..., :cin].permute(0, 3, 1, 2), wt, bias, padding=1).permute(0, 2, 3, 1)
    check(out.reshape(NB, H, W, cout), ref, name="conv small cin")


@pytest.mark.parametrize("cin,cout", [(320, 4), (128, 3), (64, 4)])
def test_conv3x3_small_cout(ops, cin, cout):
    NB, H, W = 2, 9, 16
    x = rnd(NB, H, W, cin, seed=36)
    wt = rnd(cout, cin, 3, 3, seed=37, dtype=torch.float32, scale=(9 * cin) ** -0.5)
    bias = rnd(cout, seed=38, dtype=torch.float32)
    out = torch.empty(NB * H * W, cout, dtype=torch.float32, device=dev())
    ops.conv3x3_small_cout(x.reshape(-1, cin), wt, bias, out, NB, H, W)
    torch.cuda.synchronize()
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.half().float(), bias, padding=1).permute(0, 2, 3, 1)
    check(out.reshape(NB, H, W, cout), ref, rtol=1e-3, atol=1e-3, name="conv small cout")


def test_downsample_via_im2col(ops):
    NB, H, W, Cc = 2, 18, 32, 64
    x = rnd(NB, H, W, Cc, seed=39)
    wt = rnd(Cc, Cc, 3, 3, seed=40, scale=(9 * Cc) ** -0.5)
    bias = rnd(Cc, seed=41, dtype=torch.float32)
    Ho, Wo = 9, 16
    col = torch.empty(NB * Ho * Wo, 9 * Cc, dtype=torch.float16, device=dev())
    ops.im2col_s2(x.reshape(-1, Cc), col, NB, H, W, Cc)
    out = torch.empty(NB * Ho * Wo, Cc, dtype=torch.float16, device=dev())
    ops.gemm(col, wt.permute(0, 2, 3, 1).reshape(Cc, 9 * Cc).contiguous(), out, bias=bias)
    torch.cuda.synchronize()
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, stride=2, padding=1).permute(0, 2, 3, 1)
    check(out.reshape(NB, Ho, Wo, Cc), ref, name="downsample")


@pytest.mark.parametrize("NB,H,W", [(2, 16, 24), (1, 17, 23), (3, 9, 14)])
def test_downsample_asym_via_im2col(ops, NB, H, W):
    """VAE-encoder Downsample: zero pad right / bottom by one, 3x3 stride 2 (even and odd H, W)."""
    Cc = 64
    xbuf = rnd(NB * H * W, Cc + 16, seed=54)
    x = xbuf[:, 16:]                                      # strided input rows
    wt = rnd(Cc, Cc, 3, 3, seed=55, scale=(9 * Cc) ** -0.5)
    bias = rnd(Cc, seed=56, dtype=torch.float32)
    Ho, Wo = (H - 2) // 2 + 1, (W - 2) // 2 + 1
    col = torch.empty(NB * Ho * Wo, 9 * Cc, dtype=torch.float16, device=dev())
    ops.im2col_s2_asym(x, col, NB, H, W, Cc)
    out = torch.empty(NB * Ho * Wo, Cc, dtype=torch.float16, device=dev())
    ops.gemm(col, wt.permute(0, 2, 3, 1).reshape(Cc, 9 * Cc).contiguous(), out, bias=bias)
    torch.cuda.synchronize()
    x4 = x.double().reshape(NB, H, W, Cc).permute(0, 3, 1, 2)
    ref = F.conv2d(F.pad(x4, (0, 1, 0, 1)), wt.double(), bias.double(), stride=2).permute(0, 2, 3, 1)
    check(out.reshape(NB, Ho, Wo, Cc), ref, name="downsample asym")


@pytest.mark.parametrize("cols,ld_in", [(128, 128), (1152, 1152), (9216, 9216), (1152, 1200)])
def test_softmax_rows(ops, cols, ld_in):
    """Random rows, a row with one dominant score and rows of large negative scores, against fp64 softmax in fp16."""
    rows = 37
    g = torch.Generator().manual_seed(57)
    x = torch.randn(rows, ld_in, generator=g) * 3
    x[1, :] = torch.randn(ld_in, generator=g)
    x[1, cols // 3] = 60.0                               # one dominant score
    x[2, :] = -1e4 + torch.randn(ld_in, generator=g)      # large negative scores
    x[3, :] = -80.0 + 0.5 * torch.randn(ld_in, generator=g)
    x = x.to(dev())
    y = torch.full((rows, cols + 8), 7.0, dtype=torch.float16, device=dev())
    ops.softmax_rows(x[:, :cols], y[:, :cols])
    torch.cuda.synchronize()
    ref = torch.softmax(x[:, :cols].double(), dim=-1).half()
    check(y[:, :cols], ref, rtol=2e-3, atol=1e-5, name="softmax rows")
    assert bool((y[:, cols:] == 7.0).all())


def test_time_mix_small_skip_frames(ops):
    """The decoder's 3 -> 3 channel (3,1,1) convolution with skipped leading frames, an output frame offset, strided
    input rows and the chunk-overlap blend, against fp64 conv3d and fake_ops.time_mix_small."""
    import fake_ops
    T, h, w, Cc, skip, f0 = 6, 5, 7, 3, 2, 3
    HW = h * w
    xbuf = rnd(T * HW, 8, seed=58, dtype=torch.float32)
    x = xbuf[:, :Cc]                                      # ldx = 8
    wt = rnd(Cc, Cc, 3, seed=59, dtype=torch.float32, scale=0.5)
    bias = rnd(Cc, seed=60, dtype=torch.float32)
    blend = torch.tensor([0, 0, 0, 1, 0, 1], dtype=torch.int32, device=dev())
    out0 = rnd(f0 + T + 1, Cc, h, w, seed=61, dtype=torch.float32)
    out = out0.clone()
    ops.time_mix_small(x, wt, bias, out, blend, T, HW, Cc, out_frame0=f0, skip_frames=skip)
    torch.cuda.synchronize()
    x5 = x.double().reshape(T, h, w, Cc).permute(3, 0, 1, 2)[None]               # 1, C, T, h, w
    conv = F.conv3d(x5, wt.double()[:, :, :, None, None], bias.double(), padding=(1, 0, 0))[0].permute(1, 0, 2, 3)
    ref = out0.double().clone()
    for t in range(skip, T):
        ref[f0 + t] = 0.5 * (out0[f0 + t].double() + conv[t]) if int(blend[t]) else conv[t]
    check(out, ref, rtol=1e-5, atol=1e-5, name="time_mix_small")
    fake = out0.cpu().clone()
    fake_ops.time_mix_small(x.cpu(), wt.cpu(), bias.cpu(), fake, blend.cpu(), T, HW, Cc, f0, skip)
    check(out, fake.to(dev()), rtol=1e-5, atol=1e-5, name="time_mix_small vs fake_ops")


def test_upsample2x(ops):
    NB, H, W, Cc = 2, 5, 7, 64
    x = rnd(NB, H, W, Cc, seed=42)
    out = torch.empty(NB * 4 * H * W, Cc, dtype=torch.float16, device=dev())
    ops.upsample2x(x.reshape(-1, Cc), out, NB, H, W, Cc)
    torch.cuda.synchronize()
    ref = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2, mode="nearest").permute(0, 2, 3, 1)
    assert torch.equal(out.reshape(NB, 2 * H, 2 * W, Cc).float(), ref)


def test_timestep_embedding_and_blend(ops):
    from oracle import vista_oracle as vo
    t = torch.tensor([0.25 * math.log(700.0), -1.5, 0.0, 0.25 * math.log(0.002)], device=dev())
    out = torch.empty(4, 320, dtype=torch.float16, device=dev())
    ops.timestep_embedding(t, out, 320)
    torch.cuda.synchronize()
    check(out, vo.timestep_embedding(t.cpu(), 320).to(dev()), rtol=1e-3, atol=1e-3, name="temb")
    e0, e1, lab = (rnd(4, 96, seed=s, dtype=torch.float32) for s in (43, 44, 45))
    mask = torch.tensor([1.0, 0.0, 0.0, 1.0], device=dev())
    emb = torch.empty(4, 96, device=dev())
    semb = torch.empty(4, 96, dtype=torch.float16, device=dev())
    ops.blend_emb(e0, e1, lab, mask, emb, semb)
    torch.cuda.synchronize()
    ref = e1 * mask[:, None] + e0 * (1 - mask[:, None]) + lab
    check(emb, ref, rtol=1e-6, atol=1e-6, name="blend emb")
    check(semb, F.silu(ref), name="silu emb")


def test_layout_converters(ops):
    NB, Cc, H, W = 3, 4, 5, 6
    x = rnd(NB, Cc, H, W, seed=46, dtype=torch.float32)
    tok = torch.zeros(NB * H * W, 8, dtype=torch.float16, device=dev())
    ops.nchw_to_tokens(x, tok, NB, Cc, H, W)
    back = torch.empty_like(x)
    ops.tokens_to_nchw(tok, back, NB, Cc, H, W)
    torch.cuda.synchronize()
    assert torch.equal(back, x.half().float())
    assert torch.equal(tok[:, :4].reshape(NB, H, W, Cc).float(), x.half().float().permute(0, 2, 3, 1))


def test_sampler_step_kernels(ops):
    """prepare + update around a fake network output == the reference algebra
    (sampling.py:105-106, guiders.py:23-36, denoiser.py:33-35, sampling.py:85-88)."""
    from oracle import vista_oracle as vo
    T, h, w, steps = 5, 4, 6, 3
    x0 = rnd(T, 4, h, w, seed=47, dtype=torch.float32) * 700
    z = rnd(T, 4, h, w, seed=48, dtype=torch.float32)
    concat = rnd(T, 4, h, w, seed=49, dtype=torch.float32) * 5
    mask = torch.tensor([1.0, 0, 0, 1.0, 0], device=dev())
    scales = torch.linspace(1.0, 2.5, T, device=dev())
    sig = vo.edm_sigmas(steps).to(dev())
    step = torch.zeros(1, dtype=torch.int32, device=dev())
    x = x0.clone()
    unet_in = torch.empty(2 * T * h * w, 8, dtype=torch.float16, device=dev())
    c_noise = torch.empty(2 * T, device=dev())
    xr = x0.clone()
    for i in range(steps):
        ops.sampler_prepare(x, z, mask, None, concat, sig, step, unet_in, c_noise, T, h, w)
        torch.cuda.synchronize()
        m = mask[:, None, None, None]
        xr = xr * (1 - m) + z * m
        s = sig[i]
        c_in = 1 / (s * s + 1).sqrt()
        ref_in = torch.cat([torch.cat([xr * c_in, torch.zeros_like(concat)], 1), torch.cat([xr * c_in, concat], 1)], 0)
        check(unet_in.reshape(2 * T, h, w, 8), ref_in.permute(0, 2, 3, 1), rtol=1e-3, atol=1e-3 * float(ref_in.abs().max()),
              name="prepare")
        assert torch.allclose(c_noise, torch.full_like(c_noise, 0.25 * math.log(float(s))), atol=1e-5)
        net = rnd(2 * T * h * w, 4, seed=50 + i, dtype=torch.float32)
        ops.sampler_update(x, net, z, mask, scales, sig, step, steps, T, h, w)
        torch.cuda.synchronize()
        netn = net.reshape(2 * T, h, w, 4).permute(0, 3, 1, 2)
        c_skip, c_out = 1 / (s * s + 1), -s / (s * s + 1).sqrt()
        den = netn * c_out + torch.cat([xr, xr]) * c_skip
        du, dc = den.chunk(2)
        d = du + scales[:, None, None, None] * (dc - du)
        xr = xr + (xr - d) / s * (sig[i + 1] - s)
        if i == steps - 1:
            xr = xr * (1 - m) + z * m
        check(x, xr, rtol=1e-4, atol=1e-4 * float(xr.abs().max()), name=f"update {i}")
    assert int(step.item()) == steps
