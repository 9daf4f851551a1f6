"""Every compiled epilogue specialization of the tap-GEMM (b200v_gemm, csrc/gemm_tc.cu) against an fp64 reference on the
same rounded inputs, reached through ops.gemm by its feature set, in linear and 3x3-tap mode.

Every case has a ragged token count (not a multiple of 128), an N whose last n-tile is partial and has 32-column groups
wholly beyond N (N = 328, tile_n = 256; GEGLU needs N % tile_n == 0 and keeps only the ragged token count), non-unit
s_acc / s_res1 / s_res2, residuals and row vector with their own row strides and rv_div * rv_mod != tokens.  The output
is a column slice of a wider buffer with extra rows below it, pre-filled with a NaN bit pattern: the epilogue must leave
every element outside its rows and columns untouched.  Each specialized case is also run through the generic kernel
(VB_GEMM_GENERIC=1) and must agree bit for bit: both evaluate the same sequence of explicit fmaf's.

VB_GEMM_PAIR and VB_GEMM_NQ are read once per process, so the CTA-pair kernel and the forced 16- / 8-warp epilogues run
the matrix in a child process."""
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from vista_b200.ops import TAPS_3X3
from vista_b200.weights import permute_geglu

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

M_LIN = 555                 # 5 m-tiles: ragged, and an odd m-tile count for the CTA-pair schedule
GEOM = (24, 11, 3)          # (W, H, NB): 792 tokens; pick_box -> (32, 4, 1), which divides neither W nor H; 9 m-tiles
N, TILE_N = 328, 256        # last n-tile: 72 columns, groups 3 .. 7 (CG = 32) wholly beyond N
RV_DIV, RV_MOD = 41, 6
S_ACC, S_RES1, S_RES2 = 0.75, 0.5, -1.25
COL0, EXTRA_COLS, EXTRA_ROWS = 16, 24, 7

NAN_BITS = {torch.float16: 0x7E01, torch.bfloat16: 0x7FC1, torch.float32: 0x7FC00001}

# name -> (features, K of the linear mode); one per tapgemm_kernel instantiation b200v_gemm selects, plus two that take
# the generic one
CASES = {
    "plain": ((), 128),
    "res1": (("res1",), 128),
    "res1_res2": (("res1", "res2"), 128),
    "rowvec": (("rowvec",), 128),
    "rowvec_res1": (("rowvec", "res1"), 128),
    "silu_f16": (("silu",), 128),
    "geglu_k320": (("geglu",), 320),             # 16-warp epilogue (K <= 384)
    "geglu_k640": (("geglu",), 640),             # 8-warp epilogue
    "generic_f32_out": (("rowvec", "res1", "res2", "silu", "f32"), 128),
    "generic_bf16": (("rowvec", "res1", "res2", "bf16"), 128),
}
SPECIALIZED = [c for c in CASES if not c.startswith("generic")]
MATRIX = [(c, m) for c in CASES for m in ("linear", "tap3x3") if not (c.startswith("geglu") and m == "tap3x3")]


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
    out = out.double()
    ref = ref.double()
    err = (out - ref).abs()
    bad = err > atol + rtol * ref.abs()
    rel = float((out - ref).norm() / (ref.norm() + 1e-20))
    assert not bool(bad.any()), (f"{name}: {int(bad.sum())}/{bad.numel()} mismatches, max err {float(err.max()):.4g}, "
                                 f"rel-L2 {rel:.3g}, first bad idx {bad.nonzero()[:4].tolist()}")


def strided(rows, cols, ld, seed, dtype, scale=1.0):
    """[rows, cols] view with row stride ld (columns ld - cols .. of each row hold other data)."""
    return rnd(rows, ld, seed=seed, dtype=dtype, scale=scale)[:, ld - cols:]


def problem(case, mode, tile_n=TILE_N):
    """Inputs, ops.gemm keyword arguments and the fp64 reference of one case."""
    feats, k_lin = CASES[case]
    dt = torch.bfloat16 if "bf16" in feats else torch.float16
    out_dt = torch.float32 if "f32" in feats else dt
    if mode == "linear":
        tokens, cin = M_LIN, k_lin
    else:
        (W, H, NB), cin = GEOM, 64
        tokens = W * H * NB
    a = rnd(tokens, cin, seed=1, dtype=dt)
    if "geglu" in feats:
        n = 2 * TILE_N                                           # N % tile_n == 0; the output has n / 2 columns
        w = rnd(n, cin, seed=2, dtype=dt, scale=cin ** -0.5)
        bias = rnd(n, seed=3, dtype=torch.float32)
        wp, bp = permute_geglu(w, bias, TILE_N)
        val, gate = (a.double() @ w.double().t() + bias.double()).chunk(2, dim=-1)
        return a, wp, tokens, n // 2, out_dt, dict(bias=bp, act=2, tile_n=TILE_N), val * F.gelu(gate)
    bias = rnd(N, seed=3, dtype=torch.float32)
    kw = dict(bias=bias, s_acc=S_ACC, tile_n=tile_n)
    if mode == "linear":
        w = rnd(N, cin, seed=2, dtype=dt, scale=cin ** -0.5)
        acc = a.double() @ w.double().t()
    else:
        wt = rnd(N, cin, 3, 3, seed=2, dtype=dt, scale=(9 * cin) ** -0.5)
        w = wt.permute(0, 2, 3, 1).reshape(N, 9 * cin).contiguous()
        x4 = a.double().reshape(NB, H, W, cin).permute(0, 3, 1, 2)
        acc = F.conv2d(x4, wt.double(), padding=1).permute(0, 2, 3, 1).reshape(tokens, N)
        kw.update(taps=TAPS_3X3, geom=GEOM)
    ref = S_ACC * (acc + bias.double())
    if "rowvec" in feats:
        rv = strided(RV_MOD, N, N + 12, seed=4, dtype=torch.float32)
        kw.update(rowvec=rv, rv_div=RV_DIV, rv_mod=RV_MOD)
        ref = ref + rv.double()[(torch.arange(tokens, device=dev()) // RV_DIV) % RV_MOD]
    if "silu" in feats:
        kw["act"] = 1
        ref = F.silu(ref)
    if "res1" in feats:
        r1 = strided(tokens, N, N + 24, seed=5, dtype=dt)
        kw.update(res1=r1, s_res1=S_RES1)
        ref = ref + S_RES1 * r1.double()
    if "res2" in feats:
        r2 = strided(tokens, N, N + 40, seed=6, dtype=dt)
        kw.update(res2=r2, s_res2=S_RES2)
        ref = ref + S_RES2 * r2.double()
    return a, w, tokens, N, out_dt, kw, ref


def launch(ops, a, w, tokens, n_out, out_dt, kw):
    """ops.gemm into a column slice of a NaN-filled buffer; returns (buffer, slice)."""
    bits = torch.int32 if out_dt == torch.float32 else torch.int16
    buf = torch.full((tokens + EXTRA_ROWS, COL0 + n_out + EXTRA_COLS), NAN_BITS[out_dt], dtype=bits, device=dev()).view(out_dt)
    out = buf[:tokens, COL0:COL0 + n_out]
    ops.gemm(a, w, out, **kw)
    torch.cuda.synchronize()
    return buf, out


def assert_guard(buf, tokens, n_out, name):
    bits = buf.view(torch.int32 if buf.dtype == torch.float32 else torch.int16)
    outside = torch.ones_like(bits, dtype=torch.bool)
    outside[:tokens, COL0:COL0 + n_out] = False
    touched = (bits != NAN_BITS[buf.dtype]) & outside
    assert not bool(touched.any()), f"{name}: {int(touched.sum())} elements written outside the output, first at " \
                                    f"{touched.nonzero()[:4].tolist()}"


def run_case(ops, case, mode):
    a, w, tokens, n_out, out_dt, kw, ref = problem(case, mode)
    buf, out = launch(ops, a, w, tokens, n_out, out_dt, kw)
    # bf16 output: its rounding alone is up to 2^-8 relative, twice the fp16 tolerance
    tol = 8e-3 if out_dt == torch.bfloat16 else 2e-3
    check(out, ref, rtol=tol, atol=tol, name=f"{case}/{mode}")
    assert_guard(buf, tokens, n_out, f"{case}/{mode}")
    return buf, (a, w, tokens, n_out, out_dt, kw)


@pytest.mark.parametrize("case,mode", MATRIX, ids=[f"{c}-{m}" for c, m in MATRIX])
def test_gemm_epilogue_matrix(ops, case, mode, monkeypatch):
    buf, args = run_case(ops, case, mode)
    if case in SPECIALIZED:
        monkeypatch.setenv("VB_GEMM_GENERIC", "1")
        gbuf, _ = launch(ops, *args)
        assert torch.equal(buf.view(torch.int16), gbuf.view(torch.int16)), \
            f"{case}/{mode}: specialized and generic epilogues differ"


def test_gemm_tile_n_sweep(ops):
    """One 3x3 convolution at every legal tile_n: each against the reference; whether the results are bitwise identical
    across tile_n is printed (the MMA's accumulation order is not documented to be independent of N)."""
    results = {}
    for tn in range(32, 257, 32):
        a, w, tokens, n_out, out_dt, kw, ref = problem("rowvec_res1", "tap3x3", tile_n=tn)
        buf, out = launch(ops, a, w, tokens, n_out, out_dt, kw)
        check(out, ref, name=f"tile_n {tn}")
        assert_guard(buf, tokens, n_out, f"tile_n {tn}")
        results[tn] = out.clone()
    same = [tn for tn in results if torch.equal(results[tn].view(torch.int16), results[256].view(torch.int16))]
    print(f"tile_n sweep: bitwise equal to tile_n 256 at {same} of {list(results)}")


@pytest.mark.parametrize("env", [{"VB_GEMM_PAIR": "1"}, {"VB_GEMM_NQ": "4"}, {"VB_GEMM_NQ": "2"}],
                         ids=["pair", "nq4", "nq2"])
def test_gemm_epilogue_matrix_process_wide_kernels(env):
    """The matrix above in a child process with a kernel choice that b200v_gemm reads once per process."""
    child_env = {k: v for k, v in os.environ.items() if k not in ("VB_GEMM_PAIR", "VB_GEMM_NQ", "VB_GEMM_GENERIC")}
    child_env.update(env)
    cmd = [sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", os.path.abspath(__file__),
           "-k", "test_gemm_epilogue_matrix and not process_wide"]
    r = subprocess.run(cmd, cwd=ROOT, env=child_env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                       timeout=600)
    assert r.returncode == 0, f"{env}: child pytest failed\n{r.stdout[-6000:]}"
    assert f"{len(MATRIX)} passed" in r.stdout, r.stdout[-2000:]
