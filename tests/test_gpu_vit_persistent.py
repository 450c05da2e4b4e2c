"""The persistent ViT kernels at the row counts a training step gives them.

residual_ln_bwd_kernel, mlp_gemm_kernel<1>/<2> and gelu_bwd_kernel schedule their own work: a CTA (or CTA pair) walks many
tiles through mbarrier rings, an atomic tile counter, double-buffered TMEM accumulators and register-resident column sums.
At B = 256 x 513 tokens every CTA walks dozens of tiles.  Each test here picks a shape, asserts from the device's SM count
and the kernel's own tiling constants that the shape really makes CTAs walk the tiles it is meant to cover, and then checks

  * every output against a float64 reference of the same operation computed on the GPU from the same bf16 / fp32 inputs,
    with a per-element error bound derived from the data (written in each docstring);
  * write guards: outputs are allocated with rows beyond M and pre-filled with NaN, so unwritten rows (NaN below M) and
    stores past the last row (finite above M) both fail;
  * exact probes: inputs whose every intermediate is exact in fp32 and bf16 (small integers, powers of two, GELU
    arguments so large that the kernel's GELU / GELU' are exactly x, 0 or 1), compared with torch.equal.  A tile that is
    skipped, processed twice, written to the wrong rows or read from the wrong tile changes bits.

u = 2^-24 is the unit roundoff of fp32 and 2^-8 that of bf16 (8 significant bits, round to nearest).
"""
import math

import pytest
import torch

from imagefolder_b200 import _capi

pytestmark = pytest.mark.gpu

DEV = "cuda"
NAN = float("nan")
U32 = 2.0 ** -24
U16 = 2.0 ** -8
EPS = 1e-6
CHUNK = 16384                   # rows per float64 reference chunk
# xq_gelu.cuh against the erf GELU (fp32 emulation of both functions over [-30, 30], 2e6 points: 9.2e-7 |x| and 2.8e-7),
# with room for the approximate rcp / ex2 instructions the device uses:
GELU_ERR = 2e-6                 # |gelu_f(x)  - gelu(x)|  <= GELU_ERR * |x|
DGELU_ERR = 1e-6                # |dgelu_f(x) - gelu'(x)| <= DGELU_ERR

LNB_TR = 8                      # residual_ln_bwd_kernel: rows per tile
GM_TILE = 256                   # mlp_gemm_kernel: a CTA pair owns 256 x 256 output tiles
GELU_BWD_RU = 2                 # gelu_bwd_kernel: rows per grid-stride step
GELU_RU = 4                     # gelu_fwd_kernel: rows per CTA


def n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def lib():
    return _capi.lib()


P = _capi.ptr


def stream():
    return _capi.stream_ptr(torch.device(DEV))


def guarded(rows, cols, dtype, extra=7):
    return torch.full((rows + extra, cols), NAN, dtype=dtype, device=DEV)


def guarded_vec(n, extra=32):
    return torch.full((n + extra,), NAN, dtype=torch.float32, device=DEV)


def assert_written(buf, n, what):
    """rows [0, n) all written with finite values, rows [n, end) untouched (still NaN)"""
    assert torch.isfinite(buf[:n]).all(), f"{what}: a row below the bound was not written (or is not finite)"
    assert torch.isnan(buf[n:]).all(), f"{what}: the kernel stored past its last row"


def check_bound(out, ref, bound, what):
    err = (out.double() - ref).abs()
    ratio = err / bound.clamp_min(1e-300)
    worst = int(ratio.flatten().argmax())
    if not bool((err <= bound).all()):
        o, r, b = out.flatten()[worst].item(), ref.flatten()[worst].item(), bound.flatten()[worst].item()
        raise AssertionError(f"{what}: element {worst} (of shape {tuple(out.shape)}) = {o!r}, reference {r!r}, "
                             f"bound {b:.3e}, |err| / bound = {ratio.flatten()[worst].item():.3f}")


def gelu64(x):
    return 0.5 * x * (1.0 + torch.erf(x * 0.5 ** 0.5))


def dgelu64(x):
    return 0.5 * (1.0 + torch.erf(x * 0.5 ** 0.5)) + x * torch.exp(-0.5 * x * x) * (2.0 * math.pi) ** -0.5


def chunks(n, size=CHUNK):
    for r0 in range(0, n, size):
        yield r0, min(n, r0 + size)


# ==================================================================================================================
# 1. LayerNorm backward (xq_vit_residual_ln_bwd: residual_ln_bwd_kernel + reduce_parts_kernel)
# ==================================================================================================================

def ln_schedule(M, min_tiles_per_cta):
    """grid = min(SMs, tiles of 8 rows); every CTA takes its first tile from blockIdx and the rest from the atomic counter.
    Returns (tiles, grid)."""
    ntiles = -(-M // LNB_TR)
    grid = min(n_sms(), ntiles)
    assert ntiles >= min_tiles_per_cta * grid, (
        f"M = {M}: {ntiles} tiles over {grid} CTAs is fewer than {min_tiles_per_cta} tiles per CTA; the case no longer walks")
    return ntiles, grid


def rowscale_values(Bn, seed):
    """per-sample DropPath scales from {0, 1/2, 1, 2}, every sample's value different from its neighbour's"""
    gen = torch.Generator().manual_seed(seed)
    vals = [0.0, 0.5, 1.0, 2.0]
    idx = [int(torch.randint(4, (1,), generator=gen))]
    for _ in range(Bn - 1):
        idx.append((idx[-1] + int(torch.randint(1, 4, (1,), generator=gen))) % 4)
    return torch.tensor([vals[i] for i in idx], device=DEV)


def ln_bwd(g_xout, g_y, x_out, mean, rstd, w, branch, bb, gm, rs, S, M, D):
    """one xq_vit_residual_ln_bwd call into freshly NaN-filled outputs (rows / columns beyond M / D are guards)"""
    L = lib()
    out = {"g_x": guarded(M, D, torch.float32), "g_w": guarded_vec(D), "g_b": guarded_vec(D)}
    out["g_branch"] = guarded(M, D, torch.bfloat16) if branch is not None else None
    out["g_gamma"] = guarded_vec(D) if branch is not None and gm is not None else None
    out["g_bias"] = guarded_vec(D) if branch is not None and bb is not None else None
    ws = _capi.workspace(L.xq_vit_ln_bwd_workspace_bytes(D), DEV)
    _capi.check(L.xq_vit_residual_ln_bwd(P(g_xout), P(g_y), P(x_out), P(mean), P(rstd), P(w), P(branch), P(bb), P(gm), P(rs), S,
                                         M, D, P(out["g_x"]), P(out["g_branch"]), P(out["g_w"]), P(out["g_b"]), P(out["g_gamma"]),
                                         P(out["g_bias"]), P(ws), ws.numel(), stream()), "xq_vit_residual_ln_bwd")
    return out


def ln_stats(x_out):
    """float64 mean / rstd of the fp32 stream, rounded to fp32 as the forward kernel saves them"""
    mean, rstd = torch.empty(x_out.shape[0], device=DEV), torch.empty(x_out.shape[0], device=DEV)
    for r0, r1 in chunks(x_out.shape[0]):
        x = x_out[r0:r1].double()
        mean[r0:r1] = x.mean(1).float()
        rstd[r0:r1] = (x.var(1, unbiased=False) + EPS).rsqrt().float()
    return mean, rstd


def make_ln_inputs(Bn, S, D, path, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    M = Bn * S
    x_out = torch.randn(M, D, generator=g, device=DEV) + 0.5 * torch.randn(M, 1, generator=g, device=DEV)
    mean, rstd = ln_stats(x_out)
    t = dict(x_out=x_out, mean=mean, rstd=rstd, w=torch.rand(D, generator=g, device=DEV) + 0.5,
             b=torch.randn(D, generator=g, device=DEV),
             g_y=torch.randn(M, D, generator=g, device=DEV).to(torch.bfloat16),
             g_xout=None if path == "final" else torch.randn(M, D, generator=g, device=DEV),
             branch=None, bb=None, gm=None, rs=None)
    if path in ("full", "final"):
        t["branch"] = (2 * torch.randn(M, D, generator=g, device=DEV)).to(torch.bfloat16)
        t["bb"] = torch.randn(D, generator=g, device=DEV)
        t["gm"] = torch.rand(D, generator=g, device=DEV) + 0.5
        t["rs"] = rowscale_values(Bn, seed)
    return t


def ln_bwd_reference(t, Bn, S, D, chain):
    """float64 autograd of test_gpu_vit_ops.ref_residual_ln in chunks of whole samples, plus the per-element error bounds.

    The kernel gets x_out (fp32) and the fp32-rounded mean / rstd; the reference starts from x = x_out - s*gamma*(branch+bias)
    in float64, so its residual output IS x_out and its LayerNorm statistics are the exact ones of x_out.  Per row, with
    xh = (x_out - mean) * rstd, gw = g_y * ln_w, S1 = mean_d |gw|, S2 = mean_d |gw * xh| and a = 1 + rstd * |mean| (the
    fp32 rounding of mean moves xh by up to a * u):
      G = g_xout + rstd * (gw - mean_d(gw) - xh * mean_d(gw * xh)) = g_x.  The kernel's two row sums run over D/32 terms per
      lane and a 5-level butterfly, every other step is O(1) roundings, so
        |g_x - G| <= E_G = u |G| + (D/32 + 16) a u rstd (|gw| + S1 + (1 + |xh|) S2).
      g_branch = bf16(G * s * gamma): |err| <= 2^-8 |ref| + (1 + 2^-8) (s gamma E_G + 2u |ref|).
    Column sums are fp32 chains: a lane's register sum over the tiles its CTA took (at most all of them), 8 consumer warps,
    and reduce_parts' 8 strided sums over the CTAs: chain = tiles + 8 + ceil(grid / 8) + 8 + 4.  Each sum's bound is
    chain * u * sum|terms| plus the propagated per-term input errors:
      d ln_w = sum g_y xh:            + sum |g_y| a u (1 + 4 |xh|)
      d ln_b = sum g_y:               (g_y is exact)
      P3 = sum G s, P2 = sum G s branch:  + sum s E_G,  + sum s |branch| E_G
      d gamma = P2 + bias P3:         bound(P2) + |bias| bound(P3) + 2u (sum|G s branch| + |bias| sum|G s|)
      d bias = gamma P3:              gamma bound(P3) + u |ref|."""
    from test_gpu_vit_ops import ref_residual_ln
    has_br = t["branch"] is not None
    per = max(1, CHUNK // S)
    cu = chain * U32
    ref = {"g_x": torch.empty(Bn * S, D, dtype=torch.float64, device=DEV), "E_G": torch.empty(Bn * S, D, dtype=torch.float64, device=DEV)}
    if has_br:
        ref["g_branch"] = torch.empty(Bn * S, D, dtype=torch.float64, device=DEV)
        ref["b_branch"] = torch.empty(Bn * S, D, dtype=torch.float64, device=DEV)
    z = lambda: torch.zeros(D, dtype=torch.float64, device=DEV)
    acc = {k: z() for k in ("g_w", "g_b", "g_gamma", "g_bias", "bw", "bb_", "bP2", "bP3", "aP2", "aP3")}
    for b0 in range(0, Bn, per):
        b1 = min(Bn, b0 + per)
        r0, r1 = b0 * S, b1 * S
        nb = b1 - b0
        xo = t["x_out"][r0:r1].double()
        w64 = t["w"].double().requires_grad_(True)
        lb64 = t["b"].double().requires_grad_(True)
        leaves = [w64, lb64]
        if has_br:
            br64 = t["branch"][r0:r1].double().requires_grad_(True)
            gm64 = t["gm"].double().requires_grad_(True)
            bb64 = t["bb"].double().requires_grad_(True)
            s = t["rs"][b0:b1].double().repeat_interleave(S)[:, None]
            x_in = (xo - s * t["gm"].double() * (br64.detach() + t["bb"].double())).requires_grad_(True)
            xo2, y2 = ref_residual_ln(x_in.view(nb, S, D), br64.view(nb, S, D), gm64, t["rs"][b0:b1], w64, lb64, EPS, S, bb64)
            leaves += [br64, gm64, bb64]
        else:
            x_in = xo.clone().requires_grad_(True)
            xo2, y2 = ref_residual_ln(x_in.view(nb, S, D), None, None, None, w64, lb64, EPS, S)
        gy = t["g_y"][r0:r1].double()
        loss = (y2.reshape(-1, D) * gy).sum()
        if t["g_xout"] is not None:
            loss = loss + (xo2.reshape(-1, D) * t["g_xout"][r0:r1].double()).sum()
        grads = torch.autograd.grad(loss, [x_in] + leaves)
        G = grads[0]
        ref["g_x"][r0:r1] = G
        acc["g_w"] += grads[1]
        acc["g_b"] += grads[2]
        with torch.no_grad():
            mean = xo.mean(1, keepdim=True)
            rstd = (xo.var(1, unbiased=False, keepdim=True) + EPS).rsqrt()
            xh = (xo - mean) * rstd
            gw = gy * t["w"].double()
            S1 = gw.abs().mean(1, keepdim=True)
            S2 = (gw * xh).abs().mean(1, keepdim=True)
            a = 1.0 + rstd * mean.abs()
            E_G = U32 * G.abs() + (D / 32 + 16) * a * U32 * rstd * (gw.abs() + S1 + (1.0 + xh.abs()) * S2)
            ref["E_G"][r0:r1] = E_G
            acc["bw"] += cu * (gy * xh).abs().sum(0) + (gy.abs() * a * U32 * (1.0 + 4.0 * xh.abs())).sum(0)
            acc["bb_"] += cu * gy.abs().sum(0)
            if has_br:
                acc["g_gamma"] += grads[4]
                acc["g_bias"] += grads[5]
                ref["g_branch"][r0:r1] = grads[3]
                gm = t["gm"].double()
                ref["b_branch"][r0:r1] = U16 * grads[3].abs() + (1 + U16) * (s * gm * E_G + 2 * U32 * grads[3].abs())
                br = t["branch"][r0:r1].double()
                acc["bP2"] += cu * (G * s * br).abs().sum(0) + (s * br.abs() * E_G).sum(0)
                acc["bP3"] += cu * (G * s).abs().sum(0) + (s * E_G).sum(0)
                acc["aP2"] += (G * s * br).abs().sum(0)
                acc["aP3"] += (G * s).abs().sum(0)
    ref["g_w"], ref["g_b"] = acc["g_w"], acc["g_b"]
    ref["b_w"], ref["b_b"] = acc["bw"], acc["bb_"]
    if has_br:
        bb, gm = t["bb"].double().abs(), t["gm"].double().abs()
        ref["g_gamma"], ref["g_bias"] = acc["g_gamma"], acc["g_bias"]
        ref["b_gamma"] = acc["bP2"] + bb * acc["bP3"] + 2 * U32 * (acc["aP2"] + bb * acc["aP3"])
        ref["b_bias"] = gm * acc["bP3"] + U32 * acc["g_bias"].abs()
    return ref


LN_CASES = [  # (D, Bn, S): M % 8 = 1, 7, 0; the 2-stage ring is D = 1024, the 3-stage ring D = 384 / 768
    (384, 41, 257),
    (768, 23, 513),
    (1024, 32, 333),
]


def _run_ln_case(D, Bn, S, path, min_tiles):
    M = Bn * S
    ntiles, grid = ln_schedule(M, min_tiles)
    t = make_ln_inputs(Bn, S, D, path, seed=D + S + len(path))
    args = (t["g_xout"], t["g_y"], t["x_out"], t["mean"], t["rstd"], t["w"], t["branch"], t["bb"], t["gm"], t["rs"], S, M, D)
    out = ln_bwd(*args)
    out2 = ln_bwd(*args)
    torch.cuda.synchronize()
    ref = ln_bwd_reference(t, Bn, S, D, chain=ntiles + 8 + -(-grid // 8) + 8 + 4)
    assert_written(out["g_x"], M, "g_x")
    for k in ("g_w", "g_b"):
        assert_written(out[k], D, k)
    check_bound(out["g_x"][:M], ref["g_x"], ref["E_G"], "g_x")
    check_bound(out["g_w"][:D], ref["g_w"], ref["b_w"], "d ln_w")
    check_bound(out["g_b"][:D], ref["g_b"], ref["b_b"], "d ln_b")
    if t["branch"] is not None:
        assert_written(out["g_branch"], M, "g_branch")
        assert_written(out["g_gamma"], D, "d ls_gamma")
        assert_written(out["g_bias"], D, "d branch_bias")
        check_bound(out["g_branch"][:M], ref["g_branch"], ref["b_branch"], "g_branch")
        check_bound(out["g_gamma"][:D], ref["g_gamma"], ref["b_gamma"], "d ls_gamma")
        check_bound(out["g_bias"][:D], ref["g_bias"], ref["b_bias"], "d branch_bias")
    # per-row results do not depend on which CTA took the tile
    assert torch.equal(out["g_x"][:M], out2["g_x"][:M])
    if t["branch"] is not None:
        assert torch.equal(out["g_branch"][:M], out2["g_branch"][:M])


@pytest.mark.parametrize("path", ["full", "no_branch", "final"])
@pytest.mark.parametrize("D,Bn,S", LN_CASES)
def test_residual_ln_bwd_walked_tiles_against_fp64(D, Bn, S, path):
    """xq_vit_residual_ln_bwd with every CTA walking >= 8 tiles of 8 rows on average (so the counter hands out tiles, the 2- and
    3-stage rings wrap and a consumer warp sums many rows into its register partials), tiles straddling sample boundaries of
    the per-sample rowscale, against float64 autograd.  Paths: "full" = branch + bias + LayerScale + rowscale, "no_branch",
    "final" = g_xout None (the encoder's final norm).  Error bounds: see ln_bwd_reference."""
    _run_ln_case(D, Bn, S, path, min_tiles=8)


def test_residual_ln_bwd_training_size_against_fp64():
    """the bench / training size, B = 256 x 513 tokens (M = 131 328, D = 768, every CTA ~110 tiles), full path.  Bounds: see
    ln_bwd_reference."""
    _run_ln_case(768, 256, 513, "full", min_tiles=64)


@pytest.mark.parametrize("D", [384, 768, 1024])
def test_residual_ln_bwd_exact_probe(D):
    """Exact coverage probe at the training row count (256 x 513 rows, every CTA ~110 tiles).

    (a) g_y = None, integer g_xout and branch in [-4, 4], power-of-two LayerScale gamma, rowscale in {0, 1/2, 1, 2} per
        sample, integer branch bias: G = g_xout, so g_x, g_branch = G s gamma, P3 = sum G s, P2 = sum G s branch,
        d ls_gamma = P2 + bias P3 and d branch_bias = gamma P3 are multiples of 1/4 whose every fp32 partial stays below
        2^22 (asserted from the data), i.e. exact in any summation order: torch.equal against the float64 values.
        d ln_w = d ln_b = 0 exactly.
    (b) integer g_y in [-4, 4]: d ln_b = sum g_y is exact in any order: torch.equal.
    Both calls run twice; per-row outputs and column sums are bit-identical across the calls."""
    Bn, S = 256, 513
    M = Bn * S
    ln_schedule(M, 64)
    g = torch.Generator(device=DEV).manual_seed(D)
    x_out = torch.randn(M, D, generator=g, device=DEV)
    mean, rstd = ln_stats(x_out)
    w = torch.rand(D, generator=g, device=DEV) + 0.5
    ri = lambda *shape: torch.randint(-4, 5, shape, generator=g, device=DEV).float()
    g_xout, branch = ri(M, D), ri(M, D).to(torch.bfloat16)
    bb = torch.randint(1, 3, (D,), generator=g, device=DEV).float() * (2 * torch.randint(0, 2, (D,), generator=g, device=DEV) - 1)
    gm = 2.0 ** torch.randint(-1, 2, (D,), generator=g, device=DEV).float()
    rs = rowscale_values(Bn, D)
    s = rs.repeat_interleave(S)[:, None].double()
    G = g_xout.double()
    P2 = torch.zeros(D, dtype=torch.float64, device=DEV)
    P3 = torch.zeros_like(P2)
    A2, A3 = torch.zeros_like(P2), torch.zeros_like(P2)
    for r0, r1 in chunks(M):
        t = G[r0:r1] * s[r0:r1]
        P3 += t.sum(0)
        A3 += t.abs().sum(0)
        P2 += (t * branch[r0:r1].double()).sum(0)
        A2 += (t * branch[r0:r1].double()).abs().sum(0)
    assert float((A2 + bb.double().abs() * A3).max()) * 4 < 2 ** 24, "probe values too large for exact fp32 column sums"
    for rep in range(2):
        out = ln_bwd(g_xout, None, x_out, mean, rstd, w, branch, bb, gm, rs, S, M, D)
        assert_written(out["g_x"], M, "g_x")
        assert_written(out["g_branch"], M, "g_branch")
        for k in ("g_w", "g_b", "g_gamma", "g_bias"):
            assert_written(out[k], D, k)
        assert torch.equal(out["g_x"][:M], g_xout)
        assert torch.equal(out["g_branch"][:M].double(), G * s * gm.double())
        assert torch.equal(out["g_gamma"][:D].double(), P2 + bb.double() * P3)
        assert torch.equal(out["g_bias"][:D].double(), gm.double() * P3)
        assert torch.equal(out["g_w"][:D], torch.zeros(D, device=DEV)) and torch.equal(out["g_b"][:D], torch.zeros(D, device=DEV))
        if rep:
            for k in ("g_x", "g_branch"):
                assert torch.equal(out[k][:M], first[k][:M]), k
            for k in ("g_w", "g_b", "g_gamma", "g_bias"):
                assert torch.equal(out[k][:D], first[k][:D]), k
        first = out
    g_y = ri(M, D).to(torch.bfloat16)
    assert float(g_y.float().abs().sum(0).max()) < 2 ** 24
    d_lnb = g_y.double().sum(0)
    outs = [ln_bwd(None, g_y, x_out, mean, rstd, w, None, None, None, None, S, M, D) for _ in range(2)]
    for out in outs:
        assert_written(out["g_x"], M, "g_x")
        assert_written(out["g_b"], D, "d ln_b")
        assert torch.equal(out["g_b"][:D].double(), d_lnb)
    assert torch.equal(outs[0]["g_x"][:M], outs[1]["g_x"][:M]) and torch.equal(outs[0]["g_b"][:D], outs[1]["g_b"][:D])


# ==================================================================================================================
# 2. Fused MLP GEMMs (xq_vit_fc1_gelu_fwd / xq_vit_fc2_dgelu_bwd: mlp_gemm_kernel<1> / <2>)
# ==================================================================================================================

def gemm_schedule(M, N, min_walk):
    """The launcher's schedule: nN = N / 256 column blocks, nM = ceil(M / 256) row blocks, per_col = min((SMs/2) / nN, nM)
    pairs per column block; pair p keeps column block p % nN and walks row blocks p / nN, + per_col, ...  Returns
    (per_col, fewest row blocks any pair walks, most row blocks any pair walks)."""
    max_pairs = n_sms() // 2
    nN, nM = N // GM_TILE, -(-M // GM_TILE)
    assert nN <= max_pairs
    per_col = min(max_pairs // nN, nM)
    walk_min, walk_max = nM // per_col, -(-nM // per_col)
    assert walk_min >= min_walk, f"M = {M}, N = {N}: a pair walks only {walk_min} row blocks (want >= {min_walk})"
    return per_col, walk_min, walk_max


def wide_n():
    return GM_TILE * (n_sms() // 2)


GEMM_CASES = [  # (M, K, N, fewest row blocks a pair must walk); N = None: 256 * floor(SMs / 2), one pair per column block
    pytest.param(131328, 768, 3072, 3, id="prod-768x3072"),
    pytest.param(131328, 384, 1536, 3, id="prod-384x1536"),
    pytest.param(131329, 768, 3072, 3, id="tail-1-row"),          # last row block: rank 0 one row, rank 1 none
    pytest.param(131199, 768, 3072, 3, id="tail-127-rows"),       # M = 131328 - 129, M % 256 = 127
    pytest.param(48 * 256 + 127, 384, 1536, 3, id="mid-127-rows"),
    pytest.param(80 * 256 - 3, 64, 1536, 6, id="K64"),             # one k-block per tile: the 5-stage ring spans 5 tiles
    pytest.param(80 * 256 - 3, 128, 1536, 6, id="K128"),
    pytest.param(5 * 256 - 19, 256, None, 3, id="wide-N"),         # every pair walks every row block
]


def rows_to_check(M, full=40000):
    """all rows for moderate M; beyond that (the float64 GEMM of all 131k rows would take ~20 s) one row in every 32-row
    slab of every row block -- i.e. every (row block, CTA rank, epilogue warp) the schedule produces, at a lane that varies
    from block to block -- plus every row of the first and the last two row blocks."""
    if M <= full:
        return torch.arange(M, device=DEV)
    nM = -(-M // GM_TILE)
    r = [b * GM_TILE + s * 32 + (7 * s + 5 * b) % 32 for b in range(nM) for s in range(8)]
    r += list(range(GM_TILE)) + list(range((nM - 2) * GM_TILE, M))
    return torch.tensor(sorted(set(i for i in r if i < M)), device=DEV)


def fc1_fwd(y, W1, b1, M, N, K):
    pre, act = guarded(M, N, torch.bfloat16), guarded(M, N, torch.bfloat16)
    _capi.check(lib().xq_vit_fc1_gelu_fwd(P(y), P(W1), P(b1), P(pre), P(act), M, N, K, stream()), "xq_vit_fc1_gelu_fwd")
    return pre, act


def fc2_bwd(g, W2t, pre, b1, M, N, K):
    d_pre, d_b1 = guarded(M, N, torch.bfloat16), guarded_vec(N)
    _capi.check(lib().xq_vit_fc2_dgelu_bwd(P(g), P(W2t), P(pre), P(b1), P(d_pre), P(d_b1), M, N, K, stream()),
                "xq_vit_fc2_dgelu_bwd")
    return d_pre, d_b1


@pytest.mark.parametrize("M,K,N,min_walk", GEMM_CASES)
def test_fc1_gelu_fwd_against_fp64(M, K, N, min_walk):
    """pre = y W1^T (bf16) against float64: |pre - ref| <= 2^-8 |ref| + 1.01 c (|y| @ |W1|^T), c = 2 K u -- bf16 x bf16
    products are exact in fp32 and each of the K fp32 accumulations may lose up to 2u (the tensor core may truncate
    instead of rounding); 1.01 covers the final rounding applied to that error.
    act against gelu64(pre_kernel + b1), i.e. the epilogue alone on the kernel's own rounded pre-activation:
    |act - ref| <= 2^-8 |ref| + (1 + 2^-8)(GELU_ERR + 2u) |x|  (GELU approximation, fp32 rounding of x, bf16 output)."""
    N = N or wide_n()
    gemm_schedule(M, N, min_walk)
    g = torch.Generator(device=DEV).manual_seed(M + K + N)
    y = torch.randn(M, K, generator=g, device=DEV).to(torch.bfloat16)
    W1 = (torch.randn(N, K, generator=g, device=DEV) * K ** -0.5).to(torch.bfloat16)
    b1 = 0.5 * torch.randn(N, generator=g, device=DEV)
    pre, act = fc1_fwd(y, W1, b1, M, N, K)
    torch.cuda.synchronize()
    assert_written(pre, M, "pre")
    assert_written(act, M, "act")
    W = W1.double()
    c = 2 * K * U32
    rows = rows_to_check(M)
    for i0, i1 in chunks(rows.numel(), 4096):
        r = rows[i0:i1]
        A = y[r].double()
        ref = A @ W.t()
        check_bound(pre[r], ref, U16 * ref.abs() + 1.01 * c * (A.abs() @ W.abs().t()), "pre")
    b64 = b1.double()
    for r0, r1 in chunks(M):
        x = pre[r0:r1].double() + b64
        ref = gelu64(x)
        check_bound(act[r0:r1], ref, U16 * ref.abs() + (1 + U16) * (GELU_ERR + 2 * U32) * x.abs(), "act")


@pytest.mark.parametrize("M,K,N,min_walk", GEMM_CASES)
def test_fc2_dgelu_bwd_against_fp64(M, K, N, min_walk):
    """d_pre = bf16(bf16(g W2) * gelu'(pre + b1)) against (g W2) * gelu64'(pre + b1) in float64.  With dact = g W2 (fp64),
    S = |g| @ |W2|, c = 2 K u (as in the forward), x = pre + b1:
      E = |gelu64'(x)| (2^-8 |dact| + 1.01 c S) + |dact| (DGELU_ERR + u |x|)     (rounded GEMM output, GELU' error, fp32 x)
      |d_pre - ref| <= 2^-8 |ref| + 1.02 E + 2u |ref|.
    d_b1 against the float64 column sums of the kernel's own d_pre: each thread adds one 32-row butterfly sum (5 levels) per
    row block it walks, then 2 ranks x 4 warps x per_col pairs add atomically, so
      |d_b1 - ref| <= (walk + 5 + 8 per_col + 2) u sum|d_pre|.
    The backward runs twice: d_pre is bit-identical and d_b1 meets the same bound (it is zeroed, not accumulated)."""
    N = N or wide_n()
    per_col, _, walk_max = gemm_schedule(M, N, min_walk)
    g_ = torch.Generator(device=DEV).manual_seed(M + K + N + 1)
    g = torch.randn(M, K, generator=g_, device=DEV).to(torch.bfloat16)
    W2t = (torch.randn(N, K, generator=g_, device=DEV) * K ** -0.5).to(torch.bfloat16)
    pre = guarded(M, N, torch.bfloat16)                 # rows >= M stay NaN: a read past M would poison d_b1
    for r0, r1 in chunks(M):
        pre[r0:r1] = (2 * torch.randn(r1 - r0, N, generator=g_, device=DEV)).to(torch.bfloat16)
    b1 = 0.5 * torch.randn(N, generator=g_, device=DEV)
    d_pre, d_b1 = fc2_bwd(g, W2t, pre, b1, M, N, K)
    d_pre2, d_b1_2 = fc2_bwd(g, W2t, pre, b1, M, N, K)
    torch.cuda.synchronize()
    assert_written(d_pre, M, "d_pre")
    assert_written(d_b1, N, "d_b1")
    assert torch.equal(d_pre[:M], d_pre2[:M])
    W = W2t.double()
    c = 2 * K * U32
    b64 = b1.double()
    rows = rows_to_check(M)
    for i0, i1 in chunks(rows.numel(), 4096):
        r = rows[i0:i1]
        A = g[r].double()
        dact = A @ W.t()
        x = pre[r].double() + b64
        dg = dgelu64(x)
        ref = dact * dg
        E = dg.abs() * (U16 * dact.abs() + 1.01 * c * (A.abs() @ W.abs().t())) + dact.abs() * (DGELU_ERR + U32 * x.abs())
        check_bound(d_pre[r], ref, U16 * ref.abs() + 1.02 * E + 2 * U32 * ref.abs(), "d_pre")
    col = torch.zeros(N, dtype=torch.float64, device=DEV)
    col_abs = torch.zeros_like(col)
    for r0, r1 in chunks(M):
        d = d_pre[r0:r1].double()
        col += d.sum(0)
        col_abs += d.abs().sum(0)
    bound = (walk_max + 5 + 8 * per_col + 2) * U32 * col_abs
    check_bound(d_b1[:N], col, bound, "d_b1")
    check_bound(d_b1_2[:N], col, bound, "d_b1 (second call)")


def digit_rows(M, K):
    """[M, K] bf16 rows with three non-zeros: 1 at m % K, 1/2 at (m // K) % K, 1/4 at (m // K^2) % K (added where they
    coincide) -- distinct for all m < K^3; and the three index vectors"""
    m = torch.arange(M, device=DEV)
    d = [m % K, (m // K) % K, (m // (K * K)) % K]
    A = torch.zeros(M, K, device=DEV)
    for wgt, di in zip((1.0, 0.5, 0.25), d):
        A.index_put_((m, di), torch.full((M,), wgt, device=DEV), accumulate=True)
    return A.to(torch.bfloat16), d


def digit_product(Wf, d, r0, r1):
    """rows [r0, r1) of digit_rows @ Wf^T, computed exactly by gathering columns of Wf [N, K] (fp32)"""
    return (Wf[:, d[0][r0:r1]] + 0.5 * Wf[:, d[1][r0:r1]] + 0.25 * Wf[:, d[2][r0:r1]]).t()


@pytest.mark.parametrize("M,K,N,min_walk", GEMM_CASES)
def test_fc1_gelu_fwd_exact_probe(M, K, N, min_walk):
    """y has three non-zeros per row (digit_rows, unique per row), W1 integers in [-8, 8], b1 = +-40 per column: pre is a
    multiple of 1/4 with |pre| <= 14 (exact in fp32 and bf16), x = pre + b1 lies in [26, 54] or [-54, -26], where the
    kernel's GELU is exactly x or 0.  pre and act must equal the gathered reference bit for bit on every row."""
    N = N or wide_n()
    gemm_schedule(M, N, min_walk)
    assert K ** 3 >= M
    g = torch.Generator(device=DEV).manual_seed(M + K + N + 2)
    y, d = digit_rows(M, K)
    W1 = torch.randint(-8, 9, (N, K), generator=g, device=DEV).float()
    b1 = 40.0 * (2 * torch.randint(0, 2, (N,), generator=g, device=DEV) - 1).float()
    pre, act = fc1_fwd(y, W1.to(torch.bfloat16), b1, M, N, K)
    torch.cuda.synchronize()
    assert_written(pre, M, "pre")
    assert_written(act, M, "act")
    for r0, r1 in chunks(M):
        ref = digit_product(W1, d, r0, r1)
        assert torch.equal(pre[r0:r1].float(), ref), f"pre rows {r0}..{r1}"
        assert torch.equal(act[r0:r1].float(), torch.where(b1 > 0, ref + b1, 0.0)), f"act rows {r0}..{r1}"


@pytest.mark.parametrize("M,K,N,min_walk", GEMM_CASES)
def test_fc2_dgelu_bwd_exact_probe(M, K, N, min_walk):
    """g has three non-zeros per row (digit_rows), W2 integers in [-8, 8], pre = +-16 with a random sign per element and
    b1 = 0, where the kernel's GELU' is exactly 1 or 0: d_act is a multiple of 1/4 with |d_act| <= 14 (exact in bf16),
    d_pre = d_act * mask and d_b1 = its column sums, every fp32 partial a multiple of 1/4 below 2^22 (asserted), so both
    equal the reference bit for bit.  A prefetch of pre from the wrong rows or tile changes the mask.  Two calls: d_b1 is
    not accumulated across them."""
    N = N or wide_n()
    gemm_schedule(M, N, min_walk)
    assert K ** 3 >= M
    g_ = torch.Generator(device=DEV).manual_seed(M + K + N + 3)
    g, d = digit_rows(M, K)
    W2t = torch.randint(-8, 9, (N, K), generator=g_, device=DEV).float()
    pre = guarded(M, N, torch.bfloat16)
    for r0, r1 in chunks(M):
        pre[r0:r1] = 16.0 * (2 * torch.randint(0, 2, (r1 - r0, N), generator=g_, device=DEV) - 1).to(torch.bfloat16)
    b1 = torch.zeros(N, device=DEV)
    outs = [fc2_bwd(g, W2t.to(torch.bfloat16), pre, b1, M, N, K) for _ in range(2)]
    torch.cuda.synchronize()
    col = torch.zeros(N, dtype=torch.float64, device=DEV)
    col_abs = torch.zeros_like(col)
    for r0, r1 in chunks(M):
        ref = torch.where(pre[r0:r1] > 0, digit_product(W2t, d, r0, r1), 0.0)
        col += ref.double().sum(0)
        col_abs += ref.double().abs().sum(0)
        for d_pre, _ in outs:
            assert torch.equal(d_pre[r0:r1].float(), ref), f"d_pre rows {r0}..{r1}"
    assert float(col_abs.max()) * 4 < 2 ** 24
    for d_pre, d_b1 in outs:
        assert_written(d_pre, M, "d_pre")
        assert_written(d_b1, N, "d_b1")
        assert torch.equal(d_b1[:N].double(), col)


@pytest.mark.parametrize("out_features,fused", [(200, False), (192, True)])
def test_mlp_output_width_decides_the_fused_path(out_features, fused):
    """The fused backward GEMM takes the fc2 output width as its K, which must be a multiple of 64.  An Mlp whose
    out-features is not (200) must run forward AND backward through the library path (bit-identical to it); one whose
    out-features is (192, != the input width 768) runs the fused GEMMs and matches the library path at bf16 resolution."""
    from imagefolder_b200 import vit_ops
    torch.manual_seed(out_features)
    mlp = torch.nn.Module()
    mlp.fc1 = torch.nn.Linear(768, 3072).to(DEV)
    mlp.fc2 = torch.nn.Linear(3072, out_features).to(DEV)
    y0 = torch.randn(2 * 513, 768, device=DEV).to(torch.bfloat16)
    g = torch.randn(2 * 513, out_features, device=DEV).to(torch.bfloat16)
    assert vit_ops.mlp_tc_ok(y0, mlp.fc1, mlp.fc2) is fused

    def run(enabled):
        vit_ops.MLP_TC_ENABLED[0] = enabled
        for p in mlp.parameters():
            p.grad = None
        y = y0.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = vit_ops.mlp_forward(mlp, y)
        out.backward(g)
        return out.detach(), y.grad, mlp.fc1.weight.grad, mlp.fc1.bias.grad, mlp.fc2.weight.grad

    try:
        a = run(True)
        b = run(False)
    finally:
        vit_ops.MLP_TC_ENABLED[0] = True
    for n, u, v in zip(["branch", "d_y", "d_W1", "d_b1", "d_W2"], a, b):
        if not fused and n != "d_b1":   # d_b1 is summed with fp32 atomics, whose order may differ between the two runs
            assert torch.equal(u, v), n
        else:   # same bound as test_gpu_vit_ops' library-path comparison: the paths differ only in GEMM accumulation order
            assert torch.isfinite(u.float()).all(), n
            scale = max(1e-6, v.float().abs().max().item())
            assert (u.float() - v.float()).abs().max().item() <= 8e-3 * scale, n


# ==================================================================================================================
# 3. GELU kernels (xq_vit_gelu_fwd / xq_vit_gelu_bwd)
# ==================================================================================================================

def gelu_threads(C):
    C8 = C // 8
    return 384 if C8 >= 384 else (192 if C8 >= 192 else 128)


def gelu_bwd_schedule(M, C, min_steps):
    """gelu_bwd_kernel's grid is SMs x (co-resident CTAs per SM), at most SMs x min(32, 2048 / threads); CTA b walks rows
    2b, 2b + 2 grid, ...  Returns (largest possible grid, longest per-thread fp32 chain of the bias-gradient sum)."""
    sms = n_sms()
    grid_max = sms * min(32, 2048 // gelu_threads(C))
    steps_min = -(-(M - GELU_BWD_RU * grid_max + GELU_BWD_RU) // (GELU_BWD_RU * grid_max))
    assert steps_min >= min_steps, f"M = {M}: a CTA may take only {steps_min} grid-stride steps (want >= {min_steps})"
    assert M % (GELU_BWD_RU * grid_max) != 0 and M % 2 == 1      # odd: the last step of some CTA has one row
    rows_per_thread = GELU_BWD_RU * -(-M // (GELU_BWD_RU * sms))  # the grid has at least SMs CTAs
    return grid_max, rows_per_thread + grid_max + 2


def gelu_bwd_rows(C):
    grid_max = n_sms() * min(32, 2048 // gelu_threads(C))
    return (7 * grid_max + 1) | 1                                 # >= 3.5 steps per CTA, odd


def gelu_bwd(x, bias, gy, M, C):
    gx, gb = guarded(M, C, torch.bfloat16), guarded_vec(C)
    _capi.check(lib().xq_vit_gelu_bwd(P(x), P(bias), P(gy), P(gx), P(gb), M, C, stream()), "xq_vit_gelu_bwd")
    return gx, gb


@pytest.mark.parametrize("C", [64, 1536, 3072])
def test_gelu_bwd_grid_stride_against_fp64(C):
    """gelu_bwd_kernel with every CTA taking >= 3 software-pipelined grid-stride steps (so the prefetched next rows are
    used), in its 128-, 192- and 384-thread configurations, odd M.  With x = x_bf16 + bias and r = gy gelu64'(x):
      |gx - r| <= 2^-8 |r| + (1 + 2^-8) (|gy| (DGELU_ERR + u |x|) + u |r|)
    (GELU' approximation, fp32 rounding of x and of the product, bf16 output).  d bias sums the unrounded fp32 products per
    thread over its rows, then one atomicAdd per CTA:
      |d bias - sum r| <= sum |gy| (DGELU_ERR + u |x|) + (rows per thread + grid + 2) u sum |r|."""
    M = gelu_bwd_rows(C)
    _, chain = gelu_bwd_schedule(M, C, 3)
    g = torch.Generator(device=DEV).manual_seed(C)
    x = (2 * torch.randn(M, C, generator=g, device=DEV)).to(torch.bfloat16)
    bias = 0.5 * torch.randn(C, generator=g, device=DEV)
    gy = torch.randn(M, C, generator=g, device=DEV).to(torch.bfloat16)
    gx, gb = gelu_bwd(x, bias, gy, M, C)
    gx2, gb2 = gelu_bwd(x, bias, gy, M, C)
    torch.cuda.synchronize()
    assert_written(gx, M, "gx")
    assert_written(gb, C, "d bias")
    assert torch.equal(gx[:M], gx2[:M])
    xs = x.double() + bias.double()
    g64 = gy.double()
    r = g64 * dgelu64(xs)
    e = g64.abs() * (DGELU_ERR + U32 * xs.abs())
    check_bound(gx[:M], r, U16 * r.abs() + (1 + U16) * (e + U32 * r.abs()), "gx")
    bound = e.sum(0) + chain * U32 * r.abs().sum(0)
    check_bound(gb[:C], r.sum(0), bound, "d bias")
    check_bound(gb2[:C], r.sum(0), bound, "d bias (second call)")


@pytest.mark.parametrize("C", [64, 1536, 3072])
def test_gelu_bwd_exact_probe(C):
    """x + bias = +-20 (integer bias in [-4, 4], so x is an integer in [-24, 24], exact in bf16) and integer gy in [-4, 4]:
    the kernel's GELU' is exactly 1 or 0, so gx = gy * mask and d bias = its column sums (integers below 2^24) are
    exact: torch.equal, on both of two calls."""
    M = gelu_bwd_rows(C)
    gelu_bwd_schedule(M, C, 3)
    g = torch.Generator(device=DEV).manual_seed(C + 1)
    bias = torch.randint(-4, 5, (C,), generator=g, device=DEV).float()
    sign = (2 * torch.randint(0, 2, (M, C), generator=g, device=DEV) - 1).float()
    x = (20.0 * sign - bias).to(torch.bfloat16)
    gy = torch.randint(-4, 5, (M, C), generator=g, device=DEV).float()
    ref = torch.where(sign > 0, gy, 0.0)
    for _ in range(2):
        gx, gb = gelu_bwd(x, bias, gy.to(torch.bfloat16), M, C)
        assert_written(gx, M, "gx")
        assert_written(gb, C, "d bias")
        assert torch.equal(gx[:M].float(), ref)
        assert torch.equal(gb[:C], ref.sum(0))


@pytest.mark.parametrize("M,C", [(4 * 37 + 1, 3072), (4 * 50 + 2, 1536), (4 * 61 + 3, 64), (4 * 1001 + 3, 768)])
def test_gelu_fwd_ragged_rows(M, C):
    """gelu_fwd_kernel runs ceil(M / 4) CTAs of 4 rows; M % 4 != 0 leaves the last CTA a partial tile (the row0 + u < M tail).
    Random input against gelu64(x_bf16 + bias): |y - ref| <= 2^-8 |ref| + (1 + 2^-8)(GELU_ERR + 2u) |x|.  Exact probe:
    x + bias = +-20 (integer bias), where the kernel's GELU is exactly x + bias or 0: torch.equal."""
    assert M % GELU_RU != 0
    g = torch.Generator(device=DEV).manual_seed(M)
    L = lib()
    x = (2 * torch.randn(M, C, generator=g, device=DEV)).to(torch.bfloat16)
    bias = 0.5 * torch.randn(C, generator=g, device=DEV)
    y = guarded(M, C, torch.bfloat16)
    _capi.check(L.xq_vit_gelu_fwd(P(x), P(bias), P(y), M, C, stream()), "xq_vit_gelu_fwd")
    torch.cuda.synchronize()
    assert_written(y, M, "y")
    xs = x.double() + bias.double()
    ref = gelu64(xs)
    check_bound(y[:M], ref, U16 * ref.abs() + (1 + U16) * (GELU_ERR + 2 * U32) * xs.abs(), "y")
    ib = torch.randint(-4, 5, (C,), generator=g, device=DEV).float()
    sign = (2 * torch.randint(0, 2, (M, C), generator=g, device=DEV) - 1).float()
    xp = (20.0 * sign - ib).to(torch.bfloat16)
    y = guarded(M, C, torch.bfloat16)
    _capi.check(L.xq_vit_gelu_fwd(P(xp), P(ib), P(y), M, C, stream()), "xq_vit_gelu_fwd")
    assert_written(y, M, "y (probe)")
    assert torch.equal(y[:M].float(), torch.where(sign > 0, 20.0 * sign, 0.0))
