"""The kernels around the convolutions of configs 1 and 3 against plain float64 references, in bf16 AND fp16 (the default
fp16_w2 mode stores activations as fp16): stem packing and max-pooling (csrc/pointwise.cu, bit-exact), the FCOS-tower
GroupNorm (csrc/groupnorm.cu), LayerNorm, patch merging, patch embedding and window attention (csrc/swin.cu).

Every reference is computed in float64 from the very 16-bit inputs the kernel reads.  A kernel that rounds its result
once to the 16-bit output format is then within u * |ref| of it (u = 2^-8 for bf16, 2^-11 for fp16; fp16 adds half its
subnormal spacing, 2^-25, below 2^-14), plus what its fp32 arithmetic can contribute before that rounding.  Each bound
below is exactly that: one output rounding plus an fp32 term derived, in a comment, from the kernel's arithmetic.
The tests without the gpu marker check the float64 references themselves against torch and the CPU oracle."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from tests.emulate import emulate_pack_stem, emulate_pack_stem_s1

gpu = pytest.mark.gpu
DTYPES = [torch.bfloat16, torch.float16]
U = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11, torch.float64: 0.0}          # unit roundoff of the output format
SUB = {torch.bfloat16: 0.0, torch.float16: 2.0 ** -25, torch.float64: 0.0}              # half the fp16 subnormal spacing
U32 = 2.0 ** -24                                                                           # unit roundoff of fp32
GRID_CAP_THREADS = 148 * 16 * 256          # pointwise kernels: at most 16 CTAs of 256 threads per SM, grid-stride loop above


def _name(dt):
    return {torch.bfloat16: "bf16", torch.float16: "fp16"}[dt]


def _ops():
    from nerf_rpn_b200 import ops
    return ops


def assert_within(got, ref, tol, what):
    """|got - ref| <= tol elementwise (all float64 tensors of one shape); prints the worst error and its share of the bound."""
    got, ref, tol = got.double(), ref.double(), tol.double()
    assert got.shape == ref.shape
    assert torch.isfinite(got).all(), f"{what}: non-finite outputs"
    err = (got - ref).abs()
    ratio = (err / tol).max().item()
    i = int((err / tol).argmax())
    print(f"{what}: max |err| {err.max().item():.3e}, max |err|/bound {ratio:.3f} (at ref {ref.reshape(-1)[i].item():.4g})")
    assert ratio <= 1.0, f"{what}: |err| {err.reshape(-1)[i].item():.3e} > bound {tol.reshape(-1)[i].item():.3e} at flat index {i}"


def assert_bits(got, ref16, what):
    """Same 16-bit patterns (NaN compared as NaN)."""
    assert got.dtype == ref16.dtype and got.shape == ref16.shape, what
    a, b = got.view(torch.int16), ref16.view(torch.int16)
    nan = torch.isnan(got.float()) & torch.isnan(ref16.float())
    bad = (a != b) & ~nan
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.numel()} values differ, first at {bad.nonzero()[0].tolist()}"


# ------------------------------------------------------------------------------------------------ float64 references
def gn_ref64(x, gamma, beta, eps, relu, groups=32):
    """GroupNorm over channels-last (N, X, Y, Z, C): y, and per element the mean and rstd * |gamma| it used."""
    n, c = x.shape[0], x.shape[-1]
    xd = x.double().reshape(n, -1, groups, c // groups)
    mean = xd.mean(dim=(1, 3), keepdim=True)
    rstd = (((xd - mean) ** 2).mean(dim=(1, 3), keepdim=True) + eps).rsqrt()
    g = gamma.double().view(groups, c // groups)
    y = (xd - mean) * rstd * g + beta.double().view(groups, c // groups)
    if relu:
        y = y.clamp_min(0)
    full = lambda t: t.expand_as(xd).reshape(x.shape)
    return y.reshape(x.shape), full(mean), full(rstd * g.abs())


def ln_ref64(x, c, gamma, beta, eps):
    """LayerNorm over the first c channels of every row: y, and per element the row's rstd * |gamma| and mean |x|."""
    xd = x[..., :c].double()
    mean = xd.mean(-1, keepdim=True)
    rstd = (((xd - mean) ** 2).mean(-1, keepdim=True) + eps).rsqrt()
    y = (xd - mean) * rstd * gamma.double() + beta.double()
    return y, rstd * gamma.double().abs(), xd.abs().mean(-1, keepdim=True).expand_as(xd)


MERGE_ORDER = ((0, 0, 0), (1, 0, 0), (0, 1, 0), (1, 1, 0), (0, 0, 1), (1, 0, 1), (0, 1, 1), (1, 1, 1))   # (H, W, D) parities


def merge_gather64(x, c):
    """PatchMerging's gather (feature_extractor.py:661-685): zero-pad odd extents, concatenate the 8 parities in MERGE_ORDER."""
    xd = x[..., :c].double()
    H, W, D = xd.shape[1:4]
    xp = F.pad(xd, (0, 0, 0, D % 2, 0, W % 2, 0, H % 2))
    return torch.cat([xp[:, i::2, j::2, k::2, :] for (i, j, k) in MERGE_ORDER], -1)


def patch_embed_ref64(grid):
    """(N, 4, X, Y, Z) -> (N, X//4, Y//4, Z//4, 256) with channel ((c*4 + px)*4 + py)*4 + pz = grid[c, 4i+px, 4j+py, 4k+pz]:
    the input rows of Conv3d(4, C, kernel 4, stride 4) as a GEMM against weight.reshape(C, 256)."""
    n = grid.shape[0]
    H, W, D = (e // 4 for e in grid.shape[2:])
    g = grid.double()[:, :, :4 * H, :4 * W, :4 * D].reshape(n, 4, H, 4, W, 4, D, 4)
    return g.permute(0, 2, 4, 6, 1, 3, 5, 7).reshape(n, H, W, D, 256)


def rel_position_index(heads, shift):
    from nerf_rpn_b200.model.feature_extractor import ShiftedWindowAttention
    return ShiftedWindowAttention(heads * 32, [4, 4, 4], [shift] * 3, heads).relative_position_index.reshape(-1)


def attn_ref64(qkv, qkv_bias, table, heads, shift, rel_index, tc=False):
    """Shifted-window attention (window 4^3, head_dim 32) on an (N, H, W, D, 3C) grid of q | k | v rows, in float64, as
    oracle/net.py:_window_attention states it with the qkv projection already applied: the grid is zero-padded to whole windows
    AFTER the norm, so padded tokens carry q/k/v = qkv_bias; cyclic shift by -shift on every axis wider than one window; bias from
    the relative-position table; -100 between the 27 shift regions; softmax; un-shift; crop.

    tc=True models the tcgen05 kernel: padded tokens carry the bias rounded to the activation format, and the un-normalised
    probabilities exp(s - max) are rounded to it before the PV product (the 1/sum uses the unrounded ones).

    Returns (out, fp32 term of the bound), both (N, H, W, D, C).  The fp32 term, per output o = sum_j p_j v_j:
      * scores s_j: a 32-term fp32 dot, the scale, the table entry and the -100 mask, each rounded: |ds_j| <= 64 u32
        (scale sum_d |q_d k_jd| + |table| + 100 [masked]) (twice the first-order bound gamma_32 + 3 roundings);
      * e_j = __expf(s_j - max): the argument is rounded (u32 |s_j - max|, doubled for the log2(e) product) and ex2.approx has
        a relative error below 2^-22; softmax is shift invariant, so an error of the max cancels.  With eps_j = |ds_j| +
        2 u32 |s_j - max| + 2^-20 the output moves by at most sum_j p_j eps_j (|v_j| + |o|);
      * P V: at most 128 accumulated products (tcgen05: K = 128 over both stacked windows) and the 1/sum product:
        160 u32 sum_j p_j |v_j|;
      * tc=True: the kernel's e_j differs from the reference's by eps_j relative, so where e_j lies within eps_j e_j of a
        16-bit rounding midpoint the two may round to neighbouring values: one 16-bit ulp of e_j times |v_j| / sum for those j."""
    dt = qkv.dtype
    B, H, W, D, C3 = qkv.shape
    C, win = C3 // 3, 4
    dev = qkv.device
    bias = (qkv_bias.to(dt) if tc else qkv_bias).double().to(dev)
    PH, PW, PD = (-(-e // win) * win for e in (H, W, D))
    sh = [0 if win >= e else shift for e in (PH, PW, PD)]
    pad = (0, 0, 0, PD - D, 0, PW - W, 0, PH - H)
    real = F.pad(torch.ones((B, H, W, D, 1), dtype=torch.float64, device=dev), pad)
    xp = torch.where(real > 0, F.pad(qkv.double(), pad), bias)
    if sum(sh) > 0:
        xp = torch.roll(xp, shifts=(-sh[0], -sh[1], -sh[2]), dims=(1, 2, 3))
    nh, nw, nd = PH // win, PW // win, PD // win
    t = xp.view(B, nh, win, nw, win, nd, win, C3).permute(0, 1, 3, 5, 2, 4, 6, 7).reshape(-1, 64, 3, heads, 32).permute(2, 0, 3, 1, 4)
    q, k, v = t[0], t[1], t[2]                                   # (windows, heads, 64, 32)
    scale = 32 ** -0.5
    tb = table.double().to(dev)[rel_index.to(dev)].view(64, 64, heads).permute(2, 0, 1)
    s = (q @ k.transpose(-2, -1)) * scale + tb
    masked = torch.zeros((1, 64, 64), dtype=torch.float64, device=dev)
    if sum(sh) > 0:
        region = torch.zeros((PH, PW, PD), dtype=torch.float64, device=dev)
        cnt = 0
        for hs in ((0, -win), (-win, -sh[0]), (-sh[0], None)):
            for ws in ((0, -win), (-win, -sh[1]), (-sh[1], None)):
                for ds in ((0, -win), (-win, -sh[2]), (-sh[2], None)):
                    region[hs[0]:hs[1], ws[0]:ws[1], ds[0]:ds[1]] = cnt
                    cnt += 1
        region = region.view(nh, win, nw, win, nd, win).permute(0, 2, 4, 1, 3, 5).reshape(nh * nw * nd, 64)
        masked = (region.unsqueeze(1) != region.unsqueeze(2)).double()          # (windows per sample, 64, 64)
        s = (s.view(B, -1, heads, 64, 64) - 100.0 * masked[None, :, None]).view(-1, heads, 64, 64)
        masked = masked.repeat(B, 1, 1)
    m = s.amax(-1, keepdim=True)
    e = torch.exp(s - m)
    den = e.sum(-1, keepdim=True)
    o = ((e.to(dt).double() if tc else e) @ v) / den
    p = e / den
    ds = 64 * U32 * (scale * (q.abs() @ k.abs().transpose(-2, -1)) + tb.abs() + 100.0 * masked.unsqueeze(1))
    eps = ds + 2 * U32 * (s - m).abs() + 2.0 ** -20
    pe = p * eps
    term = pe @ v.abs() + pe.sum(-1, keepdim=True) * o.abs() + 160 * U32 * (p @ v.abs())
    if tc:
        mant, emin = (11, -14) if dt == torch.float16 else (8, -126)
        ulp = torch.exp2(torch.floor(torch.log2(e.clamp_min(1e-300))).clamp_min(emin) - (mant - 1))
        frac = e / ulp - torch.floor(e / ulp)
        near = (frac - 0.5).abs() * ulp <= eps * e
        term = term + ((near.double() * ulp) @ v.abs()) / den

    def unwindow(a):
        a = a.permute(0, 2, 1, 3).reshape(B, nh, nw, nd, win, win, win, C).permute(0, 1, 4, 2, 5, 3, 6, 7).reshape(B, PH, PW, PD, C)
        if sum(sh) > 0:
            a = torch.roll(a, shifts=(sh[0], sh[1], sh[2]), dims=(1, 2, 3))
        return a[:, :H, :W, :D, :]
    return unwindow(o), unwindow(term)


# ------------------------------------------------------------------------------------------------ reference self-checks (CPU)
def test_gn_reference_matches_torch():
    g = torch.Generator().manual_seed(0)
    x = (torch.randn((2, 5, 4, 3, 256), generator=g) * 3 + 0.7)
    gamma, beta = torch.rand(256, generator=g) + 0.5, torch.randn(256, generator=g)
    for relu in (False, True):
        want = F.group_norm(x.permute(0, 4, 1, 2, 3), 32, gamma, beta, 1e-5).permute(0, 2, 3, 4, 1)
        want = F.relu(want) if relu else want
        got, _, _ = gn_ref64(x, gamma, beta, 1e-5, relu)
        torch.testing.assert_close(got.float(), want, rtol=1e-5, atol=1e-5)


def test_ln_and_merge_references_match_torch():
    g = torch.Generator().manual_seed(1)
    x = torch.randn((2, 3, 5, 1, 40), generator=g) * 2 + 0.3
    gamma, beta = torch.rand(24, generator=g) + 0.5, torch.randn(24, generator=g)
    got, _, _ = ln_ref64(x, 24, gamma, beta, 1e-5)
    torch.testing.assert_close(got.float(), F.layer_norm(x[..., :24], (24,), gamma, beta, 1e-5), rtol=1e-5, atol=1e-5)
    # patch-merge order: channel part p of output (i, j, k) is input (2i + a, 2j + b, 2k + c) with (a, b, c) = MERGE_ORDER[p]
    H, W, D, c = 5, 4, 3, 2
    coord = torch.zeros((1, H, W, D, c), dtype=torch.float64)
    for h in range(H):
        for w in range(W):
            for d in range(D):
                coord[0, h, w, d] = torch.tensor([1 + h * 100 + w * 10 + d, -(1 + h * 100 + w * 10 + d)])
    m = merge_gather64(coord, c)
    assert m.shape == (1, 3, 2, 2, 8 * c)
    for i in range(3):
        for j in range(2):
            for k in range(2):
                for p, (a, b, cc) in enumerate(((0, 0, 0), (1, 0, 0), (0, 1, 0), (1, 1, 0), (0, 0, 1), (1, 0, 1), (0, 1, 1), (1, 1, 1))):
                    h, w, d = 2 * i + a, 2 * j + b, 2 * k + cc
                    want = [0.0, 0.0] if h >= H or w >= W or d >= D else [1 + h * 100 + w * 10 + d, -(1 + h * 100 + w * 10 + d)]
                    assert m[0, i, j, k, p * c:(p + 1) * c].tolist() == want


def test_patch_embed_reference_is_the_stride4_conv():
    g = torch.Generator().manual_seed(2)
    x = torch.rand((2, 4, 9, 13, 6), generator=g, dtype=torch.float64)
    w = torch.randn((8, 4, 4, 4, 4), generator=g, dtype=torch.float64)
    got = patch_embed_ref64(x) @ w.reshape(8, 256).t()
    torch.testing.assert_close(got, F.conv3d(x, w, stride=4).permute(0, 2, 3, 4, 1), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("dims,heads,shift", [((5, 7, 4), 2, 2), ((8, 3, 9), 1, 0), ((6, 6, 6), 2, 2)])
def test_attention_reference_matches_oracle(dims, heads, shift):
    """attn_ref64 + the projection == oracle/net.py:_window_attention (float32) with random qkv / proj weights."""
    from oracle import net as onet
    C = heads * 32
    g = torch.Generator().manual_seed(sum(dims) + heads)
    x = torch.randn((2, *dims, C), generator=g)
    sd = {"a.qkv.weight": torch.randn((3 * C, C), generator=g) / C ** 0.5, "a.qkv.bias": torch.randn(3 * C, generator=g) * 0.3,
          "a.proj.weight": torch.randn((C, C), generator=g) / C ** 0.5, "a.proj.bias": torch.randn(C, generator=g) * 0.1,
          "a.relative_position_bias_table": torch.randn((343, heads), generator=g) * 0.5,
          "a.relative_position_index": rel_position_index(heads, shift)}
    want = onet._window_attention(x, sd, "a", heads, shift)
    qkv = F.linear(x.double(), sd["a.qkv.weight"].double(), sd["a.qkv.bias"].double())
    o, term = attn_ref64(qkv, sd["a.qkv.bias"], sd["a.relative_position_bias_table"], heads, shift, sd["a.relative_position_index"])
    got = F.linear(o, sd["a.proj.weight"].double(), sd["a.proj.bias"].double())
    torch.testing.assert_close(got.float(), want, rtol=2e-5, atol=2e-5)
    assert (term > 0).all() and term.max().item() < 1e-3          # the fp32 term stays well below a bf16 rounding


def test_torch_max_pool_propagates_nan():
    """The semantics the pooling kernels follow: a NaN makes every window containing it NaN, and max_pool3d_with_indices records
    the NaN's position (the last NaN of the window in scan order)."""
    x = torch.arange(27.0).reshape(1, 1, 3, 3, 3)
    x[0, 0, 0, 0, 1] = float("nan")
    o, idx = F.max_pool3d(x, 3, 2, 1, return_indices=True)
    assert torch.isnan(o.flatten()[:2]).all() and idx.flatten()[:2].tolist() == [1, 1]
    assert torch.isnan(F.max_pool3d(x, 2, 2, ceil_mode=True).flatten()).tolist() == [True] + [False] * 7


# ------------------------------------------------------------------------------------------------ stem packing (bit-exact)
PACK_CASES = [((2, 7, 5, 9)), ((1, 1, 1, 1)), ((2, 1, 6, 3)), ((1, 96, 96, 96))]       # (N, X, Y, Z); 96^3: 903 k chunks > cap


@gpu
@pytest.mark.parametrize("layout", ["ncdhw", "dataset", "uint8"])
@pytest.mark.parametrize("shape", PACK_CASES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_pack_stem_input_bit_exact(dtype, shape, layout):
    ops = _ops()
    n, X, Y, Z = shape
    g = torch.Generator(device="cuda").manual_seed(X * 7 + Y * 3 + Z)
    if layout == "uint8":
        raw = torch.randint(0, 256, (n, X, Y, Z, 4), generator=g, device="cuda", dtype=torch.uint8)
        grid = raw.permute(0, 4, 1, 2, 3)
        ref_in = raw.float().div(255.0).permute(0, 4, 1, 2, 3).contiguous()          # datasets.py: .float() / 255.0
    else:
        raw = torch.randn((n, X, Y, Z, 4), generator=g, device="cuda") * 3
        grid = raw.permute(0, 4, 1, 2, 3) if layout == "dataset" else raw.permute(0, 4, 1, 2, 3).contiguous()
        ref_in = raw.permute(0, 4, 1, 2, 3).contiguous()
    got = ops.pack_stem_input(grid, dtype=dtype)
    if shape == PACK_CASES[-1]:
        assert got[..., 0].numel() * 8 > GRID_CAP_THREADS
    assert_bits(got, emulate_pack_stem(ref_in.cpu()).to(dtype).cuda(), f"pack_stem_input {layout} {tuple(shape)}")


S1_CASES = [(2, 7, 5, 9), (1, 1, 1, 1), (1, 3, 1, 8), (1, 45, 47, 43)]                 # 45x48x43x8 = 743 k chunks > cap


@gpu
@pytest.mark.parametrize("shape", S1_CASES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_pack_stem_input_s1_bit_exact(dtype, shape):
    ops = _ops()
    n, X, Y, Z = shape
    g = torch.Generator(device="cuda").manual_seed(X + Y + Z)
    grid = torch.randn((n, 4, X, Y, Z), generator=g, device="cuda") * 3
    got = ops.pack_stem_input_s1(grid, dtype=dtype)
    if shape == S1_CASES[-1]:
        assert got[..., 0].numel() * 8 > GRID_CAP_THREADS
    assert_bits(got, emulate_pack_stem_s1(grid.cpu()).to(dtype).cuda(), f"pack_stem_input_s1 {tuple(shape)}")


@gpu
@pytest.mark.parametrize("shape", [(1, 13, 11, 15), (2, 9, 6, 7)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_stem_s1_pack_and_conv(dtype, shape):
    """VGG stem Conv3d(4, 64, k7, s1, p3) through the stride-1 packing: pack, packing.pack_stem_s1_weight, conv3d_fprop (fp32 out)
    against F.conv3d in float64 on the same 16-bit operands.  Bound: the fp32 accumulator of each output takes 28 taps x 4 MMA
    k-steps = 112 additions and each k-step sums 16 products: at most 128 roundings of partial sums bounded by sum |x w|; doubled
    for MMA accumulation that truncates instead of rounding: 256 u32 sum |x| |w|."""
    from nerf_rpn_b200 import packing
    ops = _ops()
    n, X, Y, Z = shape
    g = torch.Generator(device="cuda").manual_seed(12 + X)
    x = torch.rand((n, 4, X, Y, Z), device="cuda", generator=g)
    w = torch.randn((64, 4, 7, 7, 7), device="cuda", generator=g) * 0.05
    packed = ops.pack_stem_input_s1(x, dtype=dtype)
    wp, taps = packing.pack_stem_s1_weight(w, dtype=dtype)
    y = torch.full((n, X, Y, Z, 64), float("nan"), dtype=torch.float32, device="cuda")
    a = ops.ConvLevelArgs(packed, y, n, (X, Y + 1, Z), (X, Y, Z), 64)
    ops.conv3d_fprop([a], wp.cuda(), torch.zeros(64, device="cuda"), 64, 64, taps, out_fp32=True)
    torch.cuda.synchronize()
    x64, w64 = x.to(dtype).double(), w.to(dtype).double()
    ref = F.conv3d(x64, w64, stride=1, padding=3).permute(0, 2, 3, 4, 1)
    mag = F.conv3d(x64.abs(), w64.abs(), stride=1, padding=3).permute(0, 2, 3, 4, 1)
    assert_within(y, ref, 256 * U32 * mag + 1e-30, f"stem s1 conv {_name(dtype)} {shape}")


# ------------------------------------------------------------------------------------------------ max-pooling (bit-exact)
POOL_CASES = [(2, 7, 5, 9, 64), (2, 10, 12, 8, 64), (1, 1, 1, 1, 64), (2, 1, 6, 3, 512), (1, 9, 4, 5, 512), (1, 80, 128, 128, 64)]


def _pool(ops, kind, x):
    """(kernel output, F.max_pool3d in float64 on the CPU) for a channels-last x."""
    xd = x.cpu().double().permute(0, 4, 1, 2, 3)
    if kind == "k3s2":
        return ops.maxpool3d_k3s2(x).cpu(), F.max_pool3d(xd, 3, 2, 1).permute(0, 2, 3, 4, 1)
    return ops.maxpool3d_k2s2_ceil(x).cpu(), F.max_pool3d(xd, 2, 2, ceil_mode=True).permute(0, 2, 3, 4, 1)


@gpu
@pytest.mark.parametrize("shape", POOL_CASES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("kind", ["k3s2", "k2s2_ceil"])
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_maxpool_vs_torch(dtype, kind, shape):
    """Odd / even / unit extents (odd extents run the clipped last window of ceil mode), C = 64 and 512, and the real ResNet stem
    output 80x128x128x64, whose 10.5 M output chunks are far above the grid cap.  A maximum is exact: bit-identical."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(sum(shape))
    x = torch.randn(shape, device="cuda", generator=g).to(dtype)
    got, ref = _pool(ops, kind, x)
    if shape == POOL_CASES[-1]:
        assert got.numel() // 8 > GRID_CAP_THREADS
    assert_bits(got, ref.to(dtype), f"maxpool {kind} {shape}")


def _special(dtype, shape, seed, nan, neg_inf_corner=True):
    """Values on a coarse grid (many repeated maxima), +-inf sprinkled in, optionally an all -inf corner and NaNs."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randint(-3, 4, shape, device="cuda", generator=g).float()
    r = torch.rand(shape, device="cuda", generator=g)
    x[r < 0.01] = float("inf")
    x[r > 0.99] = float("-inf")
    if neg_inf_corner:
        x[:, :3, :3, :3, :8] = float("-inf")
    if nan:
        x[(r > 0.3) & (r < 0.305)] = float("nan")
    return x.to(dtype)


@gpu
@pytest.mark.parametrize("kind", ["k3s2", "k2s2_ceil"])
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_maxpool_inf_and_ties(dtype, kind):
    ops = _ops()
    x = _special(dtype, (2, 9, 8, 7, 64), 5, nan=False)
    got, ref = _pool(ops, kind, x)
    assert_bits(got, ref.to(dtype), f"maxpool {kind} inf/ties")


@gpu
@pytest.mark.parametrize("kind", ["k3s2", "k2s2_ceil"])
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_maxpool_propagates_nan(dtype, kind):
    """F.max_pool3d propagates NaN: every window containing one is NaN."""
    ops = _ops()
    x = _special(dtype, (2, 9, 8, 7, 64), 6, nan=True)
    got, ref = _pool(ops, kind, x)
    assert torch.isnan(ref).any()
    assert_bits(got, ref.to(dtype), f"maxpool {kind} NaN")


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_maxpool_argmax_nan_and_ties_vs_autograd(dtype):
    """Training max-pool (csrc/train.cu): output and the recorded position -- checked through the backward gather -- follow
    max_pool3d_with_indices: the first maximum of a window in scan order, or its NaN.  dy are small integers and at most 8
    windows share an input, so every gradient sum is exact in both formats.  No window is entirely -inf (where torch's recorded
    position is implementation-defined)."""
    from nerf_rpn_b200._lib import check, lib
    L = lib()
    x = _special(dtype, (2, 9, 8, 7, 64), 7, nan=True, neg_inf_corner=False)
    n, dims, c = 2, (9, 8, 7), 64
    od = tuple((d - 1) // 2 + 1 for d in dims)
    out = torch.empty((n, *od, c), dtype=dtype, device="cuda")
    idx = torch.empty((n, *od, c), dtype=torch.uint8, device="cuda")
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    f16 = 1 if dtype == torch.float16 else 0
    check(L.nrpn_maxpool3d_k3s2_argmax(p(x), n, *dims, c, p(out), p(idx), f16, s), "maxpool_argmax")
    g = torch.Generator(device="cuda").manual_seed(8)
    dy = torch.randint(-8, 9, (n, *od, c), device="cuda", generator=g).to(dtype)
    dx = torch.empty_like(x)
    check(L.nrpn_maxpool3d_k3s2_backward(p(dy), p(idx), n, *dims, c, p(dx), f16, s), "maxpool_backward")
    torch.cuda.synchronize()
    x64 = x.cpu().double().permute(0, 4, 1, 2, 3).contiguous().requires_grad_(True)
    o64 = F.max_pool3d(x64, 3, 2, 1)
    assert torch.isnan(o64).any()
    assert_bits(out.cpu(), o64.detach().permute(0, 2, 3, 4, 1).to(dtype), "maxpool argmax forward")
    o64.backward(dy.cpu().double().permute(0, 4, 1, 2, 3))
    assert_bits(dx.cpu(), x64.grad.permute(0, 2, 3, 4, 1).to(dtype), "maxpool argmax backward")


# ------------------------------------------------------------------------------------------------ GroupNorm
FCOS_P2_P5 = [(50, 50, 32), (25, 25, 16), (13, 13, 8), (7, 7, 4)]       # config 3 (200x200x128 grid, strides 4..32)


@gpu
@pytest.mark.parametrize("relu", [False, True], ids=["linear", "relu"])
@pytest.mark.parametrize("case", ["p2_p5", "offset"])
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_groupnorm(dtype, case, relu):
    """FCOS-tower GroupNorm(32, 256) over batch 2: the four pyramid levels of config 3 in one launch (P2 has 80 000 voxels, so the
    stats kernel runs at its 512-CTA cap), and a launch of a 1x2x2 level with a 50x50x32 level whose inputs sit on a common offset
    (mean / std = 20).  Bound: one output rounding plus the fp32 apply step y = x * (gamma rstd) + (beta - mean gamma rstd): rstd
    and mean rounded to fp32, two products, a difference and the final fma are 6 roundings of terms bounded by
    (|x| + |mean|) rstd |gamma| + |beta|, doubled: 12 u32 of that.  The statistics must be accurate enough not to add to it.
    Two runs are bit-identical (fixed reduction order)."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(3 + DTYPES.index(dtype))
    if case == "p2_p5":
        levels = [(torch.randn((2, *d, 256), device="cuda", generator=g) * 3 + 0.7).to(dtype) for d in FCOS_P2_P5]
    else:
        levels = [(torch.randn((2, *d, 256), device="cuda", generator=g) + 20.0).to(dtype) for d in [(50, 50, 32), (1, 2, 2)]]
    gamma = torch.rand(256, device="cuda", generator=g) + 0.5
    beta = torch.randn(256, device="cuda", generator=g)
    work = [t.clone() for t in levels]
    ops.groupnorm_relu_(work, gamma, beta, 1e-5, relu)
    again = [t.clone() for t in levels]
    ops.groupnorm_relu_(again, gamma, beta, 1e-5, relu)
    torch.cuda.synchronize()
    for l, (x, w, a) in enumerate(zip(levels, work, again)):
        assert torch.equal(w, a), "fixed-order reductions: reproducible"
        ref, mean, scale = gn_ref64(x, gamma, beta, 1e-5, relu)
        tol = U[dtype] * ref.abs() + SUB[dtype] + 12 * U32 * ((x.double().abs() + mean.abs()) * scale + beta.double().abs())
        assert_within(w, ref, tol, f"groupnorm {_name(dtype)} {case} relu={relu} level {l} {tuple(x.shape[1:4])}")


# ------------------------------------------------------------------------------------------------ LayerNorm / patch merging
def _ln_tol(dtype, ref, scale, mabs, beta, n):
    """One output rounding plus the fp32 LayerNorm of an n-wide row: the mean is a sum of n / 32 values per lane and a 5-level
    shuffle tree (n / 32 + 5 roundings of partial sums bounded by sum |x|); the variance the same over (x - mean)^2, then rsqrtf
    (2 ulp), eps, the division and three products of the output.  (n / 32 + 16) u32 of |ref - beta| + rstd |gamma| mean |x| covers
    it, plus two roundings of |beta|."""
    b = beta.double()
    return U[dtype] * ref.abs() + SUB[dtype] + (n / 32 + 16) * U32 * ((ref - b).abs() + scale * mabs) + 2 * U32 * b.abs()


LN_WIDTHS = [(96, 128), (192, 192), (384, 384), (768, 768)]                       # Swin-S stage widths (C, row pitch)
LN_GRIDS = [(2, 5, 7, 3), (1, 1, 1, 1), (1, 3, 1, 9)]                          # 210, 1 and 27 tokens


@gpu
@pytest.mark.parametrize("grid", LN_GRIDS, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("c,ld", LN_WIDTHS, ids=lambda v: str(v))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_layernorm(dtype, c, ld, grid):
    """Every row has its own scale, std 1e-3 .. 10 (so eps = 1e-5 matters for some rows), and its own offset (|mean| up to
    ~8 std).  Pad channels [C, ld) of the input hold garbage that must not be read, those of the output a sentinel that must
    survive."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(c + sum(grid))
    x = torch.full((*grid, ld), 1e4, device="cuda")
    std = 10.0 ** (torch.rand((*grid, 1), device="cuda", generator=g) * 4 - 3)
    x[..., :c] = (torch.randn((*grid, c), device="cuda", generator=g) + torch.randn((*grid, 1), device="cuda", generator=g) * 3) * std
    x[0, 0, 0, 0, :c] = torch.randn(c, device="cuda", generator=g) * 2e-3                # a 1-token grid still gets a small row
    x = x.to(dtype)
    gamma = torch.rand(c, device="cuda", generator=g) + 0.5
    beta = torch.randn(c, device="cuda", generator=g)
    out = torch.full((*grid, ld), 7.0, device="cuda", dtype=dtype)
    ops.layernorm(x, out, c, gamma, beta, 1e-5)
    torch.cuda.synchronize()
    ref, scale, mabs = ln_ref64(x, c, gamma, beta, 1e-5)
    assert_within(out[..., :c], ref, _ln_tol(dtype, ref, scale, mabs, beta, c), f"layernorm {_name(dtype)} C={c} {grid}")
    assert (out[..., c:] == 7.0).all(), "pad channels [C, ld) must stay untouched"


MERGE_GRIDS = [(2, 5, 7, 3), (1, 1, 1, 1), (1, 4, 3, 6)]


@gpu
@pytest.mark.parametrize("grid", MERGE_GRIDS, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("c,ld", LN_WIDTHS[:3], ids=lambda v: str(v))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_patch_merge_ln(dtype, c, ld, grid):
    """The three Swin-S merges (C = 96 with row pitch 128, 192, 384: LayerNorm over 8C = 3 072, the widest row).  Odd extents
    zero-pad the missing parities; garbage in the input pad channels must not be read."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(c + 7 * sum(grid))
    x = torch.full((*grid, ld), -1e4, device="cuda")
    x[..., :c] = torch.randn((*grid, c), device="cuda", generator=g) * 2 + 0.3
    x = x.to(dtype)
    gamma = torch.rand(8 * c, device="cuda", generator=g) + 0.5
    beta = torch.randn(8 * c, device="cuda", generator=g)
    n, H, W, D = grid
    out = torch.full((n, (H + 1) // 2, (W + 1) // 2, (D + 1) // 2, 8 * c), float("nan"), device="cuda", dtype=dtype)
    ops.patch_merge_ln(x, out, c, gamma, beta, 1e-5)
    torch.cuda.synchronize()
    ref, scale, mabs = ln_ref64(merge_gather64(x, c), 8 * c, gamma, beta, 1e-5)
    assert_within(out, ref, _ln_tol(dtype, ref, scale, mabs, beta, 8 * c), f"patch_merge {_name(dtype)} C={c} {grid}")


# ------------------------------------------------------------------------------------------------ patch embedding (bit-exact)
@gpu
@pytest.mark.parametrize("shape", [(2, 21, 18, 14), (1, 4, 4, 4), (2, 7, 9, 5), (1, 201, 202, 130)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_patch_embed_pack_bit_exact(dtype, shape):
    """Extents not multiples of 4 are floored, as the stride-4 conv does; 201x202x130 (50x50x32 patches: 2.6 M chunks) runs the
    grid-stride loop."""
    ops = _ops()
    n, X, Y, Z = shape
    g = torch.Generator(device="cuda").manual_seed(X + Y + Z)
    grid = torch.randn((n, 4, X, Y, Z), device="cuda", generator=g) * 3
    out = torch.empty((n, X // 4, Y // 4, Z // 4, 256), device="cuda", dtype=dtype)
    ops.patch_embed_pack(grid, out)
    assert_bits(out, patch_embed_ref64(grid).to(dtype), f"patch_embed {shape}")


# ------------------------------------------------------------------------------------------------ window attention
ATTN_CASES = [
    # (N, H, W, D), heads, shift
    ((1, 12, 12, 12), 3, 2),      # 27 windows: the last pair of the tcgen05 kernel has one window
    ((1, 12, 12, 12), 3, 0),
    ((1, 50, 50, 32), 3, 2),      # config 3 stage 1: 1 352 windows, ~4.6 pairs per CTA (persistent loop, mbarrier phase flips)
    ((1, 50, 50, 32), 3, 0),
    ((1, 7, 7, 4), 24, 2),        # stage 4; padded D extent 4: only H and W shift
    ((1, 7, 7, 4), 24, 0),
    ((2, 9, 3, 10), 6, 2),        # batch 2; padded W extent 4: only H and D shift
]


@gpu
@pytest.mark.parametrize("dims,heads,shift", ATTN_CASES, ids=lambda v: "x".join(map(str, v)) if isinstance(v, tuple) else str(v))
@pytest.mark.parametrize("kernel", ["tcgen05", "cuda_core"])
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_window_attention(dtype, kernel, dims, heads, shift, monkeypatch):
    """Both kernels (NRPN_ATTN_TC=0 selects the CUDA-core one) against attn_ref64 (with the tcgen05 kernel's rounding of the
    probabilities and of the padded tokens' bias modelled for it).  Bound: one output rounding plus the fp32 term attn_ref64
    derives.  Heads are unit-variance q/k/v (scores of a few units), so softmax rows are neither one-hot nor flat."""
    ops = _ops()
    monkeypatch.setenv("NRPN_ATTN_TC", "1" if kernel == "tcgen05" else "0")
    C = heads * 32
    g = torch.Generator(device="cuda").manual_seed(4 + heads + shift)
    qkv = torch.randn((*dims, 3 * C), device="cuda", generator=g).to(dtype)
    qkv_bias = torch.randn(3 * C, device="cuda", generator=g) * 0.3
    table = torch.randn((343, heads), device="cuda", generator=g) * 0.5
    out = torch.full((*dims, C), float("nan"), device="cuda", dtype=dtype)
    ops.window_attention(qkv, out, qkv_bias, table, C, heads, shift)
    torch.cuda.synchronize()
    ref, term = attn_ref64(qkv, qkv_bias, table, heads, shift, rel_position_index(heads, shift), tc=kernel == "tcgen05")
    assert_within(out, ref, U[dtype] * ref.abs() + SUB[dtype] + term, f"window_attention {kernel} {_name(dtype)} {dims} h{heads} s{shift}")
