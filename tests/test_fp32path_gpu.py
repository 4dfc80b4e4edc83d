"""Kernel-level parity of the fp32-accuracy path (unet.set_precision("fp32"): engine_fp32.py, csrc/fp32path.cu and the _split
entry points of csrc/norm.cu) against float64 torch on the same fp32 inputs, at the shapes the engine issues at 64x64 and at
96x64 (portrait) latents, plus the engine end to end at 96x64.

An output carried as a (hi, lo) bf16 pair is compared as hi + lo: the pair represents y to 2^-16 |y|, so every bar has the form
|hi + lo - ref| <= 2^-16 |ref| + c max|ref|, with c taken from the kernel's fp32 arithmetic (u = 2^-24).  Every test prints the
value it measured next to its bar."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24          # fp32 unit roundoff
PAIR = 2.0 ** -16       # representation error of a (hi, lo) pair
GN_ENVELOPE = 30.0      # largest group |mean| / std asserted for GroupNorm: max(30, 4 x the measured maximum, see DESIGN.md)


@pytest.fixture(scope="module")
def models():
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import make_oracle_unet
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    oracle = make_oracle_unet(seed=0)
    ours = UNet2DConditionModel()
    ours.load_state_dict(oracle.state_dict(), strict=True)
    ours = ours.to(DEV).eval()
    return oracle, ours


def _pair(hi, lo):
    return hi.double() + lo.double()


def _excess(got, ref, scale=None):
    """max (|got - ref| - 2^-16 |ref|) / max|ref|: the c that the bar |got - ref| <= 2^-16 |ref| + c max|ref| needs."""
    got, ref = got.double(), ref.double()
    m = float(ref.abs().max()) if scale is None else scale
    return float(((got - ref).abs() - PAIR * ref.abs()).max()) / max(m, 1e-300)


def _nan(shape, dtype):
    return torch.full(shape, float("nan"), dtype=dtype, device=DEV)


# ---------------------------------------------------------------------------------------------------------------------------------
# split_hi_lo
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [8, 8 * 12345, 2 * 6144 * 1280])
def test_split_hi_lo_bit_exact(n):
    from b200sd import ops
    g = torch.Generator(device=DEV).manual_seed(n)
    mag = 10.0 ** (torch.rand(n, generator=g, device=DEV) * 60 - 30)          # |x| from 1e-30 to 1e30
    sign = torch.where(torch.rand(n, generator=g, device=DEV) < 0.5, -1.0, 1.0)
    x = (mag * sign).float()
    x[0] = 0.0
    if n > 1:
        x[1] = -0.0
    if n > 16:
        x[2:10] = torch.tensor([1e-30, -1e-30, 1e30, -1e30, 1.0, -1.0, 3.0e38 / 1.1, 1.0 + 2 ** -8], device=DEV)
    hi, lo = _nan((n,), torch.bfloat16), _nan((n,), torch.bfloat16)
    ops.split_hi_lo(x, hi, lo)
    want_hi = x.bfloat16()
    assert torch.equal(hi, want_hi)
    assert torch.equal(lo, (x - want_hi.float()).bfloat16())
    err = ((_pair(hi, lo) - x.double()).abs() - PAIR * x.double().abs()).max()
    assert float(err) <= 0.0


# ---------------------------------------------------------------------------------------------------------------------------------
# geglu_f32
# ---------------------------------------------------------------------------------------------------------------------------------
GEGLU_C = 2.0 ** -21


@pytest.mark.parametrize("Cc", [320, 640, 1280])
@pytest.mark.parametrize("rows", [1, 2 * 4096, 2 * 6144, 2 * 1024, 2 * 1536, 2 * 256, 2 * 384, 2 * 64, 2 * 96])
def test_geglu_f32(rows, Cc):
    from b200sd import ops
    ch = 4 * Cc
    g = torch.Generator(device=DEV).manual_seed(rows * 7 + Cc)
    u = torch.empty(rows, 2 * ch, device=DEV)
    u[:, :ch] = torch.randn(rows, ch, generator=g, device=DEV) * 3
    u[:, ch:] = torch.rand(rows, ch, generator=g, device=DEV) * 16 - 8          # gates in [-8, 8]: both erf tails
    hi, lo = _nan((rows, ch), torch.bfloat16), _nan((rows, ch), torch.bfloat16)
    ops.geglu_f32(u, hi, lo)
    v, gate = u[:, :ch].double(), u[:, ch:].double()
    ref = v * 0.5 * gate * (1 + torch.erf(gate / math.sqrt(2)))
    c = _excess(_pair(hi, lo), ref)
    print(f"geglu_f32 rows={rows} C_half={ch}: c = {c:.3g} (bar {GEGLU_C:.3g})")
    assert c <= GEGLU_C


# ---------------------------------------------------------------------------------------------------------------------------------
# attention_f32
# ---------------------------------------------------------------------------------------------------------------------------------
def _attn_ref(q, k, v, scale):
    """float64 softmax(q k^T scale) v over [B, S, H, D] views, in query chunks; also returns max_ij scale sum_c |q_c k_c|."""
    B, Sq, H, D = q.shape
    out = torch.empty(B, Sq, H, D, dtype=torch.float64, device=DEV)
    amax = 0.0
    kd, vd = k.double().permute(0, 2, 1, 3), v.double().permute(0, 2, 1, 3)
    for i in range(0, Sq, 512):
        qd = q[:, i:i + 512].double().permute(0, 2, 1, 3)
        s = qd @ kd.transpose(-1, -2) * scale
        out[:, i:i + 512] = (torch.softmax(s, -1) @ vd).permute(0, 2, 1, 3)
        amax = max(amax, float((qd.abs() @ kd.abs().transpose(-1, -2)).max()) * scale)
    return out, amax


def _attn_bar(amax, skv):
    """Score error ~u sum|q k| scale per probability (relative), fp32 accumulation of up to Skv terms: c max|v|."""
    return U * (32 + 4 * amax + 4 * math.sqrt(skv))


def _attn_case(batch, heads, Sq, Skv, d, *, fused_qkv, sharp=4.0, ramp=8.0, seed=0):
    """Run attention_f32 with the engine's strides (fused qkv: ldq = ldk = ldv = 3C; cross: q [.., C], kv [.., 2C]) into an
    output with NaN sentinel rows after Sq and sentinel columns after C; returns (c measured, bar)."""
    from b200sd import ops
    C = heads * d
    g = torch.Generator(device=DEV).manual_seed(seed)
    scale = d ** -0.5
    qn = torch.randn(batch, Sq, heads, d, generator=g, device=DEV) * math.sqrt(sharp)
    kn = torch.randn(batch, Skv, heads, d, generator=g, device=DEV) * math.sqrt(sharp)
    vn = torch.randn(batch, Skv, heads, d, generator=g, device=DEV)
    # a ramp along one direction: later keys score higher, so each row's maximum sits in the last key tile and every new tile
    # rescales the running output
    dirn = torch.ones(d, device=DEV) / math.sqrt(d)
    qn = qn + ramp * dirn
    kn = kn + (torch.arange(Skv, device=DEV, dtype=torch.float32) / max(Skv - 1, 1) * ramp)[None, :, None, None] * dirn
    if fused_qkv:
        # one [rows, 3C] buffer as the engine's qkv GEMM writes it (q | k | v); at Sq != Skv, q and k | v in two such buffers
        qbuf = torch.zeros(batch, Sq, 3 * C, device=DEV)
        kvbuf = qbuf if Sq == Skv else torch.zeros(batch, Skv, 3 * C, device=DEV)
        qbuf[..., :C] = qn.reshape(batch, Sq, C)
        kvbuf[..., C:2 * C] = kn.reshape(batch, Skv, C)
        kvbuf[..., 2 * C:] = vn.reshape(batch, Skv, C)
        q_t, k_t, v_t, ldq, ldk, ldv, k_off, v_off = qbuf, kvbuf, kvbuf, 3 * C, 3 * C, 3 * C, C, 2 * C
    else:
        q_t = qn.reshape(batch * Sq, C).contiguous()
        kv = torch.cat([kn.reshape(batch, Skv, C), vn.reshape(batch, Skv, C)], -1).contiguous()
        k_t, v_t, ldq, ldk, ldv, k_off, v_off = kv, kv, C, 2 * C, 2 * C, 0, C
    ldo = C + 8
    out = _nan((batch * Sq + 3, ldo), torch.float32)
    ops.attention_f32(q_t, k_t, v_t, out, batch, heads, Sq, Skv, d, scale, ldq=ldq, ldk=ldk, ldv=ldv, ldo=ldo, k_off=k_off,
                      v_off=v_off)
    assert torch.isnan(out[batch * Sq:]).all(), "attention_f32 wrote past the last query row"
    assert torch.isnan(out[:, C:]).all(), "attention_f32 wrote past column C"
    got = out[:batch * Sq, :C].reshape(batch, Sq, heads, d)
    ref, amax = _attn_ref(qn, kn, vn, scale)
    vmax = float(vn.abs().max())
    c = float((got.double() - ref).abs().max()) / vmax
    return c, _attn_bar(amax, Skv)


ENGINE_ATTN = [(4096, 40), (1024, 80), (256, 160), (64, 160), (6144, 40), (1536, 80), (384, 160), (96, 160)]


@pytest.mark.parametrize("S,d", ENGINE_ATTN)
def test_attention_f32_engine_self_attention(S, d):
    c, bar = _attn_case(2, 8, S, S, d, fused_qkv=True, seed=S)
    print(f"attention_f32 self Sq=Skv={S} d={d}: |err| = {c:.3g} max|v| (bar {bar:.3g})")
    assert c <= bar


@pytest.mark.parametrize("S,d", ENGINE_ATTN)
def test_attention_f32_engine_cross_attention(S, d):
    c, bar = _attn_case(2, 8, S, 77, d, fused_qkv=False, seed=S + 1)
    print(f"attention_f32 cross Sq={S} Skv=77 d={d}: |err| = {c:.3g} max|v| (bar {bar:.3g})")
    assert c <= bar


@pytest.mark.parametrize("d", [8, 16, 32, 40, 64, 80, 128, 160])
def test_attention_f32_every_head_dim_at_tile_edges(d):
    worst, where = 0.0, None
    for Sq in (1, 63, 65, 129):
        for Skv in (1, 63, 64, 65, 77):
            for fused in (True, False):
                c, bar = _attn_case(3, 2, Sq, Skv, d, fused_qkv=fused, seed=Sq * 100 + Skv)
                assert c <= bar, f"d={d} Sq={Sq} Skv={Skv} fused={fused}: {c:.3g} > {bar:.3g}"
                if where is None or c / bar > worst:
                    worst, where = c / bar, (Sq, Skv, fused, c)
    print(f"attention_f32 d={d} edges: worst (Sq, Skv, fused, |err| / max|v|) = {where} at {worst:.2f} of its bar")


def test_attention_f32_exponentials_in_the_underflow_tail():
    """Two keys with scores 0 and x, x in [-86, -20], V = (0, 1): each output is exp(x) / (1 + exp(x)) = exp(x) to fp32, so the
    kernel's exponential must be as accurate as expf (<= 2 ulp) down to the fp32 normal range."""
    from b200sd import ops
    d, Sq = 8, 512
    x = torch.linspace(-86.0, -20.0, Sq, device=DEV)
    q = torch.zeros(Sq, d, device=DEV)
    q[:, 0] = x
    k = torch.zeros(2, d, device=DEV)
    k[1, 0] = 1.0                                     # score of key 1 = x exactly, key 0 = 0
    v = torch.zeros(2, d, device=DEV)
    v[1] = 1.0
    out = _nan((Sq, d), torch.float32)
    ops.attention_f32(q, k, v, out, 1, 1, Sq, 2, d, 1.0)
    ref = torch.exp(x.double())[:, None] / (1 + torch.exp(x.double())[:, None])
    rel = float(((out.double() - ref).abs() / ref).max())
    print(f"attention_f32 underflow tail: max relative error {rel:.3g} (bar {2 ** -21:.3g})")
    assert rel <= 2.0 ** -21


# ---------------------------------------------------------------------------------------------------------------------------------
# small_linear_f32
# ---------------------------------------------------------------------------------------------------------------------------------
def _silu64(t):
    return t * torch.sigmoid(t)


@pytest.fixture(scope="module")
def n_tp():
    from b200sd.unet import UNet2DConditionModel
    return UNet2DConditionModel()._tproj_offsets()[1]


@pytest.mark.parametrize("NK", [(1280, 320), (1280, 1280), ("n_tp", 1280), (7, 33)])
@pytest.mark.parametrize("batch", [1, 2, 8])
def test_small_linear_f32(batch, NK, n_tp):
    from b200sd import ops
    N, K = NK
    N = n_tp if N == "n_tp" else N
    g = torch.Generator(device=DEV).manual_seed(N * 31 + K + batch)
    x = torch.randn(batch, K, generator=g, device=DEV) * 2
    w = torch.randn(N, K, generator=g, device=DEV) / math.sqrt(K)
    b = torch.randn(N, generator=g, device=DEV)
    worst = 0.0
    for bias in (b, None):
        for silu_in in (False, True):
            for silu_out in (False, True):
                out = _nan((batch, N), torch.float32)
                ops.small_linear_f32(x, w, bias, silu_in=silu_in, silu_out=silu_out, out=out)
                xin = _silu64(x.double()) if silu_in else x.double()
                pre = xin @ w.double().T + (bias.double() if bias is not None else 0.0)
                ref = _silu64(pre) if silu_out else pre
                # sequential fp32 sums of ceil(K / 32) terms per lane + a 5-level shuffle tree + bias, silu: gamma_n u sum|x w|
                mag = xin.abs() @ w.double().abs().T + (bias.double().abs() if bias is not None else 0.0)
                bar = (math.ceil(K / 32) + 10) * U * mag + 4 * U * ref.abs()
                err = (out.double() - ref).abs()
                worst = max(worst, float((err / bar).max()))
                assert (err <= bar).all(), (bias is None, silu_in, silu_out, float((err / bar).max()))
    print(f"small_linear_f32 batch={batch} N={N} K={K}: worst |err| at {worst:.3f} of the gamma_n bound")


# ---------------------------------------------------------------------------------------------------------------------------------
# layernorm_split
# ---------------------------------------------------------------------------------------------------------------------------------
def _ln_bar(r):
    """fp32 mean (its error ~u r std per row), centred two-pass variance, rstd, affine: c = u (16 + 8 r)."""
    return U * (16 + 8 * r)


@pytest.mark.parametrize("C", [64, 320, 640, 1280])
@pytest.mark.parametrize("rows", [1, 3, 517, 2 * 6144])
def test_layernorm_split(rows, C):
    from b200sd import ops
    g = torch.Generator(device=DEV).manual_seed(rows + C)
    gamma = 1 + 0.2 * torch.randn(C, generator=g, device=DEV)
    beta = 0.2 * torch.randn(C, generator=g, device=DEV)
    for r in (0.0, 1.0, 10.0, 100.0):
        std = torch.rand(rows, 1, generator=g, device=DEV) * 4 + 0.1
        sign = torch.where(torch.rand(rows, 1, generator=g, device=DEV) < 0.5, -1.0, 1.0)
        x = (torch.randn(rows, C, generator=g, device=DEV) + r * sign) * std
        hi, lo = _nan((rows, C), torch.bfloat16), _nan((rows, C), torch.bfloat16)
        ops.layernorm_split(x, gamma, beta, hi, lo, eps=1e-5)
        ref = F.layer_norm(x.double(), (C,), gamma.double(), beta.double(), 1e-5)
        xd = x.double()
        r_meas = float((xd.mean(1).abs() / xd.std(1, unbiased=False)).max())
        c = _excess(_pair(hi, lo), ref)
        print(f"layernorm_split rows={rows} C={C} mean/std<={r_meas:.3g}: c = {c:.3g} (bar {_ln_bar(r_meas):.3g})")
        assert c <= _ln_bar(r_meas), (r, c)


# ---------------------------------------------------------------------------------------------------------------------------------
# groupnorm_silu_split
# ---------------------------------------------------------------------------------------------------------------------------------
def _gn_fused(hw, C, groups=32):
    """Mirror of b200sd_groupnorm_silu_split's choice between gn_fused_kernel and the gn_stats + gn_apply fallback."""
    cpg = C // groups
    G = 1
    while (G * cpg) % 8 != 0 and G < groups:
        G *= 2
    while G * 2 <= groups and groups % (G * 2) == 0 and G * cpg < 32:
        G *= 2
    Cg = G * cpg
    return Cg % 8 == 0 and groups % G == 0 and Cg // 8 <= 512 and hw * C <= 3000000


def _gn_bar(r):
    """fp32 per-thread and in-CTA sums of x and x^2 (the variance loses ~u (1 + r^2) relative), fp32 affine (~u r): r = group
    |mean| / std."""
    return U * (16 + 8 * r + 2 * r * r)


def _gn_run(x0, x1, hw, batch, silu, eps, raw):
    """Run groupnorm_silu_split with NaN-filled outputs; check raw_out / raw_lo bit-exactly; return (hi + lo, float64 reference,
    largest group |mean| / std of the input)."""
    from b200sd import ops
    C0 = x0.shape[1]
    C = C0 + (x1.shape[1] if x1 is not None else 0)
    g = torch.Generator(device=DEV).manual_seed(C + hw)
    gamma = 1 + 0.2 * torch.randn(C, generator=g, device=DEV)
    beta = 0.2 * torch.randn(C, generator=g, device=DEV)
    hi, lo = _nan((batch * hw, C), torch.bfloat16), _nan((batch * hw, C), torch.bfloat16)
    rh, rl = (_nan((batch * hw, C), torch.bfloat16), _nan((batch * hw, C), torch.bfloat16)) if raw else (None, None)
    ops.groupnorm_silu_split(x0, x1, gamma, beta, hi, lo, batch, hw, 32, eps, silu, raw_out=rh, raw_lo=rl)
    x = torch.cat([x0, x1], 1) if x1 is not None else x0
    if raw:
        assert torch.equal(rh, x.bfloat16())
        assert torch.equal(rl, (x - rh.float()).bfloat16())
    xd = x.double().reshape(batch, hw, C).permute(0, 2, 1)
    ref = F.group_norm(xd, 32, gamma.double(), beta.double(), eps)
    if silu:
        ref = _silu64(ref)
    ref = ref.permute(0, 2, 1).reshape(batch * hw, C)
    grp = xd.reshape(batch, 32, -1)
    r = float((grp.mean(-1).abs() / grp.std(-1, unbiased=False)).max())
    return _pair(hi, lo), ref, r


@pytest.fixture(scope="module")
def gn_signatures(models):
    """Every groupnorm_silu_split call EngineF32 issues in one eager forward at 64x64 and 96x64 latents, batch 2."""
    from b200sd import ops
    _, ours = models
    seen = set()
    real = ops.groupnorm_silu_split

    def spy(x0, x1, gamma, beta, out, out_lo, batch, hw, groups=32, eps=1e-5, silu=True, raw_out=None, raw_lo=None):
        seen.add((hw, x0.shape[1], x1.shape[1] if x1 is not None else 0, bool(silu), float(eps), raw_out is not None,
                  raw_lo is not None, groups))
        return real(x0, x1, gamma, beta, out, out_lo, batch, hw, groups, eps, silu, raw_out=raw_out, raw_lo=raw_lo)

    ours.set_precision("fp32")
    ours.use_cuda_graph = False
    ops.groupnorm_silu_split = spy
    try:
        with torch.no_grad():
            for H, W in ((64, 64), (96, 64)):
                ours(torch.randn(2, 4, H, W, device=DEV), torch.tensor([999, 37], device=DEV), torch.randn(2, 77, 768, device=DEV))
    finally:
        ops.groupnorm_silu_split = real
        ours.use_cuda_graph = True
    return sorted(seen)


def test_groupnorm_split_every_engine_signature(gn_signatures):
    paths = {_gn_fused(hw, c0 + c1) for hw, c0, c1, *_ in gn_signatures}
    assert paths == {True, False}, "the engine's GroupNorm calls no longer cover both the fused kernel and the fallback"
    g = torch.Generator(device=DEV).manual_seed(5)
    for hw, c0, c1, silu, eps, raw, raw_lo, groups in gn_signatures:
        assert groups == 32 and raw == raw_lo
        for batch in (1, 2):
            x0 = torch.randn(batch * hw, c0, generator=g, device=DEV) * 1.5 + 0.5
            x1 = torch.randn(batch * hw, c1, generator=g, device=DEV) * 0.7 - 0.3 if c1 else None
            got, ref, r = _gn_run(x0, x1, hw, batch, silu, eps, raw)
            c = _excess(got, ref)
            path = "fused" if _gn_fused(hw, c0 + c1) else "fallback"
            print(f"groupnorm_split hw={hw} C={c0}+{c1} silu={silu} eps={eps:g} raw={raw} batch={batch} ({path}, mean/std<={r:.2g}):"
                  f" c = {c:.3g} (bar {_gn_bar(r):.3g})")
            assert c <= _gn_bar(r), (hw, c0, c1, batch, c)


@pytest.mark.parametrize("hw,C", [(4096, 320), (4096, 960)], ids=["fused", "fallback"])
def test_groupnorm_split_mean_over_std_sweep(hw, C):
    """Groups whose mean is r times their std: asserted up to the envelope, printed beyond it."""
    assert _gn_fused(hw, C) == (C == 320)
    g = torch.Generator(device=DEV).manual_seed(C)
    for r in (0.0, 1.0, 3.0, 10.0, 30.0, 100.0, 300.0):
        sign = torch.where(torch.rand(1, C, generator=g, device=DEV) < 0.5, -1.0, 1.0).reshape(32, -1)[:, :1]
        sign = sign.expand(32, C // 32).reshape(1, C)              # one sign per group
        x = torch.randn(2 * hw, C, generator=g, device=DEV) + r * sign
        got, ref, r_meas = _gn_run(x, None, hw, 2, True, 1e-5, False)
        c = _excess(got, ref)
        inside = r <= GN_ENVELOPE
        print(f"groupnorm_split {'fused' if C == 320 else 'fallback'} mean/std={r:g}: c = {c:.3g}"
              + (f" (bar {_gn_bar(r_meas):.3g})" if inside else " (beyond the envelope: not asserted)"))
        if inside:
            assert c <= _gn_bar(r_meas), (r, c)


@pytest.mark.parametrize("hw,C", [(1024, 320), (6144, 640)], ids=["fused", "fallback"])
def test_groupnorm_split_statistics_exact_on_exact_sums(hw, C):
    """Integer inputs 100 + {-1, 0, 1}: every fp32 partial sum of x and x^2 is exact at these shapes (< 2^24 per CTA and group),
    so the statistics must be exact to the final rounding, even at mean / std ~ 120, and the only error left is the fp32
    affine (~u r).  Evaluating the final E[x^2] - mean^2 in fp32 would cost ~u r^2."""
    assert _gn_fused(hw, C) == (C == 320)
    g = torch.Generator(device=DEV).manual_seed(hw)
    x = 100.0 + torch.randint(-1, 2, (2 * hw, C), generator=g, device=DEV).float()
    got, ref, r = _gn_run(x, None, hw, 2, False, 1e-5, False)
    c = _excess(got, ref)
    bar = U * (16 + 8 * r)
    print(f"groupnorm_split exact sums {'fused' if C == 320 else 'fallback'} mean/std={r:.3g}: c = {c:.3g} (bar {bar:.3g})")
    assert c <= bar


def test_groupnorm_split_rejects_mixed_source_dtypes():
    from b200sd import ops
    from b200sd._lib import B200SDError
    x0 = torch.randn(64, 32, device=DEV)
    x1 = torch.randn(64, 32, device=DEV).bfloat16()
    g, b = torch.ones(64, device=DEV), torch.zeros(64, device=DEV)
    hi, lo = torch.empty(64, 64, dtype=torch.bfloat16, device=DEV), torch.empty(64, 64, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(B200SDError, match="same dtype"):
        ops.groupnorm_silu_split(x0, x1, g, b, hi, lo, 1, 64, 32)


def test_groupnorm_split_workspace_is_per_stream():
    """The fallback keeps arrival counters and partials in its workspace: two streams must not share one."""
    from b200sd import ops
    x = torch.randn(2 * 4096, 960, device=DEV)
    g, b = torch.ones(960, device=DEV), torch.zeros(960, device=DEV)
    outs = [torch.empty(2 * 4096, 960, dtype=torch.bfloat16, device=DEV) for _ in range(4)]
    ops.groupnorm_silu_split(x, None, g, b, outs[0], outs[1], 2, 4096, 32)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.groupnorm_silu_split(x, None, g, b, outs[2], outs[3], 2, 4096, 32)
        ws_side = ops._ws_cache[(("gn", side.cuda_stream), torch.cuda.current_device())]
    torch.cuda.current_stream().wait_stream(side)
    ws_main = ops._ws_cache[(("gn", torch.cuda.current_stream().cuda_stream), torch.cuda.current_device())]
    assert ws_side.data_ptr() != ws_main.data_ptr()
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[2]) and torch.equal(outs[1], outs[3])


# ---------------------------------------------------------------------------------------------------------------------------------
# the 3-term product: EngineF32._gemm2's two ops.gemm launches on weights packed by _pack_lin / _pack_conv
# ---------------------------------------------------------------------------------------------------------------------------------
K3 = 3.0    # A and W each carried to 2^-16 relative, plus the dropped A_lo W_lo term: |err| <= 3 2^-16 (|A| |W|^T)


def _gemm2(a, w12, out, *, bias=None, residual=None, conv=None, rowbias=None):
    """EngineF32._gemm2 on an fp32 operand a (split into (hi, lo) by split_hi_lo first, as the engine's producers do)."""
    from b200sd import ops
    a_hi, a_lo = torch.empty_like(a, dtype=torch.bfloat16), torch.empty_like(a, dtype=torch.bfloat16)
    ops.split_hi_lo(a, a_hi, a_lo)
    w1, w2 = w12
    args = ops.gemm(a_hi, w1, out, a1=a_lo, bias=bias, residual=residual, conv=conv, launch=False)
    if rowbias is not None:
        args.rowbias, args.ldrb, args.rows_per_image = rowbias
    ops.gemm_run(args)
    ops.gemm(a_hi, w2, out, residual=out, conv=conv)
    torch.cuda.synchronize()


def _k_measured(out, ref, aw, extra):
    """The k with |out - ref| <= k 2^-16 (|A||W|^T) + 2^-20 (|bias| + |rowbias| + |residual|)."""
    err = (out.double() - ref).abs() - 2.0 ** -20 * extra
    return float((err / (PAIR * aw)).max())


LINEAR_CASES = [(2 * 6144, 320, 320), (2 * 6144, 960, 320), (2 * 6144, 2560, 320), (2 * 6144, 320, 1280),
                (2 * 96, 1280, 1280), (2 * 96, 3840, 1280), (2 * 96, 10240, 1280), (2 * 96, 1280, 5120), (2 * 77, 2560, 768)]


@pytest.mark.parametrize("M,N,K", LINEAR_CASES)
def test_three_term_linear(M, N, K):
    from b200sd.engine_fp32 import _pack_lin
    g = torch.Generator(device=DEV).manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g, device=DEV)
    w = torch.randn(N, K, generator=g, device=DEV) / math.sqrt(K)
    bias = torch.randn(N, generator=g, device=DEV)
    res = torch.randn(M, N, generator=g, device=DEV) * 3
    out = _nan((M, N), torch.float32)
    _gemm2(a, _pack_lin(w), out, bias=bias, residual=res)
    ad, wd = a.double(), w.double()
    ref = ad @ wd.T + bias.double() + res.double()
    aw = ad.abs() @ wd.abs().T
    k = _k_measured(out, ref, aw, bias.double().abs() + res.double().abs())
    print(f"3-term linear M={M} N={N} K={K} (+bias +residual): k = {k:.3g} (bar {K3})")
    assert k <= K3


CONV_CASES = [(2, 96, 64, 320, 320), (2, 12, 8, 1280, 1280)]


@pytest.mark.parametrize("B,H,W,Cin,Cout", CONV_CASES)
def test_three_term_conv3x3_with_time_embedding_row(B, H, W, Cin, Cout):
    """conv1 of a resnet: bias + the per-image time-embedding row (rowbias pointer into the concatenated time_emb_proj output)."""
    from b200sd.engine_fp32 import _pack_conv
    g = torch.Generator(device=DEV).manual_seed(H * Cin)
    x = torch.randn(B, Cin, H, W, generator=g, device=DEV)
    w = torch.randn(Cout, Cin, 3, 3, generator=g, device=DEV) / math.sqrt(9 * Cin)
    bias = torch.randn(Cout, generator=g, device=DEV)
    n_tp, off = Cout + 320, 200
    tproj = torch.randn(B, n_tp, generator=g, device=DEV)
    a = x.permute(0, 2, 3, 1).reshape(B * H * W, Cin).contiguous()
    out = _nan((B * H * W, Cout), torch.float32)
    _gemm2(a, _pack_conv(w), out, bias=bias, conv=(B, H, W), rowbias=(tproj.data_ptr() + off * 4, n_tp, H * W))
    rb = tproj[:, off:off + Cout].double()
    ref = F.conv2d(x.double(), w.double(), padding=1) + bias.double()[None, :, None, None] + rb[:, :, None, None]
    aw = F.conv2d(x.double().abs(), w.double().abs(), padding=1)
    to_rows = lambda t: t.permute(0, 2, 3, 1).reshape(B * H * W, Cout)
    extra = to_rows(bias.double().abs()[None, :, None, None] + rb.abs()[:, :, None, None] + torch.zeros_like(aw))
    k = _k_measured(out, to_rows(ref), to_rows(aw), extra)
    print(f"3-term conv3x3 ({B}, {H}, {W}, {Cin}->{Cout}) +bias +time row: k = {k:.3g} (bar {K3})")
    assert k <= K3


def test_three_term_conv3x3_with_residual():
    """conv2 of a resnet: bias + the fp32 residual (shortcut) in the first launch's epilogue."""
    from b200sd.engine_fp32 import _pack_conv
    B, H, W, Cin, Cout = 2, 24, 16, 640, 1280
    g = torch.Generator(device=DEV).manual_seed(11)
    x = torch.randn(B, Cin, H, W, generator=g, device=DEV)
    w = torch.randn(Cout, Cin, 3, 3, generator=g, device=DEV) / math.sqrt(9 * Cin)
    bias = torch.randn(Cout, generator=g, device=DEV)
    res = torch.randn(B * H * W, Cout, generator=g, device=DEV)
    out = _nan((B * H * W, Cout), torch.float32)
    _gemm2(x.permute(0, 2, 3, 1).reshape(B * H * W, Cin).contiguous(), _pack_conv(w), out, bias=bias, residual=res, conv=(B, H, W))
    to_rows = lambda t: t.permute(0, 2, 3, 1).reshape(B * H * W, Cout)
    ref = to_rows(F.conv2d(x.double(), w.double(), padding=1)) + bias.double() + res.double()
    aw = to_rows(F.conv2d(x.double().abs(), w.double().abs(), padding=1))
    k = _k_measured(out, ref, aw, bias.double().abs() + res.double().abs())
    print(f"3-term conv3x3 ({B}, {H}, {W}, {Cin}->{Cout}) +bias +residual: k = {k:.3g} (bar {K3})")
    assert k <= K3


def test_three_term_downsample_im2col_s2():
    """Downsample2D as EngineF32 runs it: split, im2col (stride 2, pad 1) of hi and lo, then a linear on [Cout][9 Cin] weights."""
    from b200sd import ops
    from b200sd.engine_fp32 import _pack_lin
    B, H, W, Cc = 2, 96, 64, 320
    g = torch.Generator(device=DEV).manual_seed(12)
    x = torch.randn(B, Cc, H, W, generator=g, device=DEV)
    w = torch.randn(Cc, Cc, 3, 3, generator=g, device=DEV) / math.sqrt(9 * Cc)
    bias = torch.randn(Cc, generator=g, device=DEV)
    a = x.permute(0, 2, 3, 1).reshape(B * H * W, Cc).contiguous()
    xh, xl = torch.empty_like(a, dtype=torch.bfloat16), torch.empty_like(a, dtype=torch.bfloat16)
    ops.split_hi_lo(a, xh, xl)
    rows = B * (H // 2) * (W // 2)
    oh, ol = _nan((rows, 9 * Cc), torch.bfloat16), _nan((rows, 9 * Cc), torch.bfloat16)
    ops.im2col_s2(xh, oh, B, H, W)
    ops.im2col_s2(xl, ol, B, H, W)
    w1, w2 = _pack_lin(w.permute(0, 2, 3, 1).reshape(Cc, -1))
    out = _nan((rows, Cc), torch.float32)
    ops.gemm(oh, w1, out, a1=ol, bias=bias)
    ops.gemm(oh, w2, out, residual=out)
    to_rows = lambda t: t.permute(0, 2, 3, 1).reshape(rows, Cc)
    ref = to_rows(F.conv2d(x.double(), w.double(), bias.double(), stride=2, padding=1))
    aw = to_rows(F.conv2d(x.double().abs(), w.double().abs(), stride=2, padding=1))
    k = _k_measured(out, ref, aw, bias.double().abs().expand(rows, Cc))
    print(f"3-term downsample ({B}, {H}, {W}, {Cc}): k = {k:.3g} (bar {K3})")
    assert k <= K3


def test_three_term_upsample_then_conv():
    """Upsample2D as EngineF32 runs it: split, nearest 2x upsample of hi and lo, then the 3x3 conv at the upsampled size."""
    from b200sd import ops
    from b200sd.engine_fp32 import _pack_conv
    B, H, W, Cc = 2, 12, 8, 1280
    g = torch.Generator(device=DEV).manual_seed(13)
    x = torch.randn(B, Cc, H, W, generator=g, device=DEV)
    w = torch.randn(Cc, Cc, 3, 3, generator=g, device=DEV) / math.sqrt(9 * Cc)
    bias = torch.randn(Cc, generator=g, device=DEV)
    a = x.permute(0, 2, 3, 1).reshape(B * H * W, Cc).contiguous()
    xh, xl = torch.empty_like(a, dtype=torch.bfloat16), torch.empty_like(a, dtype=torch.bfloat16)
    ops.split_hi_lo(a, xh, xl)
    rows = B * 4 * H * W
    uh, ul = _nan((rows, Cc), torch.bfloat16), _nan((rows, Cc), torch.bfloat16)
    ops.upsample2x(xh, uh, B, H, W)
    ops.upsample2x(xl, ul, B, H, W)
    w1, w2 = _pack_conv(w)
    out = _nan((rows, Cc), torch.float32)
    ops.gemm(uh, w1, out, a1=ul, bias=bias, conv=(B, 2 * H, 2 * W))
    ops.gemm(uh, w2, out, residual=out, conv=(B, 2 * H, 2 * W))
    up = F.interpolate(x.double(), scale_factor=2.0, mode="nearest")
    to_rows = lambda t: t.permute(0, 2, 3, 1).reshape(rows, Cc)
    ref = to_rows(F.conv2d(up, w.double(), bias.double(), padding=1))
    aw = to_rows(F.conv2d(up.abs(), w.double().abs(), padding=1))
    k = _k_measured(out, ref, aw, bias.double().abs().expand(rows, Cc))
    print(f"3-term upsample + conv3x3 ({B}, {H}, {W}, {Cc}): k = {k:.3g} (bar {K3})")
    assert k <= K3


# ---------------------------------------------------------------------------------------------------------------------------------
# end to end at the portrait geometry
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1])
def test_fp32_path_portrait_96x64_vs_oracle(models, seed):
    oracle, ours = models
    g = torch.Generator().manual_seed(100 + seed)
    x = torch.randn(2, 4, 96, 64, generator=g).to(DEV)
    ctx = torch.randn(2, 77, 768, generator=g).to(DEV)
    oc = oracle.to(DEV)
    ours.set_precision("fp32")
    try:
        with torch.no_grad():
            for t in (torch.tensor([999, 37]), torch.tensor([733.37, 12.5])):
                t = t.to(DEV)
                want = oc(x, t, ctx).sample
                got = ours(x, t, ctx).sample
                again = ours(x, t, ctx).sample           # graph replay
                r = float((got - want).abs().max() / want.abs().max())
                print(f"fp32 path 96x64 seed {seed} t={t.tolist()}: max-rel {r:.3g} (bar 1e-4)")
                assert r <= 1e-4, (t.tolist(), r)
                assert torch.equal(got, again), "graph replay must be bit-identical"
    finally:
        oracle.to("cpu")
