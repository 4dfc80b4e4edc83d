"""GPU parity of the tcgen05 GEMM / implicit-GEMM conv kernel against fp32 torch math on the same
bf16-rounded operands.  Tolerance: bf16 output rounding (2^-8 relative) + fp32 accumulation order."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _close(got, want, rel=1.0 / 128):
    got, want = got.float(), want.float()
    scale = float(want.abs().max()) + 1e-6
    err = float((got - want).abs().max())
    assert err <= rel * scale, f"max abs err {err:.4g} vs scale {scale:.4g} (rel {err / scale:.3g})"


def _setup():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False


@pytest.mark.parametrize("M,N,K", [(128, 160, 64), (128, 16, 128), (256, 320, 320), (8192, 320, 320),
                                   (154, 640, 768), (2048, 1920, 640), (100, 256, 1280), (8192, 640, 2560)])
def test_gemm_plain(M, N, K):
    from b200sd import ops
    _setup()
    torch.manual_seed(M + N + K)
    a = torch.randn(M, K, device=DEV).bfloat16()
    w = (torch.randn(N, K, device=DEV) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device=DEV)
    res = torch.randn(M, N, device=DEV).bfloat16()
    out = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    ops.gemm(a, w, out, bias=bias, residual=res)
    want = a.float() @ w.float().t() + bias + res.float()
    _close(out, want)


@pytest.mark.parametrize("M,N,K,conv", [(128, 1280, 5120, None), (512, 1280, 1280, None), (8192, 320, 320, None),
                                        (2048, 640, 9 * 640, (2, 32, 32)), (128, 1280, 9 * 1280, (2, 8, 8))])
def test_gemm_deep_k_f32(M, N, K, conv):
    """fp32-output GEMM / conv3x3 (+bias) against fp32 torch math: small-M / deep-K layers (split-K) and a short-K one."""
    from b200sd import ops
    _setup()
    torch.manual_seed(M + N + K)
    C = K // 9 if conv else K
    a = torch.randn(M, C, device=DEV).bfloat16()
    w = (torch.randn(N, K, device=DEV) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device=DEV)
    out = torch.empty(M, N, device=DEV, dtype=torch.float32)
    ops.gemm(a, w, out, bias=bias, conv=conv)
    if conv is None:
        want = a.float() @ w.float().t() + bias
    else:
        B, H, W = conv
        x = a.float().reshape(B, H, W, C).permute(0, 3, 1, 2)
        w_oihw = w.float().reshape(N, 3, 3, C).permute(0, 3, 1, 2)
        want = F.conv2d(x, w_oihw, bias, padding=1).permute(0, 2, 3, 1).reshape(M, N)
    _close(out, want, rel=1e-3)


def test_gemm_f32_out_no_bias():
    from b200sd import ops
    _setup()
    a = torch.randn(512, 640, device=DEV).bfloat16()
    w = (torch.randn(320, 640, device=DEV) / 25).bfloat16()
    out = torch.empty(512, 320, device=DEV, dtype=torch.float32)
    ops.gemm(a, w, out)
    _close(out, a.float() @ w.float().t(), rel=1e-4)


@pytest.mark.parametrize("split", [2, 4, 8])
def test_gemm_split_k(split):
    from b200sd import ops
    _setup()
    M, N, K = 128, 1280, 5120
    a = torch.randn(M, K, device=DEV).bfloat16()
    w = (torch.randn(N, K, device=DEV) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device=DEV)
    out = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    want = a.float() @ w.float().t() + bias
    for _ in range(2):  # twice: the self-cleaning tile counters must be reusable
        out.zero_()
        ops.gemm(a, w, out, bias=bias, split_k=split)
        _close(out, want)


def test_gemm_dual_source_concat():
    from b200sd import ops
    _setup()
    M, C0, C1, N = 2048, 640, 320, 640
    a0 = torch.randn(M, C0, device=DEV).bfloat16()
    a1 = torch.randn(M, C1, device=DEV).bfloat16()
    w = (torch.randn(N, C0 + C1, device=DEV) / 30).bfloat16()
    out = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    ops.gemm(a0, w, out, a1=a1)
    _close(out, torch.cat([a0, a1], 1).float() @ w.float().t())


@pytest.mark.parametrize("C", [320, 640])
def test_gemm_geglu(C):
    from b200sd import ops
    from b200sd.packing import pack_geglu
    _setup()
    M = 1024
    x = torch.randn(M, C, device=DEV).bfloat16()
    w = (torch.randn(8 * C, C, device=DEV) / C ** 0.5)
    b = torch.randn(8 * C, device=DEV)
    tile = ops.geglu_tile(8 * C)
    wp, bp = pack_geglu(w, b, tile)
    out = torch.empty(M, 4 * C, device=DEV, dtype=torch.bfloat16)
    ops.gemm(x, wp, out, bias=bp, epilogue=ops.EPI_GEGLU, block_n=tile)
    h = x.float() @ w.bfloat16().float().t() + b
    val, gate = h.chunk(2, dim=-1)
    _close(out, val * F.gelu(gate))


@pytest.mark.parametrize("B,H,W,Cin,Cout", [(2, 64, 64, 320, 320), (2, 32, 32, 640, 640), (2, 16, 16, 1280, 1280),
                                            (2, 8, 8, 1280, 1280), (1, 8, 8, 1280, 1280), (3, 8, 8, 640, 320),
                                            (1, 96, 64, 320, 320), (2, 12, 8, 1280, 1280), (1, 48, 32, 640, 640)])
def test_conv3x3(B, H, W, Cin, Cout):
    from b200sd import ops
    from b200sd.packing import pack_conv3x3
    _setup()
    torch.manual_seed(H * W + Cin)
    x = torch.randn(B, Cin, H, W, device=DEV).bfloat16()
    w = (torch.randn(Cout, Cin, 3, 3, device=DEV) / (9 * Cin) ** 0.5).bfloat16()
    bias = torch.randn(Cout, device=DEV)
    temb = torch.randn(B, Cout, device=DEV)
    x_nhwc = x.permute(0, 2, 3, 1).contiguous().reshape(B * H * W, Cin)
    out = torch.empty(B * H * W, Cout, device=DEV, dtype=torch.bfloat16)
    ops.gemm(x_nhwc, pack_conv3x3(w), out, bias=bias, rowbias=temb, conv=(B, H, W), rows_per_image=H * W)
    want = F.conv2d(x.float(), w.float(), bias, padding=1) + temb[:, :, None, None]
    want = want.permute(0, 2, 3, 1).reshape(B * H * W, Cout)
    _close(out, want)


def test_conv3x3_dual_source_residual():
    from b200sd import ops
    from b200sd.packing import pack_conv3x3
    _setup()
    B, H, W, C0, C1, Cout = 2, 16, 16, 1280, 640, 1280
    x0 = torch.randn(B, C0, H, W, device=DEV).bfloat16()
    x1 = torch.randn(B, C1, H, W, device=DEV).bfloat16()
    w = (torch.randn(Cout, C0 + C1, 3, 3, device=DEV) / (9 * (C0 + C1)) ** 0.5).bfloat16()
    bias = torch.randn(Cout, device=DEV)
    res = torch.randn(B * H * W, Cout, device=DEV).bfloat16()
    n0 = x0.permute(0, 2, 3, 1).contiguous().reshape(-1, C0)
    n1 = x1.permute(0, 2, 3, 1).contiguous().reshape(-1, C1)
    out = torch.empty(B * H * W, Cout, device=DEV, dtype=torch.bfloat16)
    ops.gemm(n0, pack_conv3x3(w), out, a1=n1, bias=bias, residual=res, conv=(B, H, W))
    want = F.conv2d(torch.cat([x0, x1], 1).float(), w.float(), bias, padding=1)
    want = want.permute(0, 2, 3, 1).reshape(B * H * W, Cout) + res.float()
    _close(out, want)


def test_gemm_rejects_bad_shapes():
    from b200sd import ops
    from b200sd._lib import B200SDError
    a = torch.randn(128, 100, device=DEV).bfloat16()  # K not a multiple of 64
    w = torch.randn(64, 100, device=DEV).bfloat16()
    out = torch.empty(128, 64, device=DEV, dtype=torch.bfloat16)
    with pytest.raises(B200SDError):
        ops.gemm(a, w, out)


@pytest.mark.parametrize("M,N,K,split", [(8192, 320, 320, 1), (512, 1280, 5120, 0), (128, 1280, 2560, 4)])
def test_gemm_fp32_residual_and_output(M, N, K, split):
    """fp32 residual stream: out(fp32) = A W^T + bias + residual(fp32), incl. in-place (out is residual)."""
    from b200sd import ops
    _setup()
    torch.manual_seed(M + K)
    a = torch.randn(M, K, device=DEV).bfloat16()
    w = (torch.randn(N, K, device=DEV) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device=DEV)
    res = torch.randn(M, N, device=DEV)
    want = a.float() @ w.float().t() + bias + res
    out = res.clone()
    ops.gemm(a, w, out, bias=bias, residual=out, split_k=split)
    _close(out, want, rel=2e-5)
    outb = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    ops.gemm(a, w, outb, bias=bias, residual=res, split_k=split)
    _close(outb, want)


@pytest.mark.parametrize("B,H,W,Cin,Cout,conv,res", [
    (2, 64, 64, 320, 320, True, True),      # 64x64 level conv2 (+fp32 residual), no split
    (2, 32, 32, 640, 640, True, False),     # split-K cluster: every rank publishes the rows it stores
    (2, 16, 16, 1280, 1280, True, True),    # deep split
    (2, 64, 64, 320, 320, False, True),     # plain GEMM (transformer proj_out), hw % 128 == 0
    (8, 64, 64, 320, 640, True, False),     # CTA pairs at batch 8
    (2, 32, 48, 640, 640, True, False),     # portrait geometry
    (2, 8, 8, 1280, 1280, True, True),      # 8x8 level: one tile holds both images, the split-K ranks separate them
    (2, 8, 8, 1280, 1280, False, True),     # same for the plain GEMM (proj_out), split 2
    (2, 8, 12, 1280, 1280, True, False),    # portrait 8x12: 96-row tiles, trailing ranks publish zeros
])
def test_gemm_groupnorm_statistics(B, H, W, Cin, Cout, conv, res):
    """The fp32-output epilogue also publishes per-CTA column sums / sums of squares (gn_part); GroupNorm from those
    partials (no statistics pass over the tensor) must match F.group_norm of the GEMM output."""
    from b200sd import ops
    from b200sd.packing import pack_conv3x3
    _setup()
    torch.manual_seed(B * H + Cin + Cout)
    hw, M = H * W, B * H * W
    a = torch.randn(M, Cin, device=DEV).bfloat16()
    bias = torch.randn(Cout, device=DEV)
    residual = torch.randn(M, Cout, device=DEV) * 3 + 1 if res else None
    out = torch.empty(M, Cout, device=DEV)
    if conv:
        w = pack_conv3x3((torch.randn(Cout, Cin, 3, 3, device=DEV) / (9 * Cin) ** 0.5).bfloat16())
        args = ops.gemm(a, w, out, bias=bias, residual=residual, conv=(B, H, W), launch=False)
    else:
        w = (torch.randn(Cout, Cin, device=DEV) / Cin ** 0.5).bfloat16()
        args = ops.gemm(a, w, out, bias=bias, residual=residual, launch=False)
    parts = ops.gemm_attach_gn_parts(args, hw, DEV)
    assert parts is not None, "shape should be covered"
    ops.gemm_run(args)
    # the partial rows of an image add up to its column sums
    pb = parts.buf.view(-1, 2, Cout)
    assert pb.shape[0] >= B * parts.ppi
    got = pb[:B * parts.ppi].view(B, parts.ppi, 2, Cout).sum(1)
    o3 = out.view(B, hw, Cout).double()
    assert (got[:, 0] - o3.sum(1)).abs().max().item() <= 1e-4 * o3.abs().sum(1).max().item() + 1e-3
    assert (got[:, 1] - (o3 * o3).sum(1)).abs().max().item() <= 1e-4 * (o3 * o3).sum(1).max().item()
    # GroupNorm from the partials
    g = torch.randn(Cout, device=DEV)
    bt = torch.randn(Cout, device=DEV)
    y = torch.empty(M, Cout, device=DEV, dtype=torch.bfloat16)
    stats = torch.empty(B, 32, 2, device=DEV)
    assert ops.gn_parts_supported(Cout)
    ops.groupnorm_silu_parts(out, None, parts, None, g, bt, y, B, hw, 32, 1e-5, True, stats_out=stats)
    xn = out.view(B, hw, Cout).permute(0, 2, 1)
    want = F.silu(F.group_norm(xn, 32, g, bt, 1e-5)).permute(0, 2, 1).reshape(M, Cout)
    _close(y, want, 1.0 / 128)
    xg = out.view(B, hw, 32, Cout // 32).double()
    mean = xg.mean(dim=(1, 3))
    rstd = 1.0 / torch.sqrt(xg.var(dim=(1, 3), unbiased=False) + 1e-5)
    assert (stats[:, :, 0] - mean).abs().max().item() < 1e-4 * (1 + mean.abs().max().item())
    assert ((stats[:, :, 1] - rstd) / rstd).abs().max().item() < 1e-3


def test_groupnorm_parts_concat():
    """[x | skip] GroupNorm with each source's statistics coming from its own producer (up-block resnets)."""
    from b200sd import ops
    _setup()
    torch.manual_seed(5)
    B, H, W, C0, C1 = 2, 32, 32, 640, 320
    hw, M = H * W, B * H * W
    outs, parts = [], []
    for Cc in (C0, C1):
        a = torch.randn(M, 320, device=DEV).bfloat16()
        w = (torch.randn(Cc, 320, device=DEV) / 320 ** 0.5).bfloat16()
        o = torch.empty(M, Cc, device=DEV)
        args = ops.gemm(a, w, o, bias=torch.randn(Cc, device=DEV), launch=False)
        p = ops.gemm_attach_gn_parts(args, hw, DEV)
        assert p is not None
        ops.gemm_run(args)
        outs.append(o)
        parts.append(p)
    C = C0 + C1
    g, bt = torch.randn(C, device=DEV), torch.randn(C, device=DEV)
    y = torch.empty(M, C, device=DEV, dtype=torch.bfloat16)
    raw = torch.empty(M, C, device=DEV, dtype=torch.bfloat16)
    assert ops.gn_parts_supported(C)
    ops.groupnorm_silu_parts(outs[0], outs[1], parts[0], parts[1], g, bt, y, B, hw, 32, 1e-5, True, raw_out=raw)
    xc = torch.cat(outs, 1)
    xn = xc.view(B, hw, C).permute(0, 2, 1)
    want = F.silu(F.group_norm(xn, 32, g, bt, 1e-5)).permute(0, 2, 1).reshape(M, C)
    _close(y, want, 1.0 / 128)
    _close(raw, xc, 1.0 / 128)


def test_gemm_gn_layout_straddling_tiles():
    """A 128-row tile spanning two images: the persistent kernel publishes one partial row per 32 output rows (never straddles a
    64-row image); images that are not a multiple of 32 rows and bf16 outputs get no statistics layout -- the caller keeps the
    stand-alone GroupNorm."""
    from b200sd import ops
    _setup()
    torch.manual_seed(9)
    a = torch.randn(2 * 64, 320, device=DEV).bfloat16()
    w = (torch.randn(1280, 320, device=DEV) / 18).bfloat16()
    out = torch.empty(2 * 64, 1280, device=DEV)
    args = ops.gemm(a, w, out, launch=False)
    parts = ops.gemm_attach_gn_parts(args, 64, DEV)
    if parts is not None:
        ops.gemm_run(args)
        pp = parts.buf.view(-1, 2, 1280)
        assert pp.shape[0] >= 2 * parts.ppi
        for b in range(2):
            x = out[b * 64:(b + 1) * 64].double()
            got = pp[b * parts.ppi:(b + 1) * parts.ppi].double().sum(0)
            assert (got[0] - x.sum(0)).abs().max().item() < 1e-3
            assert (got[1] - (x * x).sum(0)).abs().max().item() < 1e-2
    a3 = torch.randn(2 * 48, 320, device=DEV).bfloat16()
    assert ops.gemm_attach_gn_parts(ops.gemm(a3, w, torch.empty(2 * 48, 1280, device=DEV), launch=False), 48, DEV) is None
    outb = torch.empty(2 * 256, 1280, device=DEV, dtype=torch.bfloat16)   # bf16 output: not covered either
    a2 = torch.randn(2 * 256, 1280, device=DEV).bfloat16()
    assert ops.gemm_attach_gn_parts(ops.gemm(a2, w, outb, launch=False), 256, DEV) is None
