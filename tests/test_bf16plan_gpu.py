"""Launch-by-launch parity of the bf16 UNet plan (engine.py: the plan bench.py times) against float64 torch.

The signatures are recorded, not hand-picked: a fixture wraps the ops entry points the plan closures look up at run time and
runs eager forwards of the full-size random-init UNet at the batches the sampler issues (UNet batch 1, 2, 3, 16 and 128; 64x64
and 96x64 latents), context plan included.  Every recorded call is then rerun on fresh random operands and compared with a
float64 reference, per element:

  GEMM (A W^T + bias + rowbias + residual):  |out - ref| <= rho |ref| + k(K) u (|A||W|^T + |bias| + |rowbias| + |residual|)
      u = 2^-24 (fp32), rho = 2^-8 for a bf16 output (its rounding) and 0 for fp32.  k(K) = 16 + K / 64 covers the fp32
      accumulation of K / 16 tensor-core steps, the split-K partial sums and the <= 3 epilogue adds: rounding errors of the
      steps add like a random walk well inside this (K = 320: 21, K = 23040: 376; the printed k is the measured one).
      Residuals cancel 63/64 of the rest on the checked rows, so a residual rounded early (2^-9 |residual|) shows.
  GEGLU (val * gelu(gate)): the same k(K) u bound on each pre-activation, propagated through |gelu(gate)| and |val| |gelu'|,
      plus 2^-21 |val| |gate| for the GELU itself (gelu_erf_fast: < 3e-7 |x| by its construction) and rho |ref|.
  GroupNorm statistics from the GEMM epilogue: |sum - ref| <= (2 * 128 + parts + 8) u sum|x| (fp32 sums of <= 128 rows per part).
  GroupNorm / LayerNorm (bf16 out): 2^-8 |ref| + u (16 + 8 r + 2 r^2) max|ref|, r = largest |mean| / std of a group or row.
  Attention (bf16 P, fp32 row sums, bf16 out), per query row: 2^-8 |ref| + 1.25 * 2^-8 sum_j p_j |v_j|: P rounded to bf16
      costs <= 2^-8 sum p|v|, the rest (exp2 approximations <= 7.5e-5 relative, fp32 sums) stays under the remaining quarter.
  small_linear / timestep embedding (fp32): gamma_n bounds of their sequential sums; argument rounding 24 u |t f| for the sinusoid.
  upsample2x, im2col_s2 and GroupNorm's raw_out are copies: bit-exact.

At UNet batch 128 only the first, a middle and the last image (plus the last 128 rows of a linear GEMM) are compared."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24
RHO = 2.0 ** -8
BAND = 128            # NaN sentinel rows after every output (and after every GEMM A operand)
GELU_C = 2.0 ** -21
ATTN_C = 1.25
GEOMETRIES = [(2, 64, 64), (2, 96, 64), (16, 64, 64), (16, 96, 64), (1, 64, 64), (3, 64, 64), (128, 96, 64)]

# what the recorded GEMMs must cover between them (the path table below is printed by test_gemm_paths_cover_the_engine)
REQUIRED_PATHS = {"tile", "split cluster", "CTA pair", "persistent linear", "persistent GEGLU", "persistent split-16",
                  "tile GEGLU N=10240", "96-row conv tile", "two-image conv tile", "rowbias", "in-place fp32 residual",
                  "fp32 residual -> bf16 out", "dual source", "gn_part"}


def _nan(shape, dtype):
    return torch.full(shape, float("nan"), dtype=dtype, device=DEV)


def _k_acc(K):
    return 16 + K / 64


def _sample_images(n):
    return list(range(n)) if n <= 3 else [0, n // 2, n - 1]


def _silu64(t):
    return t * torch.sigmoid(t)


def _gelu64(t):
    return 0.5 * t * (1 + torch.erf(t / math.sqrt(2)))


def _dgelu64(t):
    return 0.5 * (1 + torch.erf(t / math.sqrt(2))) + t * torch.exp(-0.5 * t * t) / math.sqrt(2 * math.pi)


# ---------------------------------------------------------------------------------------------------------------------------------
# signature fixture
# ---------------------------------------------------------------------------------------------------------------------------------
_GEMM_FIELDS = ("M", "N", "K", "C0", "C1", "ldc", "ldr", "ldrb", "conv_taps", "batch", "H", "W", "rows_per_image", "epilogue",
                "out_dtype", "residual_dtype", "block_n", "split_k", "pair")


@pytest.fixture(scope="module")
def sigs():
    """{op name: {signature: geometry label}} of every call one eager forward issues at each geometry, and the GEMM paths."""
    from b200sd import ops
    from b200sd.unet import UNet2DConditionModel
    from oracle.unet_ref import make_oracle_unet
    oracle = make_oracle_unet(seed=0)
    ours = UNet2DConditionModel()
    ours.load_state_dict(oracle.state_dict(), strict=True)
    del oracle
    ours = ours.to(DEV).eval()
    seen = {}
    paths = {}
    geo = [None]

    def rec(name, key):
        seen.setdefault(name, {}).setdefault(key, geo[0])

    real = {n: getattr(ops, n) for n in ("gemm_run", "attention", "groupnorm_silu", "groupnorm_silu_parts", "layernorm",
                                          "small_linear", "cast_act", "timestep_embedding", "conv_in", "conv_out",
                                          "nhwc_bias_to_nchw", "upsample2x", "im2col_s2")}
    nimg = [0]

    def gemm_run(args):
        d = {f: getattr(args, f) for f in _GEMM_FIELDS}
        d.update(bias=bool(args.bias), rowbias=bool(args.rowbias), gn=bool(args.gn_part), nimg=nimg[0],
                 res=0 if not args.residual else (2 if args.residual == args.out else 1))
        key = tuple(sorted(d.items()))
        rec("gemm", key)
        paths.setdefault(key, ops.gemm_path(args))
        return real["gemm_run"](args)

    def attention(q, k, v, out, batch, heads, Sq, Skv, d, scale, ldq=None, ldk=None, ldv=None, ldo=None, q_off=0, k_off=0,
                  v_off=0, ws=None):
        rec("attention", (batch, heads, Sq, Skv, d, ldq, ldk, ldv, ldo, q_off, k_off, v_off, q.data_ptr() == k.data_ptr()))
        return real["attention"](q, k, v, out, batch, heads, Sq, Skv, d, scale, ldq, ldk, ldv, ldo, q_off, k_off, v_off, ws)

    def groupnorm_silu(x0, x1, gamma, beta, out, batch, hw, groups=32, eps=1e-5, silu=True, raw_out=None, stats_out=None):
        rec("groupnorm_silu", (batch, hw, x0.shape[-1], x1.shape[-1] if x1 is not None else 0, x0.dtype, groups, float(eps),
                               bool(silu), raw_out is not None))
        return real["groupnorm_silu"](x0, x1, gamma, beta, out, batch, hw, groups, eps, silu, raw_out, stats_out)

    def groupnorm_silu_parts(x0, x1, p0, p1, gamma, beta, out, batch, hw, groups=32, eps=1e-5, silu=True, raw_out=None,
                             stats_out=None):
        rec("groupnorm_silu_parts", (batch, hw, x0.shape[-1], x1.shape[-1] if x1 is not None else 0, x0.dtype, p0.ppi, p0.ld,
                                     p1.ppi if p1 is not None else 0, p1.ld if p1 is not None else 0, groups, float(eps),
                                     bool(silu), raw_out is not None))
        return real["groupnorm_silu_parts"](x0, x1, p0, p1, gamma, beta, out, batch, hw, groups, eps, silu, raw_out, stats_out)

    def layernorm(x, gamma, beta, out, eps=1e-5):
        rec("layernorm", (x.numel() // x.shape[-1], x.shape[-1], x.dtype, out.dtype, float(eps)))
        return real["layernorm"](x, gamma, beta, out, eps)

    def small_linear(x, w, bias, silu_in=False, silu_out=False, out=None):
        rec("small_linear", (x.shape[0], w.shape[0], x.shape[1], bias is not None, bool(silu_in), bool(silu_out)))
        return real["small_linear"](x, w, bias, silu_in, silu_out, out)

    def cast_act(x, out_bf16, silu=False):
        rec("cast_act", (x.numel(), bool(silu)))
        return real["cast_act"](x, out_bf16, silu)

    def timestep_embedding(t, dim, out=None):
        rec("timestep_embedding", (t.numel(), dim))
        return real["timestep_embedding"](t, dim, out)

    def conv_in(x, w, bias, out):
        rec("conv_in", (tuple(x.shape), w.shape[0], out.dtype))
        return real["conv_in"](x, w, bias, out)

    def conv_out(x, w, bias, out):
        rec("conv_out", (tuple(out.shape), x.shape[-1]))
        return real["conv_out"](x, w, bias, out)

    def nhwc_bias_to_nchw(x, bias, out):
        rec("nhwc_bias_to_nchw", (tuple(out.shape), x.shape[-1]))
        return real["nhwc_bias_to_nchw"](x, bias, out)

    def upsample2x(x, out, batch, H, W):
        rec("upsample2x", (batch, H, W, x.shape[-1], x.dtype))
        return real["upsample2x"](x, out, batch, H, W)

    def im2col_s2(x, out, batch, H, W, pad=1):
        rec("im2col_s2", (batch, H, W, x.shape[-1], x.dtype, pad))
        return real["im2col_s2"](x, out, batch, H, W, pad)

    spies = dict(gemm_run=gemm_run, attention=attention, groupnorm_silu=groupnorm_silu, groupnorm_silu_parts=groupnorm_silu_parts,
                 layernorm=layernorm, small_linear=small_linear, cast_act=cast_act, timestep_embedding=timestep_embedding,
                 conv_in=conv_in, conv_out=conv_out, nhwc_bias_to_nchw=nhwc_bias_to_nchw, upsample2x=upsample2x,
                 im2col_s2=im2col_s2)
    ours.use_cuda_graph = False
    for n, f in spies.items():
        setattr(ops, n, f)
    try:
        with torch.no_grad():
            for B, H, W in GEOMETRIES:
                geo[0], nimg[0] = f"b{B} {H}x{W}", B
                t = torch.linspace(3.25, 981.5, B, device=DEV)
                ours(torch.randn(B, 4, H, W, device=DEV), t, torch.randn(B, 77, 768, device=DEV))
                torch.cuda.synchronize()
                ours._engines.clear()
                torch.cuda.empty_cache()
    finally:
        for n, f in real.items():
            setattr(ops, n, f)
        ours.use_cuda_graph = True
    del ours
    torch.cuda.empty_cache()
    return seen, paths


# ---------------------------------------------------------------------------------------------------------------------------------
# GEMM
# ---------------------------------------------------------------------------------------------------------------------------------
def _path_labels(s, p):
    L = set()
    geglu = s["epilogue"] == 1
    if p["kernel"] == "tile":
        L.add("split cluster" if p["split_k"] > 1 else ("CTA pair" if p["pair"] else "tile"))
        if geglu and s["N"] == 10240:
            L.add("tile GEGLU N=10240")
    elif p["kernel"] == "persistent":
        L.add("persistent GEGLU" if geglu else "persistent linear")
    elif p["psplit"] == 16:
        L.add("persistent split-16")
    else:
        L.add(f"persistent split-{p['psplit']}")
    if s["conv_taps"] == 9:
        if p["rows_valid"] == 96:
            L.add("96-row conv tile")
        if p["tile_n"] == 2:
            L.add("two-image conv tile")
    if s["rowbias"]:
        L.add("rowbias")
    if s["res"] == 2 and s["residual_dtype"] == 0:
        L.add("in-place fp32 residual")
    if s["res"] and s["residual_dtype"] == 0 and s["out_dtype"] == 1:
        L.add("fp32 residual -> bf16 out")
    if s["C1"]:
        L.add("dual source")
    if s["gn"]:
        L.add("gn_part")
    return L


class _GemmCase:
    """Fresh operands for one recorded GEMM signature, the float64 reference on the checked rows, and the check."""

    def __init__(self, s, seed):
        from b200sd import packing
        self.s = s
        g = torch.Generator(device=DEV).manual_seed(seed)
        M, N, K, C0, C1 = s["M"], s["N"], s["K"], s["C0"], s["C1"]
        self.M, self.N, self.K = M, N, K
        self.conv = s["conv_taps"] == 9
        self.geglu = s["epilogue"] == 1
        nimg = s["batch"] if self.conv else s["nimg"]
        rn = lambda *sh: torch.randn(*sh, generator=g, device=DEV)
        self.a0 = _nan((M + BAND, C0), torch.bfloat16)
        self.a0[:M] = rn(M, C0).bfloat16()
        self.a1 = None
        if C1:
            self.a1 = _nan((M + BAND, C1), torch.bfloat16)
            self.a1[:M] = rn(M, C1).bfloat16()
        self.bias = self.rb = None
        if self.geglu:
            h = N // 2
            wv = (rn(h, K) / math.sqrt(K)).bfloat16().float()
            wg = (rn(h, K) * 3 / math.sqrt(K)).bfloat16().float()      # gates reach both erf tails
            bv, bg = rn(h) * 0.5, rn(h) * 0.5
            self.w, self.bias = packing.pack_geglu(torch.cat([wv, wg]), torch.cat([bv, bg]), s["block_n"])
            self.outw = N // 2
        else:
            self.w = (rn(N, K) / math.sqrt(K)).bfloat16()
            if s["bias"]:
                self.bias = rn(N)
            self.outw = N
        if s["rowbias"]:
            self.rb_buf = rn(M // s["rows_per_image"], s["ldrb"])
            self.rb_off = (s["ldrb"] - N) // 8 * 4
        self.out_dtype = torch.float32 if s["out_dtype"] == 0 else torch.bfloat16
        assert s["ldc"] == self.outw

        # checked rows
        imgs = _sample_images(nimg)
        rpi = M // nimg
        rows = torch.cat([torch.arange(b * rpi, (b + 1) * rpi, device=DEV) for b in imgs])
        if not self.conv and nimg > 3:
            rows = torch.unique(torch.cat([rows, torch.arange(max(M - 128, 0), M, device=DEV)]))
        self.rows = rows
        a = self.a0[:M] if self.a1 is None else torch.cat([self.a0[:M], self.a1[:M]], 1)
        if self.conv:
            Hh, Ww, Cc = s["H"], s["W"], C0 + C1
            x = a.reshape(nimg, Hh, Ww, Cc)[imgs].permute(0, 3, 1, 2).double()
            to_rows = lambda t: t.permute(0, 2, 3, 1).reshape(-1, t.shape[1])
            mm = lambda xx, ww: to_rows(F.conv2d(xx, ww.reshape(ww.shape[0], 3, 3, Cc).permute(0, 3, 1, 2), padding=1))
        else:
            x = a[rows].double()
            mm = lambda xx, ww: xx @ ww.T
        if self.geglu:
            self.pv, self.pg = mm(x, wv.double()) + bv.double(), mm(x, wg.double()) + bg.double()
            self.mv, self.mg = mm(x.abs(), wv.double().abs()) + bv.double().abs(), mm(x.abs(), wg.double().abs()) + bg.double().abs()
            self.ref = self.pv * _gelu64(self.pg)
            return
        w64 = self.w.double()
        pre = mm(x, w64)
        mag = mm(x.abs(), w64.abs())
        if self.bias is not None:
            pre = pre + self.bias.double()
            mag = mag + self.bias.double().abs()
        if s["rowbias"]:
            rbv = self.rb_buf[:, self.rb_off:self.rb_off + N].double()[rows // s["rows_per_image"]]
            pre, mag = pre + rbv, mag + rbv.abs()
        self.res = None
        if s["res"]:
            assert s["residual_dtype"] == 0 and s["ldr"] == N
            res = rn(M, N) * float(pre.std())
            res[rows] = (-pre * (63 / 64)).float()
            self.res = res
            pre = pre + res[rows].double()
            mag = mag + res[rows].double().abs()
        self.ref, self.mag = pre, mag

    def run(self, persist=-1, pair=None, split_k=None, gn_hw=0):
        """One launch under a path override; returns (output, GnParts or None, path)."""
        from b200sd import ops
        from b200sd._lib import lib
        s = self.s
        out = _nan((self.M + BAND, self.outw), self.out_dtype)
        residual = None
        if s["res"] == 2:
            out[:self.M] = self.res
            residual = out
        elif s["res"] == 1:
            residual = self.res
        lib().b200sd_debug_set(0, persist)
        try:
            args = ops.gemm(self.a0, self.w, out, a1=self.a1, bias=self.bias, residual=residual, M=self.M,
                            conv=(s["batch"], s["H"], s["W"]) if self.conv else None, epilogue=s["epilogue"],
                            block_n=s["block_n"], split_k=s["split_k"] if split_k is None else split_k,
                            pair=s["pair"] if pair is None else pair, launch=False)
            args.ldc = self.outw
            if s["rowbias"]:
                args.rowbias = self.rb_buf.data_ptr() + self.rb_off * 4
                args.ldrb, args.rows_per_image = s["ldrb"], s["rows_per_image"]
            parts = ops.gemm_attach_gn_parts(args, gn_hw, DEV) if gn_hw else None
            path = ops.gemm_path(args)
            ops.gemm_run(args)
            torch.cuda.synchronize()
        finally:
            lib().b200sd_debug_set(0, -1)
        return out, parts, path

    def check(self, out):
        """(measured k, worst |err| / bar); asserts the sentinel band."""
        assert torch.isnan(out[self.M:]).all(), "GEMM wrote past row M"
        got = out[self.rows].double()
        rho = RHO if self.out_dtype == torch.bfloat16 else 0.0
        kU = _k_acc(self.K) * U
        err = (got - self.ref).abs()
        fixed = rho * self.ref.abs()          # the part of the bar that is not the accumulation
        if self.geglu:
            gl, dg = _gelu64(self.pg).abs(), _dgelu64(self.pg).abs() + 0.5 * kU * self.mg
            mag = gl * self.mv + self.pv.abs() * dg * self.mg
            fixed = fixed + GELU_C * self.pv.abs() * self.pg.abs() + (kU * self.mv) * dg * (kU * self.mg)
        else:
            mag = self.mag
        bar = fixed + kU * mag
        k = float(((err - fixed).clamp(min=0) / (U * mag)).max())
        return k, float((err / bar).max())


def _desc(s, p):
    kind = ("conv" if s["conv_taps"] == 9 else "lin") + ("-geglu" if s["epilogue"] == 1 else "")
    extra = [n for n, on in (("bias", s["bias"]), ("rowbias", s["rowbias"]), ("gn", s["gn"]), ("dual", s["C1"])) if on]
    if s["res"]:
        extra.append("res-inplace" if s["res"] == 2 else "res")
    return (f"{kind} M{s['M']} N{s['N']} K{s['K']} out={'f32' if s['out_dtype'] == 0 else 'bf16'} {'+'.join(extra)} | "
            f"{p['kernel']} split{p['split_k']} psplit{p['psplit']} pair{p['pair']} bn{p['block_n']} tiles {p['m_tiles']}x"
            f"{p['n_tiles']} rows{p['rows_valid']} tile_n{p['tile_n']}")


def _gn_hw(s):
    return (s["H"] * s["W"] if s["conv_taps"] == 9 else s["M"] // s["nimg"]) if s["gn"] else 0


def test_gemm_paths_cover_the_engine(sigs):
    seen, paths = sigs
    covered = {}
    for key, geo in seen["gemm"].items():
        s = dict(key)
        for lab in _path_labels(s, paths[key]):
            covered.setdefault(lab, geo)
    print("GEMM paths of the bf16 plan (first geometry that takes each):")
    for lab in sorted(covered):
        print(f"  {lab:28s} {covered[lab]}")
    print(f"  ({len(seen['gemm'])} distinct GEMM signatures)")
    assert REQUIRED_PATHS <= set(covered), f"not taken by the engine any more: {sorted(REQUIRED_PATHS - set(covered))}"


def test_gemm_every_engine_signature(sigs):
    seen, paths = sigs
    worst = (0.0, None)
    for i, (key, geo) in enumerate(sorted(seen["gemm"].items(), key=lambda kv: str(kv[0]))):
        s = dict(key)
        case = _GemmCase(s, seed=i)
        out, parts, path = case.run(gn_hw=_gn_hw(s))
        assert path == paths[key], "gemm_path changed between the engine's call and the rerun"
        k, r = case.check(out)
        print(f"[{geo}] {_desc(s, path)}: k = {k:.3g} (bar k = {_k_acc(s['K']):.0f}), worst {r:.3f} of the bar")
        assert r <= 1.0, (geo, _desc(s, path), k, r)
        if parts is not None:
            _check_gn_parts(case, out, parts, _gn_hw(s), geo)
        if r > worst[0]:
            worst = (r, _desc(s, path))
        del case
    print(f"GEMM: worst signature at {worst[0]:.3f} of its bar: {worst[1]}")


def test_gemm_every_engine_signature_on_the_other_paths(sigs):
    """Each signature under forced persistent on / off (debug key 0), CTA pairs on / off and an explicit cluster split_k."""
    seen, _ = sigs
    taken = set()
    for i, (key, geo) in enumerate(sorted(seen["gemm"].items(), key=lambda kv: str(kv[0]))):
        s = dict(key)
        case = _GemmCase(s, seed=1000 + i)
        variants = [dict(persist=1), dict(persist=0), dict(pair=1), dict(pair=-1)]
        kb = s["K"] // 64
        if s["epilogue"] == 0:
            for sk in (2, 4, 8):
                if kb >= sk and (sk - 1) * -(-kb // sk) < kb:
                    variants.append(dict(split_k=sk, pair=-1))
        for v in variants:
            out, parts, path = case.run(gn_hw=_gn_hw(s), **v)
            k, r = case.check(out)
            taken |= _path_labels(s, path)
            print(f"[{geo}] {v} {_desc(s, path)}: k = {k:.3g}, worst {r:.3f} of the bar")
            assert r <= 1.0, (geo, v, _desc(s, path), k, r)
            if parts is not None:
                _check_gn_parts(case, out, parts, _gn_hw(s), geo)
        del case
    print(f"paths taken by the overrides: {sorted(taken)}")


def _check_gn_parts(case, out, parts, hw, geo):
    """Per-image column sums / sums of squares the epilogue published == float64 sums of the stored fp32 output."""
    M, N = case.M, case.N
    nimg = M // hw
    buf = parts.buf.reshape(-1, 2, N).double()
    imgs = _sample_images(nimg)
    worst = 0.0
    for b in imgs:
        y = out[b * hw:(b + 1) * hw].double()
        got = buf[b * parts.ppi:(b + 1) * parts.ppi].sum(0)
        ref = torch.stack([y.sum(0), (y * y).sum(0)])
        mag = torch.stack([y.abs().sum(0), (y * y).sum(0)])
        bar = (2 * 128 + parts.ppi + 8) * U * mag
        worst = max(worst, float(((got - ref).abs() / bar).max()))
    assert worst <= 1.0, (geo, "gn_part statistics", worst)


# ---------------------------------------------------------------------------------------------------------------------------------
# GroupNorm
# ---------------------------------------------------------------------------------------------------------------------------------
def _gn_ref(x, batch, hw, gamma, beta, eps, silu):
    C = x.shape[1]
    xd = x.double().reshape(batch, hw, C).permute(0, 2, 1)
    ref = F.group_norm(xd, 32, gamma.double(), beta.double(), eps)
    if silu:
        ref = _silu64(ref)
    grp = xd.reshape(batch, 32, -1)
    r = float((grp.mean(-1).abs() / grp.std(-1, unbiased=False)).max())
    return ref.permute(0, 2, 1).reshape(batch * hw, C), r


def _gn_bar(r):
    return U * (16 + 8 * r + 2 * r * r) + 2.0 ** -20       # + SiLU on __expf


def _gn_inputs(batch, hw, c0, c1, g):
    x0 = torch.randn(batch * hw, c0, generator=g, device=DEV) * 1.5 + 0.5
    x1 = torch.randn(batch * hw, c1, generator=g, device=DEV) * 0.7 - 0.3 if c1 else None
    C = c0 + c1
    gamma = 1 + 0.2 * torch.randn(C, generator=g, device=DEV)
    beta = 0.2 * torch.randn(C, generator=g, device=DEV)
    return x0, x1, gamma, beta


def _gn_compare(name, key, out, x, batch, hw, gamma, beta, eps, silu):
    n = batch * hw
    assert torch.isnan(out[n:]).all(), f"{name} wrote past the last row"
    worst = 0.0
    for b in _sample_images(batch):
        ref, r = _gn_ref(x[b * hw:(b + 1) * hw], 1, hw, gamma, beta, eps, silu)
        got = out[b * hw:(b + 1) * hw].double()
        e = (got - ref).abs() - RHO * ref.abs()
        c = float(e.max()) / float(ref.abs().max())
        assert c <= _gn_bar(r), (name, key, b, c, _gn_bar(r))
        worst = max(worst, c / _gn_bar(r))
    print(f"{name} {key}: worst image at {worst:.3f} of its bar")


def test_groupnorm_silu_engine_signatures(sigs):
    from b200sd import ops
    seen, _ = sigs
    g = torch.Generator(device=DEV).manual_seed(7)
    for key in sorted(seen.get("groupnorm_silu", {}), key=str):
        batch, hw, c0, c1, dt, groups, eps, silu, raw = key
        x0, x1, gamma, beta = _gn_inputs(batch, hw, c0, c1, g)
        x0, x1 = x0.to(dt), (x1.to(dt) if x1 is not None else None)
        C, n = c0 + c1, batch * hw
        out = _nan((n + BAND, C), torch.bfloat16)
        rawo = _nan((n + BAND, C), torch.bfloat16) if raw else None
        ops.groupnorm_silu(x0, x1, gamma, beta, out[:n], batch, hw, groups, eps, silu, raw_out=rawo[:n] if raw else None)
        torch.cuda.synchronize()
        x = torch.cat([x0, x1], 1) if x1 is not None else x0
        if raw:
            assert torch.equal(rawo[:n], x.bfloat16()) and torch.isnan(rawo[n:]).all()
        _gn_compare("groupnorm_silu", key[:5], out, x.float(), batch, hw, gamma, beta, eps, silu)


def _parts(x, batch, hw, ppi):
    """GnParts of x as its producer would publish them: per image, ppi row chunks of [sum | sum of squares]."""
    from b200sd import ops
    N = x.shape[1]
    buf = torch.empty(batch * ppi, 2, N, dtype=torch.float64, device=DEV)
    for b in range(batch):
        for i, ch in enumerate(torch.tensor_split(x[b * hw:(b + 1) * hw].double(), ppi)):
            buf[b * ppi + i, 0], buf[b * ppi + i, 1] = ch.sum(0), (ch * ch).sum(0)
    return ops.GnParts(buf.float().reshape(-1).contiguous(), ppi, N)


def test_groupnorm_silu_parts_engine_signatures(sigs):
    from b200sd import ops
    seen, _ = sigs
    keys = sorted(seen.get("groupnorm_silu_parts", {}), key=str)
    assert any(k[3] > 0 for k in keys), "no [x | skip] GroupNorm with both producers' statistics recorded"
    g = torch.Generator(device=DEV).manual_seed(8)
    for key in keys:
        batch, hw, c0, c1, dt, ppi0, ld0, ppi1, ld1, groups, eps, silu, raw = key
        x0, x1, gamma, beta = _gn_inputs(batch, hw, c0, c1, g)
        p0 = _parts(x0, batch, hw, ppi0)
        p1 = _parts(x1, batch, hw, ppi1) if c1 else None
        C, n = c0 + c1, batch * hw
        out = _nan((n + BAND, C), torch.bfloat16)
        rawo = _nan((n + BAND, C), torch.bfloat16) if raw else None
        ops.groupnorm_silu_parts(x0, x1, p0, p1, gamma, beta, out[:n], batch, hw, groups, eps, silu,
                                 raw_out=rawo[:n] if raw else None)
        torch.cuda.synchronize()
        x = torch.cat([x0, x1], 1) if x1 is not None else x0
        if raw:
            assert torch.equal(rawo[:n], x.bfloat16()) and torch.isnan(rawo[n:]).all()
        _gn_compare("groupnorm_silu_parts", (batch, hw, c0, c1, ppi0, ppi1), out, x, batch, hw, gamma, beta, eps, silu)


# ---------------------------------------------------------------------------------------------------------------------------------
# LayerNorm, small_linear, cast_act, timestep embedding
# ---------------------------------------------------------------------------------------------------------------------------------
def test_layernorm_engine_signatures(sigs):
    from b200sd import ops
    seen, _ = sigs
    keys = sorted(seen["layernorm"], key=str)
    assert max(k[0] for k in keys) == 128 * 6144
    g = torch.Generator(device=DEV).manual_seed(9)
    for rows, C, dt, odt, eps in keys:
        x = (torch.randn(rows, C, generator=g, device=DEV) * 2 + torch.randn(rows, 1, generator=g, device=DEV) * 3).to(dt)
        gamma = 1 + 0.2 * torch.randn(C, generator=g, device=DEV)
        beta = 0.2 * torch.randn(C, generator=g, device=DEV)
        out = _nan((rows + BAND, C), odt)
        ops.layernorm(x, gamma, beta, out[:rows], eps)
        torch.cuda.synchronize()
        assert torch.isnan(out[rows:]).all()
        worst = 0.0
        for i in range(0, rows, 65536):
            xd = x[i:i + 65536].double()
            ref = F.layer_norm(xd, (C,), gamma.double(), beta.double(), eps)
            r = float((xd.mean(1).abs() / xd.std(1, unbiased=False)).max())
            c = float(((out[:rows][i:i + 65536].double() - ref).abs() - RHO * ref.abs()).max()) / float(ref.abs().max())
            bar = U * (16 + 8 * r + 2 * r * r)
            assert c <= bar, (rows, C, i, c, bar)
            worst = max(worst, c / bar)
        print(f"layernorm rows={rows} C={C} {dt}->{odt}: worst chunk at {worst:.3f} of its bar")


def test_small_linear_engine_signatures(sigs):
    from b200sd import ops
    seen, _ = sigs
    keys = sorted(seen["small_linear"], key=str)
    assert {k[0] for k in keys} >= {1, 2, 3, 16, 128} and {(k[4], k[5]) for k in keys} >= {(False, True), (True, False)}
    for B, N, K, has_bias, silu_in, silu_out in keys:
        g = torch.Generator(device=DEV).manual_seed(B * 131 + N + K)
        x = torch.randn(B, K, generator=g, device=DEV) * 2
        w = (torch.randn(N, K, generator=g, device=DEV) / math.sqrt(K)).bfloat16()
        b = torch.randn(N, generator=g, device=DEV) if has_bias else None
        out = _nan((B + 3, N), torch.float32)
        ops.small_linear(x, w, b, silu_in=silu_in, silu_out=silu_out, out=out[:B])
        torch.cuda.synchronize()
        assert torch.isnan(out[B:]).all()
        xin = _silu64(x.double()) if silu_in else x.double()
        pre = xin @ w.double().T + (b.double() if b is not None else 0.0)
        ref = _silu64(pre) if silu_out else pre
        mag = xin.abs() @ w.double().abs().T + (b.double().abs() if b is not None else 0.0)
        bar = (math.ceil(K / 32) + 10) * U * mag + 4 * U * ref.abs()
        r = float(((out[:B].double() - ref).abs() / bar).max())
        print(f"small_linear B={B} N={N} K={K} silu_in={silu_in} silu_out={silu_out}: worst {r:.3f} of the gamma_n bar")
        assert r <= 1.0


def test_cast_act_engine_signatures(sigs):
    from b200sd import ops
    seen, _ = sigs
    for n, silu in sorted(seen["cast_act"]):
        x = torch.randn(n, generator=torch.Generator(device=DEV).manual_seed(n), device=DEV) * 4
        out = _nan((n + 64,), torch.bfloat16)
        ops.cast_act(x, out[:n], silu=silu)
        torch.cuda.synchronize()
        assert torch.isnan(out[n:]).all()
        ref = _silu64(x.double()) if silu else x.double()
        c = float(((out[:n].double() - ref).abs() - RHO * ref.abs()).max() / ref.abs().max())
        print(f"cast_act n={n} silu={silu}: |err| - 2^-8 |ref| = {c:.3g} max|ref| (bar 2^-20)")
        assert c <= 2.0 ** -20


def test_timestep_embedding_fractional_t(sigs):
    from b200sd import ops
    seen, _ = sigs
    for B, dim in sorted(seen["timestep_embedding"]):
        g = torch.Generator(device=DEV).manual_seed(B)
        t = torch.rand(B, generator=g, device=DEV) * 999.0
        t[0] = 999.0
        t[-1] = 0.4375
        out = _nan((B + 2, dim), torch.float32)
        ops.timestep_embedding(t, dim, out=out[:B])
        torch.cuda.synchronize()
        assert torch.isnan(out[B:]).all()
        half = dim // 2
        f = torch.exp(-math.log(10000.0) * torch.arange(half, device=DEV, dtype=torch.float64) / half)
        arg = t.double()[:, None] * f[None]
        ref = torch.cat([torch.cos(arg), torch.sin(arg)], 1)
        bar = 24 * U * torch.cat([arg.abs(), arg.abs()], 1) + 4 * U
        r = float(((out[:B].double() - ref).abs() / bar).max())
        print(f"timestep_embedding B={B} dim={dim}: worst {r:.3f} of the 24 u |t f| bar")
        assert r <= 1.0


# ---------------------------------------------------------------------------------------------------------------------------------
# conv_in, conv_out (CUDA cores and the batch >= 8 tensor-core pair), nhwc_bias_to_nchw, upsample2x, im2col_s2
# ---------------------------------------------------------------------------------------------------------------------------------
def test_conv_in_engine_signatures(sigs):
    from b200sd import ops
    from b200sd.packing import pack_conv3x3_f32
    seen, _ = sigs
    for (B, Cin, H, W), Cout, odt in sorted(seen["conv_in"], key=str):
        g = torch.Generator(device=DEV).manual_seed(B + H)
        x = torch.randn(B, Cin, H, W, generator=g, device=DEV)
        w = torch.randn(Cout, Cin, 3, 3, generator=g, device=DEV) / 6
        b = torch.randn(Cout, generator=g, device=DEV)
        n = B * H * W
        out = _nan((n + BAND, Cout), odt)
        ops.conv_in(x, pack_conv3x3_f32(w), b, out[:n])
        torch.cuda.synchronize()
        assert torch.isnan(out[n:]).all()
        imgs = _sample_images(B)
        got = out[:n].reshape(B, H, W, Cout)[imgs].double()
        ref = F.conv2d(x[imgs].double(), w.double(), b.double(), padding=1).permute(0, 2, 3, 1)
        mag = (F.conv2d(x[imgs].double().abs(), w.double().abs(), padding=1) + b.double().abs()[:, None, None]).permute(0, 2, 3, 1)
        rho = RHO if odt == torch.bfloat16 else 0.0
        r = float(((got - ref).abs() / (rho * ref.abs() + 40 * U * mag)).max())
        print(f"conv_in B={B} {H}x{W} -> {odt}: worst {r:.3f} of the 40 u bar")
        assert r <= 1.0


def _conv_out_case(B, H, W, Cin, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(B * H * W, Cin, generator=g, device=DEV).bfloat16()
    w = torch.randn(4, Cin, 3, 3, generator=g, device=DEV) / math.sqrt(9 * Cin)
    b = torch.randn(4, generator=g, device=DEV)
    imgs = _sample_images(B)
    xd = x.reshape(B, H, W, Cin)[imgs].permute(0, 3, 1, 2).double()
    ref = F.conv2d(xd, w.double(), b.double(), padding=1)
    mag = F.conv2d(xd.abs(), w.double().abs(), padding=1) + b.double().abs()[:, None, None]
    return x, w, b, imgs, ref, mag


def test_conv_out_engine_signatures(sigs):
    """CUDA-core conv_out (batch < 8) and the tensor-core conv_out GEMM on [x | x] . [w_hi | w_lo] + nhwc_bias_to_nchw
    (batch >= 8), both against float64 conv2d with the fp32 weights."""
    from b200sd import ops
    from b200sd.packing import pack_conv3x3_f32, pack_conv_out_tc
    seen, _ = sigs
    shapes = {k[0] for k in seen["conv_out"]} | {k[0] for k in seen["nhwc_bias_to_nchw"]}
    assert any(s[0] >= 8 for s in shapes) and any(s[0] < 8 for s in shapes)
    for (B, C4, H, W) in sorted(shapes):
        x, w, b, imgs, ref, mag = _conv_out_case(B, H, W, 320, B * 7 + H)
        out = _nan((B + 1, 4, H, W), torch.float32)
        if B >= 8:
            tmp = _nan((B * H * W, 32), torch.float32)
            ops.gemm(x, pack_conv_out_tc(w), tmp, a1=x, conv=(B, H, W))
            ops.nhwc_bias_to_nchw(tmp, b, out[:B])
            bar_w = 2.0 ** -16            # hi + lo carries the fp32 weights to ~2^-17 relative
            path = "tensor cores"
        else:
            ops.conv_out(x, pack_conv3x3_f32(w), b, out[:B])
            bar_w = 0.0
            path = "CUDA cores"
        torch.cuda.synchronize()
        assert torch.isnan(out[B:]).all()
        got = out[:B][imgs].double()
        bar = (bar_w + _k_acc(2 * 9 * 320) * U) * mag
        r = float(((got - ref).abs() / bar).max())
        print(f"conv_out ({path}) B={B} {H}x{W}: worst {r:.3f} of the bar")
        assert r <= 1.0


def test_nhwc_bias_to_nchw_every_channel():
    from b200sd import ops
    g = torch.Generator(device=DEV).manual_seed(3)
    for B, C, hw, ld in ((1, 4, 4096, 32), (3, 4, 6144, 32), (2, 3, 64, 4), (2, 8, 100, 8)):
        x = torch.randn(B * hw, ld, generator=g, device=DEV)
        b = torch.randn(C, generator=g, device=DEV) * 10
        out = _nan((B + 1, C, hw), torch.float32)
        ops.nhwc_bias_to_nchw(x, b, out[:B].reshape(B, C, hw, 1))
        torch.cuda.synchronize()
        assert torch.isnan(out[B:]).all()
        want = (x[:, :C] + b).reshape(B, hw, C).permute(0, 2, 1)
        assert torch.equal(out[:B], want), (B, C, hw, ld)


def test_upsample2x_and_im2col_s2_bit_exact(sigs):
    from b200sd import ops
    seen, _ = sigs
    for B, H, W, C, dt in sorted(seen["upsample2x"], key=str):
        x = torch.randn(B * H * W, C, device=DEV).to(dt)
        n = B * 4 * H * W
        out = _nan((n + BAND, C), torch.bfloat16)
        ops.upsample2x(x, out[:n], B, H, W)
        torch.cuda.synchronize()
        want = F.interpolate(x.float().reshape(B, H, W, C).permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest")
        assert torch.equal(out[:n], want.permute(0, 2, 3, 1).reshape(n, C).bfloat16()) and torch.isnan(out[n:]).all()
    for B, H, W, C, dt, pad in sorted(seen["im2col_s2"], key=str):
        x = torch.randn(B * H * W, C, device=DEV).to(dt)
        n = B * (H // 2) * (W // 2)
        out = _nan((n + BAND, 9 * C), torch.bfloat16)
        ops.im2col_s2(x, out[:n], B, H, W, pad)
        torch.cuda.synchronize()
        cols = F.unfold(x.float().reshape(B, H, W, C).permute(0, 3, 1, 2), 3, padding=pad, stride=2)   # [B, C*9, L]
        want = cols.reshape(B, C, 9, -1).permute(0, 3, 2, 1).reshape(n, 9 * C)
        assert torch.equal(out[:n], want.bfloat16()) and torch.isnan(out[n:]).all(), (B, H, W, C)
    print(f"upsample2x {len(seen['upsample2x'])} and im2col_s2 {len(seen['im2col_s2'])} signatures bit-exact")


# ---------------------------------------------------------------------------------------------------------------------------------
# attention
# ---------------------------------------------------------------------------------------------------------------------------------
def _attn_rows(q, k, v, scale):
    """float64 softmax(q k^T scale) v and sum_j p_j |v_j| for one (batch, head): q [Sq, d], k / v [Skv, d]."""
    qd, kd, vd = q.double(), k.double(), v.double()
    outs, pvs = [], []
    for i in range(0, qd.shape[0], 2048):
        p = torch.softmax(qd[i:i + 2048] @ kd.T * scale, -1)
        outs.append(p @ vd)
        pvs.append(p @ vd.abs())
    return torch.cat(outs), torch.cat(pvs)


def _attn_check(out, q, k, v, batch, heads, Sq, Skv, d, scale, bhs):
    C = heads * d
    worst = 0.0
    for b, h in bhs:
        got = out[b * Sq:(b + 1) * Sq, h * d:(h + 1) * d].double()
        ref, pv = _attn_rows(q[b, :, h], k[b, :, h], v[b, :, h], scale)
        bar = RHO * ref.abs() + ATTN_C * RHO * pv
        r = float(((got - ref).abs() / bar).max())
        assert r <= 1.0, (batch, Sq, Skv, d, b, h, r)
        worst = max(worst, r)
    return worst


def test_attention_engine_signatures(sigs):
    """Engine strides (fused qkv ld = 3C; cross kv ld = 2C), sharp scores with a ramp (every 64-key tile raises the row max),
    NaN sentinel rows around the output; every (batch, head) at small batches, sampled ones (the last included) at large."""
    from b200sd import ops
    seen, _ = sigs
    for key in sorted(seen["attention"], key=str):
        batch, heads, Sq, Skv, d, ldq, ldk, ldv, ldo, q_off, k_off, v_off, fused = key
        C = heads * d
        g = torch.Generator(device=DEV).manual_seed(Sq * 3 + Skv + batch)
        scale = d ** -0.5
        dirn = torch.ones(d, device=DEV) / math.sqrt(d)
        qn = (torch.randn(batch, Sq, heads, d, generator=g, device=DEV) * 2 + 6 * dirn).bfloat16()
        ramp = torch.arange(Skv, device=DEV, dtype=torch.float32) / max(Skv - 1, 1) * 6
        kn = (torch.randn(batch, Skv, heads, d, generator=g, device=DEV) * 2 + ramp[None, :, None, None] * dirn).bfloat16()
        vn = torch.randn(batch, Skv, heads, d, generator=g, device=DEV).bfloat16()
        if fused:
            assert Sq == Skv and ldq == ldk == ldv == 3 * C and (k_off, v_off) == (C, 2 * C)
            qb = torch.cat([qn.reshape(batch * Sq, C), kn.reshape(batch * Sq, C), vn.reshape(batch * Sq, C)], 1).contiguous()
            kb = vb = qb
        else:
            assert (ldq, ldk, ldv, k_off, v_off) == (C, 2 * C, 2 * C, 0, C)
            qb = qn.reshape(batch * Sq, C).contiguous()
            kb = vb = torch.cat([kn.reshape(batch * Skv, C), vn.reshape(batch * Skv, C)], 1).contiguous()
        n = batch * Sq
        outb = _nan((n + 2 * BAND, C), torch.bfloat16)
        out = outb[BAND:BAND + n]
        ops.attention(qb, kb, vb, out, batch, heads, Sq, Skv, d, scale, ldq=ldq, ldk=ldk, ldv=ldv, ldo=ldo, q_off=q_off,
                      k_off=k_off, v_off=v_off)
        torch.cuda.synchronize()
        assert torch.isnan(outb[:BAND]).all() and torch.isnan(outb[BAND + n:]).all(), "attention wrote outside its rows"
        if batch <= 3:
            bhs = [(b, h) for b in range(batch) for h in (range(heads) if Sq <= 1536 else (0, heads - 1))]
        else:
            bhs = [(0, 0), (batch // 2, 3), (batch - 1, heads - 1)]
        w = _attn_check(out, qn, kn, vn, batch, heads, Sq, Skv, d, scale, bhs)
        print(f"attention {'self' if fused else 'cross'} B={batch} Sq={Sq} Skv={Skv} d={d}: worst row at {w:.3f} of its bar")


@pytest.mark.parametrize("d", [40, 80, 160])
def test_attention_polynomial_exponential_lanes(d):
    """Every query row: key 0 scores 0 (v = 0), the other 63 keys score -6.5 in log2 units exactly (scale_log2 = 1, f = -1/2,
    the middle of the polynomial's range); v = 1 on the keys of the score pairs that take poly_exp2x2 (every 4th pair: keys
    8m + 6, 8m + 7) and 0 elsewhere, so the output is the polynomial's exponentials alone over the row sum."""
    from b200sd import ops
    Sq, Skv = 256, 64
    scale = float(torch.tensor(math.log(2.0), dtype=torch.float32))
    q = torch.zeros(Sq, d, device=DEV)
    q[:, 0] = 1.0
    k = torch.zeros(Skv, d, device=DEV)
    k[1:, 0] = -6.5
    v = torch.zeros(Skv, d, device=DEV)
    lanes = torch.tensor([j for j in range(Skv) if j % 8 in (6, 7)], device=DEV)
    v[lanes] = 1.0
    qb, kb, vb = q.bfloat16(), k.bfloat16(), v.bfloat16()
    outb = _nan((Sq + 2 * BAND, d), torch.bfloat16)
    out = outb[BAND:BAND + Sq]
    ops.attention(qb, kb, vb, out, 1, 1, Sq, Skv, d, scale)
    torch.cuda.synchronize()
    assert torch.isnan(outb[:BAND]).all() and torch.isnan(outb[BAND + Sq:]).all()
    ref, pv = _attn_rows(qb, kb, vb, scale)
    err = (out.double() - ref).abs()
    c = float(((err - RHO * ref.abs()) / (RHO * pv)).max())
    print(f"attention poly_exp2x2 lanes d={d}: (|err| - 2^-8 |ref|) = {c:.3g} 2^-8 sum p|v| (bar {ATTN_C})")
    assert c <= ATTN_C
