"""CPU test of the UNet walk every engine builds its plan with (UNet2DConditionModel._walk): block order, skip routing and
activation liveness, with recording callbacks instead of kernels: a callback that reads a released activation fails.  No GPU."""
import pytest
import torch

from oracle import unet_ref as U


def _walk(m):
    events, skips_of, live = [], {}, set()
    n = [0]

    def new(tag):
        n[0] += 1
        t = _Act()
        t.tag = f"{tag}#{n[0]}"
        live.add(t)
        return t

    def resnet(prefix, r, x, skip, h, w):
        assert x in live and (skip is None or skip in live), f"{prefix} reads a released activation"
        events.append(("resnet", prefix, h, w))
        skips_of[prefix] = skip
        return new(prefix)

    def xformer(prefix, a, x, h, w):
        assert x in live
        events.append(("xformer", prefix, h, w))
        return new(prefix)

    def downsample(prefix, s, x, h, w):
        assert x in live and s is not None
        events.append(("downsample", prefix, h, w))
        return new(prefix)

    def upsample(prefix, s, x, h, w):
        assert x in live and s is not None
        events.append(("upsample", prefix, h, w))
        return new(prefix)

    released = []

    def release(t):
        assert t in live, f"{t.tag} released twice"
        live.discard(t)
        released.append(t)

    x0 = new("conv_in")
    out, h, w = m._walk(x0, 16, 16, resnet=resnet, xformer=xformer, downsample=downsample, upsample=upsample, release=release)
    return events, skips_of, released, live, x0, out, (h, w), n[0]


class _Act:
    __slots__ = ("tag",)


def _expected_prefixes(m):
    want = []
    for i, b in enumerate(m.down_blocks):
        for j in range(len(b.resnets)):
            want.append(f"down{i}.res{j}")
            if hasattr(b, "attentions"):
                want.append(f"down{i}.attn{j}")
        if hasattr(b, "downsamplers"):
            want.append(f"down{i}.ds")
    want += ["mid.res0", "mid.attn0", "mid.res1"]
    for i, b in enumerate(m.up_blocks):
        for j in range(len(b.resnets)):
            want.append(f"up{i}.res{j}")
            if hasattr(b, "attentions"):
                want.append(f"up{i}.attn{j}")
        if hasattr(b, "upsamplers"):
            want.append(f"up{i}.us")
    return want


def _model(kind):
    from b200sd.unet import UNet2DConditionModel
    if kind == "tiny":
        return UNet2DConditionModel(**U.TINY_OVERRIDES)
    orig = UNet2DConditionModel.reset_parameters
    UNet2DConditionModel.reset_parameters = lambda self: None
    try:
        with torch.device("meta"):      # the SD v1.5 topology without allocating 3.4 GB
            return UNet2DConditionModel()
    finally:
        UNet2DConditionModel.reset_parameters = orig


@pytest.mark.parametrize("kind", ["tiny", "sd15"])
def test_walk_order_skips_and_liveness(kind):
    m = _model(kind)
    events, skips_of, released, live, x0, out, hw, produced = _walk(m)
    assert [e[1] for e in events] == _expected_prefixes(m)
    assert hw == (16, 16)

    # every up-resnet reads the activation its mirrored down step pushed: the stack of down outputs, popped in reverse
    pushed = [x0.tag]
    by_prefix = {}
    # re-derive the down outputs from the event order (each callback returned exactly one new activation, numbered in order)
    for k, (_kind, prefix, _h, _w) in enumerate(events):
        by_prefix[prefix] = k + 2            # x0 is #1
    for i, b in enumerate(m.down_blocks):
        for j in range(len(b.resnets)):
            last = f"down{i}.attn{j}" if hasattr(b, "attentions") else f"down{i}.res{j}"
            pushed.append(f"{last}#{by_prefix[last]}")
        if hasattr(b, "downsamplers"):
            pushed.append(f"down{i}.ds#{by_prefix[f'down{i}.ds']}")
    for i, b in enumerate(m.up_blocks):
        for j in range(len(b.resnets)):
            assert skips_of[f"up{i}.res{j}"].tag == pushed.pop(), f"up{i}.res{j}"
    assert not pushed
    assert all(skips_of[p] is None for p in skips_of if not p.startswith("up"))

    # release: exactly once for every produced activation except the output, and the output stays live
    assert len(released) == len(set(map(id, released))) == produced - 1
    assert live == {out} and out not in released

    # the spatial size each block runs at halves per downsampler and doubles back per upsampler
    sizes = {p: (h, w) for _k, p, h, w in events}
    assert sizes["down0.res0"] == (16, 16) and sizes["mid.attn0"] == (16 >> (len(m.down_blocks) - 1),) * 2
    assert sizes[f"up{len(m.up_blocks) - 1}.res0"] == (16, 16)

