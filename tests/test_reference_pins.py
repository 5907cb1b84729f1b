"""Pins against the REFERENCE'S OWN CODE (VERDICT r1 weak #2 / next-round task 1a).

tests/golden/reference_pins.pt holds outputs of the reference's importable files — training/util/loss.py,
training/util/unet_prep.py, GeoWizard/geowizard/utils/normal_ensemble.py, Marigold/marigold/util/ensemble.py,
Marigold/src/util/{metric,alignment}.py — run on seeded inputs by tests/golden/make_reference_pins.py (committed; the
tests run without the reference).  Here
  * not gpu: the ORACLE restatements must reproduce them, and the fixture must match a separate record of the reference's
    outputs (tests/golden/reference_recorded.npz), so a stale fixture cannot hide drift;
  * gpu: the CUDA kernels (losses forward + backward, normals / depth ensembling, min-max, resize) must reproduce them.
The UNet / VAE arithmetic itself lives in diffusers==0.30.2 (absent): it stays pinned by the oracle only (parity
"partial" by rule, DESIGN.md §4).
"""
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
from oracle import pipeline as OP  # noqa: E402
from oracle.unet import replace_unet_conv_in  # noqa: E402

PINS = os.path.join(HERE, "golden", "reference_pins.pt")
RECORDED = os.path.join(HERE, "golden", "reference_recorded.npz")


@pytest.fixture(scope="module")
def pins():
    return torch.load(PINS)


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


# ------------------------------------------------------------------------------------------------ oracle vs reference
def test_oracle_losses_match_reference(pins):
    s = pins["ssi"]
    p = s["pred"].clone().requires_grad_(True)
    l = OP.ssi_loss(p, s["target"], s["mask"])
    l.backward()
    assert torch.equal(l.detach(), s["loss"]) or abs(l.item() - s["loss"].item()) <= 1e-6 * abs(s["loss"].item())
    assert _rel(p.grad, s["grad"]) <= 1e-6
    sc, sh = OP.compute_scale_and_shift_masked(s["pred"].squeeze(1), s["target"].squeeze(1), s["mask"].squeeze(1))
    assert torch.allclose(sc, s["scale"], rtol=1e-6) and torch.allclose(sh, s["shift"], rtol=1e-6)
    a = pins["angular"]
    p = a["pred"].clone().requires_grad_(True)
    l = OP.angular_loss(p, a["target"], a["mask"])
    l.backward()
    assert abs(l.item() - a["loss"].item()) <= 1e-6 * abs(a["loss"].item())
    assert _rel(p.grad, a["grad"]) <= 1e-6


def test_oracle_replace_unet_conv_in_matches_reference(pins):
    c = pins["conv_in"]

    class Stub(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.conv_in = torch.nn.Conv2d(4, 16, 3, padding=1)
            self.config = {"in_channels": 4}
    st = Stub()
    with torch.no_grad():
        st.conv_in.weight.copy_(c["w0"])
        st.conv_in.bias.copy_(c["b0"])
    replace_unet_conv_in(st, repeat=2)
    assert torch.equal(st.conv_in.weight.detach(), c["w"]) and torch.equal(st.conv_in.bias.detach(), c["b"])
    assert st.config["in_channels"] == c["in_channels"] == 8


def test_oracle_ensemble_normals_index_bit_exact(pins):
    for name, case in pins["ensemble_normals"].items():
        got, idx = OP.ensemble_normals(case["preds"])
        assert idx == case["index"], name
        assert torch.equal(got, case["out"]), name


def test_oracle_metric_and_alignment_match_reference(pins):
    a = pins["align"]
    m = a["mask"]
    # oracle align_lstsq has no mask argument: restrict to the valid pixels, apply to the whole map
    pm, gm = a["pred"][m], a["gt"][m]
    x = torch.linalg.lstsq(torch.stack([pm, torch.ones_like(pm)], 1).double(), gm.double()[:, None]).solution
    assert abs(x[0].item() - a["scale"]) <= 1e-5 * abs(a["scale"]) and abs(x[1].item() - a["shift"]) <= 1e-4
    full = OP.align_lstsq(a["pred"][m], a["gt"][m])
    assert _rel(full, a["aligned"][m]) <= 1e-5
    met = pins["metrics"]
    want = met["values"]["abs_relative_difference"]["full"]
    got = OP.abs_rel(met["pred"], met["gt"])
    assert abs(got.item() - want.item()) <= 1e-6 * want.item()


def test_fixture_is_current_against_live_reference(pins):
    """Two of the reference functions, re-run on the fixture's own inputs in a separate pass
    (make_reference_pins.py --record): the committed fixture must hold exactly what the reference produced."""
    rec = np.load(RECORDED)
    s = pins["ssi"]
    assert torch.equal(s["loss"], torch.from_numpy(rec["ssi_loss"]))
    assert sorted(pins["ensemble_normals"]) == ["a", "b", "c"]
    for name, case in pins["ensemble_normals"].items():
        assert torch.equal(case["out"], torch.from_numpy(rec[f"ensemble_normals_{name}"])), name


# ------------------------------------------------------------------------------------------------ CUDA vs reference
@pytest.mark.gpu
def test_cuda_loss_kernels_match_reference(pins):
    from diffusion_e2e_ft_b200 import ops
    one = torch.ones((), device="cuda")
    s = pins["ssi"]
    p, t, m = s["pred"].cuda(), s["target"].cuda(), s["mask"].cuda()
    assert abs(ops.ssi_loss(p, t, m).item() - s["loss"].item()) <= 2e-6 * abs(s["loss"].item())
    assert _rel(ops.ssi_loss_bwd(p, t, m, one), s["grad"]) <= 2e-5
    a = pins["angular"]
    p, t, m = a["pred"].cuda(), a["target"].cuda(), a["mask"].cuda()
    assert abs(ops.angular_loss(p, t, m).item() - a["loss"].item()) <= 2e-6 * abs(a["loss"].item())
    assert _rel(ops.angular_loss_bwd(p, t, m, one), a["grad"]) <= 2e-5


@pytest.mark.gpu
def test_cuda_ensemble_normals_index_bit_exact(pins):
    """north_star: bit-exact for index/argmax in the ensembling path."""
    from diffusion_e2e_ft_b200 import ensemble_normals_with_index
    for name, case in pins["ensemble_normals"].items():
        got, idx = ensemble_normals_with_index(case["preds"].cuda())
        assert int(idx) == case["index"], (name, int(idx), case["index"])
        assert torch.allclose(got.cpu(), case["out"], rtol=0, atol=2e-7), name      # same member; x / (|x| + 1e-5) in fp32


@pytest.mark.gpu
def test_cuda_ensemble_depths_matches_reference(pins):
    from diffusion_e2e_ft_b200 import ensemble_depths
    e = pins["ensemble_depths"]
    for red, want in e["results"].items():
        a, u = ensemble_depths(e["members"].cuda(), regularizer_strength=0.02, max_iter=2, tol=1e-3, reduction=red)
        assert _rel(a, want["aligned"]) <= 2e-5, (red, _rel(a, want["aligned"]))
        assert _rel(u, want["uncertainty"]) <= 2e-4, (red, _rel(u, want["uncertainty"]))


@pytest.mark.gpu
def test_cuda_replace_unet_conv_in_on_engine_unet(pins):
    """training/util/unet_prep.py:6-21 (weights duplicated, weights AND bias divided by `repeat`) applied by the same
    rule to the ENGINE module and to the oracle: the widened engine UNet must match the widened oracle UNet, and —
    because the bias is halved too (a reference quirk, SURVEY.md App. C) — it must NOT reproduce the 4-channel output."""
    import make_golden as MG
    import engine_checks as EC
    from oracle.unet import UNet2DConditionRef, tiny_config, seeded_init
    ref4 = seeded_init(UNet2DConditionRef(tiny_config(in_channels=4)), seed=1234).eval()
    unet, _ = EC.engine_from_oracle(ref4, None, "cuda:0")
    x4 = MG.inputs(31, 2, 4, 16, 16)
    x8 = torch.cat([x4, x4], 1)
    ctx = MG.inputs(32, 2, 2, 128, scale=0.5)
    with torch.no_grad():
        y4 = unet(x4.cuda(), 999, ctx.cuda()).sample
        assert EC.rel_l2(y4, ref4(x4, 999, ctx).sample) <= 3e-3
        replace_unet_conv_in(unet, repeat=2)
        replace_unet_conv_in(ref4, repeat=2)
        assert unet.config["in_channels"] == 8 and unet.conv_in.weight.shape[1] == 8
        assert torch.equal(unet.conv_in.weight.detach().cpu(), ref4.conv_in.weight.detach())
        y8 = unet(x8.cuda(), 999, ctx.cuda()).sample
        want8 = ref4(x8, 999, ctx).sample
    assert EC.rel_l2(y8, want8) <= 3e-3
    assert EC.rel_l2(y8, y4) > 1e-2                      # halved bias: the widened model is a different function


@pytest.mark.gpu
def test_cuda_preprocessing_matches_torchvision_semantics():
    """marigold_pipeline.py:237-247,315-321: antialiased bilinear resize (down and up), uint8 rounding, [-1,1] map and
    min-max normalisation against torch.nn.functional.interpolate(antialias=True) (what torchvision's resize calls)."""
    from diffusion_e2e_ft_b200.ensemble import minmax_normalise_, normalise_rgb, resize_bilinear_aa, resize_nearest
    g = torch.Generator().manual_seed(5)
    img = torch.randint(0, 256, (3, 480, 640), generator=g, dtype=torch.uint8)
    F = torch.nn.functional
    for size in ((360, 480), (576, 768), (97, 131), (480, 640)):
        want = F.interpolate(img[None].float(), size=size, mode="bilinear", antialias=True, align_corners=False)[0]
        got = resize_bilinear_aa(img.cuda().float(), size)
        assert (got.cpu() - want).abs().max().item() <= 1e-2, size                  # values in [0, 255]: 4e-5 relative
        want_n = torch.round(want).clamp(0, 255) / 255.0 * 2.0 - 1.0
        got_n = normalise_rgb(got, round_u8=True).cpu()
        # round-half-even on x.5 ties (frequent for 4:3 scale factors) flips with the last bit of the float sum: a
        # differing pixel is off by exactly one uint8 level, and only a few per cent of the pixels are ties
        d = (got_n - want_n).abs()
        assert d.max().item() <= 2.0 / 255.0 + 1e-6 and (d > 1e-6).float().mean().item() <= 0.05, size
    d = torch.rand(1, 200, 300, generator=g) * 3 - 1
    got, mm = minmax_normalise_(d.cuda().clone())
    assert torch.allclose(got.cpu(), (d - d.min()) / (d.max() - d.min()), atol=1e-6)
    assert mm.tolist() == [d.min().item(), d.max().item()]
    n = torch.randn(3, 50, 70, generator=g)
    assert torch.equal(resize_nearest(n.cuda(), (120, 99)).cpu(), F.interpolate(n[None], size=(120, 99), mode="nearest")[0])
