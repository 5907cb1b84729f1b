"""Generate tests/golden/reference_pins.pt by RUNNING THE REFERENCE'S OWN CODE (imported by path from a
checkout of diffusion-e2e-ft, read-only) on seeded inputs.  Only the reference files that import without diffusers
can be run:

    training/util/loss.py                        ScaleAndShiftInvariantLoss, AngularLoss   (+ autograd gradients)
    training/util/unet_prep.py                   replace_unet_conv_in
    GeoWizard/geowizard/utils/normal_ensemble.py ensemble_normals
    Marigold/marigold/util/ensemble.py           ensemble_depths (scipy BFGS)
    Marigold/src/util/metric.py                  abs_relative_difference (+ the other depth metrics)
    Marigold/src/util/alignment.py               align_depth_least_square

The UNet / VAE arithmetic itself lives in diffusers==0.30.2 (absent, not installable offline) and stays pinned only
by the oracle restatement (SURVEY.md §8c).  The tests run without the reference, so the outputs are committed as a
small fixture and tests/test_reference_pins.py compares the oracle AND the CUDA kernels with it.

    python tests/golden/make_reference_pins.py <checkout>            -> reference_pins.pt
    python tests/golden/make_reference_pins.py --record <checkout>   -> reference_recorded.npz (see record())
"""
import importlib.util
import os
import sys

import numpy as np
import torch

REF = None                 # the reference checkout, from the command line
HERE = os.path.dirname(os.path.abspath(__file__))


def load_ref(rel, name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def gen(seed):
    return torch.Generator().manual_seed(seed)


def loss_inputs():
    g = gen(101)
    pred_d = torch.randn(2, 1, 40, 48, generator=g) * 0.3
    gt_d = torch.rand(2, 1, 40, 48, generator=g) * 9.9 + 0.1
    mask = torch.rand(2, 1, 40, 48, generator=g) > 0.2
    pred_n = torch.nn.functional.normalize(torch.randn(2, 3, 40, 48, generator=g), dim=1) * 0.98
    gt_n = torch.nn.functional.normalize(torch.randn(2, 3, 40, 48, generator=g), dim=1)
    return pred_d, gt_d, mask, pred_n, gt_n


def main():
    torch.set_num_threads(4)
    loss = load_ref("training/util/loss.py", "ref_loss")
    prep = load_ref("training/util/unet_prep.py", "ref_unet_prep")
    nens = load_ref("GeoWizard/geowizard/utils/normal_ensemble.py", "ref_normal_ensemble")
    ens = load_ref("Marigold/marigold/util/ensemble.py", "ref_ensemble")
    metric = load_ref("Marigold/src/util/metric.py", "ref_metric")
    align = load_ref("Marigold/src/util/alignment.py", "ref_alignment")
    out = {}

    # ---- losses + their autograd gradients (training/train.py:542-563 path)
    pred_d, gt_d, mask, pred_n, gt_n = loss_inputs()
    p = pred_d.clone().requires_grad_(True)
    l = loss.ScaleAndShiftInvariantLoss()(p, gt_d, mask)
    l.backward()
    out["ssi"] = dict(pred=pred_d, target=gt_d, mask=mask, loss=l.detach(), grad=p.grad.clone())
    sc, sh = loss.compute_scale_and_shift_masked(pred_d.squeeze(1), gt_d.squeeze(1), mask.squeeze(1))
    out["ssi"]["scale"], out["ssi"]["shift"] = sc, sh
    p = pred_n.clone().requires_grad_(True)
    l = loss.AngularLoss()(p, gt_n, mask)
    l.backward()
    out["angular"] = dict(pred=pred_n, target=gt_n, mask=mask, loss=l.detach(), grad=p.grad.clone())

    # ---- replace_unet_conv_in on a stand-in module exposing conv_in / config (unet_prep.py:6-21)
    class Stub(torch.nn.Module):
        def __init__(self):
            super().__init__()
            torch.manual_seed(7)
            self.conv_in = torch.nn.Conv2d(4, 16, 3, padding=1)
            self.config = {"in_channels": 4}
    st = Stub()
    w0, b0 = st.conv_in.weight.detach().clone(), st.conv_in.bias.detach().clone()
    prep.replace_unet_conv_in(st, repeat=2)
    out["conv_in"] = dict(w0=w0, b0=b0, w=st.conv_in.weight.detach().clone(), b=st.conv_in.bias.detach().clone(),
                          in_channels=st.config["in_channels"])

    # ---- normals ensembling (index must be bit-exact: marigold_pipeline.py:59-71 / normal_ensemble.py:6-22)
    cases = {}
    for name, (seed, shape) in dict(a=(7, (6, 3, 32, 32)), b=(6, (10, 3, 24, 40)), c=(3, (3, 3, 17, 19))).items():
        preds = torch.randn(*shape, generator=gen(seed))
        if name == "b":                      # correlated ensemble members, as real predictions are
            base = torch.randn(1, *shape[1:], generator=gen(9))
            preds = base + 0.3 * preds
        got = nens.ensemble_normals(preds)
        nrm = preds / (torch.norm(preds, p=2, dim=1).unsqueeze(1) + 1e-5)
        idx = [i for i in range(shape[0]) if torch.equal(nrm[i], got)]
        assert len(idx) == 1
        cases[name] = dict(preds=preds, out=got, index=idx[0])
    out["ensemble_normals"] = cases

    # ---- depth metrics + least-squares alignment (Marigold/eval.py protocol)
    g = gen(55)
    gt = torch.rand(2, 48, 64, generator=g) * 9.5 + 0.5
    pr = (gt - 0.5) / 9.5 * 0.8 + 0.1 + 0.02 * torch.randn(2, 48, 64, generator=g)
    vm = torch.rand(2, 48, 64, generator=g) > 0.1
    al, s, t = align.align_depth_least_square(gt[0].numpy(), pr[0].numpy(), vm[0].numpy())
    al_t = torch.from_numpy(np.asarray(al)).float()
    out["align"] = dict(gt=gt[0], pred=pr[0], mask=vm[0], aligned=al_t, scale=float(np.asarray(s).reshape(-1)[0]),
                        shift=float(np.asarray(t).reshape(-1)[0]))
    aligned2 = torch.stack([al_t, torch.from_numpy(np.asarray(
        align.align_depth_least_square(gt[1].numpy(), pr[1].numpy(), vm[1].numpy(), return_scale_shift=False))).float()])
    aligned2 = aligned2.clamp(0.5, 10.0)
    mets = {}
    for fn in ("abs_relative_difference", "squared_relative_difference", "rmse_linear", "rmse_log", "log10",
               "delta1_acc", "delta2_acc", "delta3_acc", "i_rmse", "silog_rmse"):
        if hasattr(metric, fn):
            mets[fn] = dict(masked=torch.as_tensor(getattr(metric, fn)(aligned2.clone(), gt.clone(), vm.clone())).clone())
            try:
                mets[fn]["full"] = torch.as_tensor(getattr(metric, fn)(aligned2.clone(), gt.clone())).clone()
            except TypeError:
                pass                                       # metrics that require the mask argument
    out["metrics"] = dict(pred=aligned2, gt=gt, mask=vm, values=mets)

    # ---- depth ensembling (Marigold/marigold/util/ensemble.py:40-132)
    g = gen(77)
    base = torch.rand(1, 48, 64, generator=g)
    sc = 0.5 + torch.rand(5, 1, 1, generator=g)
    sh = 0.2 * torch.randn(5, 1, 1, generator=g)
    members = (base * sc + sh + 0.01 * torch.randn(5, 48, 64, generator=g)).float()
    ed = {}
    for red in ("median", "mean"):
        a, u = ens.ensemble_depths(members.clone(), regularizer_strength=0.02, max_iter=2, tol=1e-3, reduction=red)
        ed[red] = dict(aligned=a.clone(), uncertainty=u.clone())
    out["ensemble_depths"] = dict(members=members, results=ed)

    path = os.path.join(HERE, "reference_pins.pt")
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path), "bytes")


def record():
    """Re-run two reference functions on the inputs stored in reference_pins.pt and keep their outputs in
    reference_recorded.npz, a record separate from the fixture: tests/test_reference_pins.py checks the fixture's
    outputs against it bit for bit, so a regenerated or edited fixture cannot drift from what the reference computes."""
    loss = load_ref("training/util/loss.py", "ref_loss")
    nens = load_ref("GeoWizard/geowizard/utils/normal_ensemble.py", "ref_normal_ensemble")
    pins = torch.load(os.path.join(HERE, "reference_pins.pt"))
    s = pins["ssi"]
    rec = {"ssi_loss": loss.ScaleAndShiftInvariantLoss()(s["pred"], s["target"], s["mask"]).detach().numpy()}
    for name, case in pins["ensemble_normals"].items():
        rec[f"ensemble_normals_{name}"] = nens.ensemble_normals(case["preds"]).numpy()
    path = os.path.join(HERE, "reference_recorded.npz")
    np.savez(path, **rec)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if len(sys.argv) < 2 or not os.path.isdir(sys.argv[-1]):
        sys.exit("usage: make_reference_pins.py [--record] <checkout of diffusion-e2e-ft>")
    REF = sys.argv[-1]
    if "--record" in sys.argv[1:-1]:
        record()
    else:
        main()
