"""Whole-path check against the committed golden outputs of the reference (tests/golden/net_*.npz, written by
oracle/make_golden.py from the unmodified reference): ERFNet -> activation -> mask -> LSQ -> backprojection loss,
forward + backward, through the same calls the reference's main.py makes (BP/main.py:286-305,338-339).

TEST INFRASTRUCTURE (used by tests/test_net_gpu.py and __graft_entry__.smoke()): it drives the product package on
cuda:0 and compares with the fixtures; nothing here is on the product path.

Gate (SURVEY.md 7.2 #1): |ours - fp64| <= 4 * |reference fp32 - fp64| + tol, norm-wise per tensor.
"""
import json
import os

import numpy as np
import torch

from . import inputs

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def build_net(L, order, mask_pct, B):
    from lanedetection_end2end_b200.Networks.utils import define_args
    from lanedetection_end2end_b200.Networks.LSQ_layer import Net
    args = define_args().parse_args(["--image_dir", "x", "--gt_dir", "y", "--nclasses", str(L), "--order", str(order),
                                     "--batch_size", str(B), "--mask_percentage", str(mask_pct),
                                     "--loss_policy", "backproject"])
    return Net(args), args


class FullPathCase:
    """Case `name` of the whole-path goldens, ready to run: the fixture `g` and its `meta`, the model with the golden
    parameters (cuda:0, train mode, dropout p = 0), the reference's `args`, and the inputs x, xgt, valid on cuda:0."""

    def __init__(self, name, golden_dir=GOLDEN):
        g = np.load(os.path.join(golden_dir, name + ".npz"))
        meta = json.loads(str(g["meta"]))
        L, order, B = meta["L"], meta["order"], meta["B"]
        model, args = build_net(L, order, meta["mask_pct"], B)
        sd = model.state_dict()
        for k, v in inputs.make_erfnet_params(3, L, seed=meta["param_seed"]).items():
            sd[k] = torch.from_numpy(v)
        model.load_state_dict(sd)
        model = model.cuda().train()
        for m in model.modules():
            if hasattr(m, "dropout"):
                m.dropout.p = 0
        # the grid must be bit-identical to the reference's (same torch ops on the same cv2 homography)
        np.testing.assert_array_equal(model.grid[0].cpu().numpy(), np.load(os.path.join(golden_dir, "lsq_bp_l2_d2.npz"))["grid0"])
        self.name, self.g, self.meta, self.model, self.args = name, g, meta, model, args
        self.L, self.order, self.B = L, order, B
        self.x = torch.from_numpy(inputs.make_images(B, 256, 512, seed=meta["image_seed"])).cuda()
        xgt_np, valid_np = inputs.make_loss_targets(B, 4, seed=meta["target_seed"])
        self.xgt, self.valid = torch.from_numpy(xgt_np).cuda(), torch.from_numpy(valid_np).cuda()

    def tap_modules(self):
        """The modules whose outputs the fixture samples, by fixture name."""
        net = self.model.net
        mods = {"encoder.initial_block": net.encoder.initial_block, "decoder.output_conv": net.decoder.output_conv}
        mods.update({"encoder.layers.%d" % i: l for i, l in enumerate(net.encoder.layers)})
        mods.update({"decoder.layers.%d" % i: l for i, l in enumerate(net.decoder.layers)})
        return mods

    def hook_taps(self):
        """Forward hooks that store each tapped module's latest output in the returned dict; returns (taps, handles)."""
        taps, hooks = {}, []
        for n, mod in self.tap_modules().items():
            hooks.append(mod.register_forward_hook(lambda _m, _i, o, n=n: taps.__setitem__(n, o)))
        return taps, hooks


def compare_full_path(case, taps, betas, loss, tol=1e-4, enforce=True):
    """Compare one training step of `case.model` with the golden: the sampled activations in `taps`, the curve
    coefficients `betas` (L tensors [B, order+1, 1] float64), the `loss`, every parameter gradient and the BatchNorm
    running statistics after one step.  Returns a report dict with the worst norm-wise errors (ours vs fp64,
    reference-fp32 vs fp64); with `enforce` every gate is asserted."""
    g, model = case.g, case.model
    assert len(betas) == case.L and betas[0].dtype == torch.float64 and betas[0].shape == (case.B, case.order + 1, 1)

    rep = {"case": case.name, "act": (0.0, 0.0, ""), "grad": (0.0, 0.0, ""), "grad_significant": (0.0, 0.0, "")}

    def check(ok, msg):
        if enforce:
            assert ok, msg

    # layer-wise activations (sampled entries)
    for n, t in taps.items():
        k64, k32 = "act_f64/%s" % n, "act_f32/%s" % n
        got = t.detach().double().cpu().contiguous().numpy().reshape(-1)[g[k64 + "/idx"]]
        scale = g[k64 + "/stat"][2]
        e_ours = float(np.abs(got - g[k64 + "/val"]).max() / scale)
        e_ref = float(np.abs(g[k32 + "/val"] - g[k64 + "/val"]).max() / scale)
        if e_ours > rep["act"][0]:
            rep["act"] = (e_ours, e_ref, n)
        check(e_ours <= 4 * e_ref + tol, ("activation", n, e_ours, e_ref))
    # curve coefficients, loss
    b64, b32 = g["beta_f64"], g["beta_f32"]
    ours = torch.stack([b.squeeze(-1) for b in betas], 1).detach().cpu().numpy()
    nw = lambda a, b: float((np.abs(a - b).max(-1) / np.abs(b).max(-1)).max())
    rep["beta"] = (nw(ours, b64), nw(b32, b64))
    check(rep["beta"][0] <= 4 * rep["beta"][1] + tol, ("beta", rep["beta"]))
    l64, l32 = float(g["loss_f64"]), float(g["loss_f32"])
    rep["loss"] = (abs(float(loss.detach()) - l64) / abs(l64), abs(l32 - l64) / abs(l64))
    check(rep["loss"][0] <= 4 * rep["loss"][1] + tol, ("loss", rep["loss"]))
    # parameter gradients (sampled entries)
    gscale = max(g[k][2] for k in g.files if k.startswith("grad_f64/") and k.endswith("/stat"))
    no_grad = set(json.loads(str(g["params_without_grad"])))
    for n, p in model.named_parameters():
        if n in no_grad:
            check(p.grad is None, n)
            continue
        k64, k32 = "grad_f64/" + n, "grad_f32/" + n
        got = p.grad.double().cpu().numpy().reshape(-1)[g[k64 + "/idx"]]
        scale = max(g[k64 + "/stat"][2], 1e-6 * gscale)
        e_ours = float(np.abs(got - g[k64 + "/val"]).max() / scale)
        e_ref = float(np.abs(g[k32 + "/val"] - g[k64 + "/val"]).max() / scale)
        if e_ours > rep["grad"][0]:
            rep["grad"] = (e_ours, e_ref, n)
        # the same, restricted to gradients that are not analytically zero (conv biases in front of a training-mode
        # BatchNorm are pure round-off on both sides: their "relative" error is O(1) for the reference as well)
        if g[k64 + "/stat"][2] >= 1e-3 * gscale and e_ours > rep["grad_significant"][0]:
            rep["grad_significant"] = (e_ours, e_ref, n)
        check(e_ours <= 4 * e_ref + 10 * tol, ("gradient", n, e_ours, e_ref))
    # BN running statistics after one step
    for n, b in model.named_buffers():
        if n.endswith("running_mean") or n.endswith("running_var"):
            ref = g["buf_f64/" + n]
            check(np.abs(b.cpu().numpy() - ref).max() <= 1e-4 * max(np.abs(ref).max(), 1e-3), n)
    return rep


def run_full_path(name, tol=1e-4, enforce=True, golden_dir=GOLDEN):
    """Run case `name` (net_l2_d2 / net_l4_d3 / net_l2_d2_b32) eagerly in the CURRENT ops_net.CONV_MODE: one forward
    and backward through the calls the reference's main.py makes, then compare_full_path."""
    from lanedetection_end2end_b200.Loss_crit import backprojection_loss
    case = FullPathCase(name, golden_dir)
    model, B, L = case.model, case.B, case.L
    taps, hooks = case.hook_taps()
    out = model(case.x, torch.zeros(B, 4), True)
    for h in hooks:
        h.remove()
    betas = [b for b in out[:4] if b is not None]
    crit = backprojection_loss(case.args)
    loss = sum(crit(betas[l], case.xgt[:, l], case.valid[:, l])[0] for l in range(L)) / L
    loss.backward()
    torch.cuda.synchronize()
    return compare_full_path(case, taps, betas, loss, tol, enforce)
