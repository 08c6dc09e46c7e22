"""Generate tests/golden/*.npz by running the UNMODIFIED reference on CPU
(TEST INFRASTRUCTURE; ``LANEFIT_REFERENCE=<checkout of the original project> python -m oracle.make_golden``;
without the variable, oracle/reference_import.py picks the oracle/_ref/ install or the default checkout).

The reference has no golden vectors of its own (SURVEY.md 8c), so these files
are the pin: outputs of the reference's own modules (float32 = its arithmetic,
float64 = the same modules cast to double, the arbiter) on inputs that
``oracle/inputs.py`` regenerates bit-identically anywhere (sha256 stored).
"""
import json
import os
import sys
import zlib

import numpy as np
import torch

from . import inputs
from . import reference_import as ri

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
N_ACT_SAMPLES = 256
N_GRAD_SAMPLES = 64


def sample_indices(name, numel, k):
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    return rng.integers(0, numel, size=min(k, numel)).astype(np.int64)


def summarize(prefix, t, k, out):
    a = t.detach().double().numpy().reshape(-1)
    idx = sample_indices(prefix, a.size, k)
    out[prefix + "/idx"] = idx
    out[prefix + "/val"] = a[idx]
    out[prefix + "/stat"] = np.array([a.mean(), a.std(), np.abs(a).max(), np.sqrt((a * a).sum())])


# ---------------------------------------------------------------------------
# LSQ-layer goldens
# ---------------------------------------------------------------------------

LSQ_CASES = [
    # name, variant, L, order, mask_pct, act, reg_ls, cholesky, maps, B
    ("bp_l2_d2", "Backprojection_Loss", 2, 2, 0.3, "square", 0.0, False, "lane", 2),
    ("bp_l4_d3", "Backprojection_Loss", 4, 3, 0.2, "square", 0.0, False, "lane", 2),
    ("bp_l2_d1", "Backprojection_Loss", 2, 1, 0.3, "square", 0.0, False, "lane", 2),
    ("bp_l2_d2_chol", "Backprojection_Loss", 2, 2, 0.3, "square", 0.0, True, "lane", 2),
    ("bp_l2_d2_reg_relu", "Backprojection_Loss", 2, 2, 0.3, "relu", 1.0, False, "lane", 2),
    ("bp_l2_d2_sigmoid", "Backprojection_Loss", 2, 2, 0.3, "sigmoid", 0.0, False, "lane", 1),
    ("bp_l2_d2_uniform", "Backprojection_Loss", 2, 2, 0.3, "square", 0.0, False, "uniform", 2),
    ("bev_l2_d2", "Birds_Eye_View_Loss", 2, 2, 0.3, "square", 0.0, False, "lane", 2),
]


def lsq_case_inputs(name, L, order, maps, B, H=256, W=512):
    seed = zlib.crc32(name.encode()) % 100000
    if maps == "lane":
        o = inputs.make_lane_maps(B, L, H, W, seed=seed)
    else:
        o = inputs.make_uniform_maps(B, L, H, W, seed=seed)
    if "sigmoid" in name or "relu" in name:
        o = (o - 0.3) * 4.0          # exercise negative inputs too
    g = inputs.make_grad_beta(B, L, order, seed=7)
    return o.astype(np.float32), g


def run_lsq_case(case):
    name, variant, L, order, mask_pct, act, reg_ls, chol, maps, B = case
    ns = ri.import_reference(variant)
    H, W = 256, 512
    o_np, g_np = lsq_case_inputs(name, L, order, maps, B)
    out = {"meta": json.dumps(dict(name=name, variant=variant, L=L, order=order, mask_pct=mask_pct, act=act,
                                   reg_ls=reg_ls, cholesky=chol, maps=maps, B=B, H=H, W=W)),
           "input_sha": inputs.sha256_of(o_np, g_np)}
    size = torch.Size([B, L, H, W])
    from math import ceil
    zero_rows = ceil(H * mask_pct)
    idx_row = torch.linspace(0, zero_rows - 1, zero_rows).long()
    if variant == "Backprojection_Loss":
        M, _ = ns.utils.get_homography(H, False)
        M = torch.from_numpy(M).unsqueeze(0).expand([B, 3, 3]).float()
        grid32 = ns.LSQ_layer.ProjectiveGridGenerator(size, M, True)
        ls = ns.LSQ_layer.Weighted_least_squares(size, L, order, True, reg_ls, chol)
    else:
        _, M, _ = ns.LSQ_layer.Init_Projective_transform(L, B, H)
        grid32 = ns.LSQ_layer.ProjectiveGridGenerator(size, M, True)(M)
        ls = ns.LSQ_layer.Weighted_least_squares(size, L, order, True, reg_ls, chol)
    actf = ns.LSQ_layer.activation_layer(act, True)
    out["grid0"] = grid32[0].numpy().copy()       # [HW,2] float32 (1 MB) -- kept only for the first case
    for tag, dt in (("f32", torch.float32), ("f64", torch.float64)):
        o = torch.from_numpy(o_np).to(dt).requires_grad_(True)
        ls.tensor_ones = ls.tensor_ones.to(dt)
        ls.reg_ls = ls.reg_ls.to(dt)
        grid = grid32.to(dt)
        masked = actf(o).index_fill(2, idx_row, 0)
        betas = ls(masked, grid)
        betas = [b for b in betas if b is not None][:L]
        beta = torch.stack([b.squeeze(-1) for b in betas], 1)          # [B,L,d+1]
        g = torch.from_numpy(g_np).to(beta.dtype)
        (beta * g).sum().backward()
        out["beta_" + tag] = beta.detach().double().numpy()
        summarize("grad_" + tag, o.grad, 4096, out)
        out["beta_dtype_" + tag] = str(betas[0].dtype)
    return name, out


# ---------------------------------------------------------------------------
# Whole-path goldens (ERFNet -> LSQ -> backprojection loss, fwd + bwd)
# ---------------------------------------------------------------------------

NET_CASES = [
    # name, nclasses, order, mask_pct, B
    ("net_l2_d2", 2, 2, 0.3, 2),
    ("net_l4_d3", 4, 3, 0.2, 2),
]
# the BASELINE batch size of config 2 (VERDICT r1: all whole-path goldens were B = 2); generated separately
# (`--only-net-b32`, ~2 min of CPU for the fp32 + fp64 reference passes) so the files above stay bit-identical
NET_CASE_B32 = ("net_l2_d2_b32", 2, 2, 0.3, 32)


def tap_modules(m):
    mods = {"encoder.initial_block": m.net.encoder.initial_block}
    for i, l in enumerate(m.net.encoder.layers):
        mods["encoder.layers.%d" % i] = l
    for i, l in enumerate(m.net.decoder.layers):
        mods["decoder.layers.%d" % i] = l
    mods["decoder.output_conv"] = m.net.decoder.output_conv
    return mods


def run_net_case(case):
    name, L, order, mask_pct, B = case
    ns = ri.import_reference("Backprojection_Loss")
    H, W = 256, 512
    args = ri.make_args(ns, ["--nclasses", str(L), "--order", str(order), "--batch_size", str(B),
                             "--mask_percentage", str(mask_pct), "--end_to_end", "True",
                             "--loss_policy", "backproject"])
    torch.manual_seed(0)
    m = ns.LSQ_layer.Net(args)
    P = inputs.make_erfnet_params(3, L, seed=11)
    sd = m.state_dict()
    for k, v in P.items():
        assert tuple(sd[k].shape) == v.shape, (k, sd[k].shape, v.shape)
        sd[k] = torch.from_numpy(v)
    m.load_state_dict(sd)
    for mod in m.modules():
        if hasattr(mod, "dropout"):
            mod.dropout.p = 0            # goldens are dropout-free (SURVEY.md 7.2 #8)
    m.train()
    x_np = inputs.make_images(B, H, W, seed=3)
    xgt_np, valid_np = inputs.make_loss_targets(B, 4, seed=5)
    out = {"meta": json.dumps(dict(name=name, L=L, order=order, mask_pct=mask_pct, B=B, H=H, W=W,
                                   param_seed=11, image_seed=3, target_seed=5)),
           "input_sha": inputs.sha256_of(x_np, xgt_np, valid_np),
           "param_sha": inputs.sha256_of(*[P[k] for k in sorted(P)]),
           "state_dict_keys": json.dumps([(k, list(v.shape), str(v.dtype)) for k, v in m.state_dict().items()])}
    crit = ns.Loss_crit.backprojection_loss(args)
    for tag, dt in (("f32", torch.float32), ("f64", torch.float64)):
        if dt == torch.float64:
            m = m.double()
            m.grid = m.grid.double()
            m.ls_layer.tensor_ones = m.ls_layer.tensor_ones.double()
            m.ls_layer.reg_ls = m.ls_layer.reg_ls.double()
            # reset BN running stats so both passes start from the same buffers
            for mod in m.modules():
                if isinstance(mod, torch.nn.BatchNorm2d):
                    mod.reset_running_stats()
        m.zero_grad()
        taps = {}
        hooks = [mod.register_forward_hook(lambda _m, _i, o, n=n: taps.__setitem__(n, o))
                 for n, mod in tap_modules(m).items()]
        x = torch.from_numpy(x_np).to(dt)
        res = m(x, torch.zeros(B, 4), True)
        for h in hooks:
            h.remove()
        betas = [b for b in res[:4] if b is not None]
        masked, output = res[4], res[5]
        xgt, valid = torch.from_numpy(xgt_np), torch.from_numpy(valid_np)
        total, xcals = 0, []
        for l in range(L):
            ll, xc = crit(betas[l], xgt[:, l], valid[:, l])
            total = total + ll
            xcals.append(xc)
        loss = total / L
        loss.backward()
        out["loss_" + tag] = np.array(float(loss))
        out["beta_" + tag] = torch.stack([b.squeeze(-1) for b in betas], 1).detach().double().numpy()
        out["xcal_" + tag] = torch.stack(xcals, 1).detach().numpy()
        for n, t in taps.items():
            summarize("act_%s/%s" % (tag, n), t, N_ACT_SAMPLES, out)
        summarize("act_%s/masked" % tag, masked, N_ACT_SAMPLES, out)
        for n, p in m.named_parameters():
            if p.grad is not None:
                summarize("grad_%s/%s" % (tag, n), p.grad, N_GRAD_SAMPLES, out)
        for n, b in m.named_buffers():
            if n.endswith("running_mean") or n.endswith("running_var"):
                out["buf_%s/%s" % (tag, n)] = b.detach().double().numpy()
    out["params_without_grad"] = json.dumps([n for n, p in m.named_parameters() if p.grad is None])
    return name, out


def run_homography():
    ns = ri.import_reference("Backprojection_Loss")
    out = {}
    for r in (256, 320):
        M, Mi = ns.utils.get_homography(r, False)
        out["M_%d" % r], out["Minv_%d" % r] = M, Mi
    ns = ri.import_reference("Birds_Eye_View_Loss")
    _, M, Mi = ns.LSQ_layer.Init_Projective_transform(2, 1, 256)
    out["M_bev_f32"], out["Minv_bev_f32"] = M[0].numpy(), Mi[0].numpy()
    return "homography", out


# ---------------------------------------------------------------------------
# Area_Loss goldens (A12).  The reference's forward ends in ``torch.masked_select(loss_fit, mask.byte())``
# (BP/Loss_crit.py:140-141 == BEV/Loss_crit.py:131-132), which torch >= 2 rejects (uint8 masks were removed).  The
# reference targets torch 1.1 where a byte mask IS a boolean mask, so the run below shims exactly that dispatch
# (masked_select accepts uint8 by viewing it as bool) and executes every other line of the reference unmodified.
# ---------------------------------------------------------------------------
AREA_CASES = [(2, "none"), (2, "linear"), (2, "quadratic"), (1, "none")]


def run_area_loss():
    out = {}
    orig = torch.masked_select

    def masked_select_torch11(x, mask):
        return orig(x, mask.bool() if mask.dtype == torch.uint8 else mask)

    rng = np.random.default_rng(1234)
    B = 6
    params = rng.normal(size=(B, 3, 1)) * np.array([1e-3, 0.2, 0.5]).reshape(1, 3, 1)
    gt = rng.normal(size=(B, 3)) * np.array([1e-3, 0.2, 0.5])
    gt[2] = 0.0                    # absent lane: all-zero ground truth -> excluded from the mean
    gt[4, 1] = 0.0                 # one zero entry also excludes the lane (prod(gt != 0))
    out["params"], out["gt"] = params, gt
    torch.masked_select = masked_select_torch11
    try:
        for variant in ("Backprojection_Loss", "Birds_Eye_View_Loss"):
            ns = ri.import_reference(variant)
            for order, wf in AREA_CASES:
                for tag, dt in (("f32", torch.float32), ("f64", torch.float64)):
                    p = torch.from_numpy(params).to(dt).requires_grad_(True)
                    loss = ns.Loss_crit.Area_Loss(order, wf)(p, torch.from_numpy(gt).to(dt))
                    loss.backward()
                    key = "%s/o%d_%s_%s" % (variant[:2], order, wf, tag)
                    out[key + "/loss"] = np.array(float(loss))
                    out[key + "/grad"] = p.grad.double().numpy()
            # every lane absent -> the reference returns the python int 0
            z = ns.Loss_crit.Area_Loss(2, "none")(torch.from_numpy(params).float(), torch.zeros(B, 3))
            out["%s/all_absent" % variant[:2]] = np.array(float(z))
    finally:
        torch.masked_select = orig
        ri.purge()
    return "area_loss", out


def run_clas_heads():
    """Classification heads (`--clas 1`, BP/Networks/LSQ_layer.py:157-207): the reference's own class on a seeded encoder
    map, fp32 and fp64, forward + backward of sum(out * g)."""
    ns = ri.import_reference("Backprojection_Loss")
    B = 2
    x_np = inputs.make_encoder_map(B, seed=21)
    out = {"meta": json.dumps(dict(B=B, map_seed=21, param_seeds={"line": 31, "horizon": 32}, g_seeds={"line": 41, "horizon": 42}))}
    for kind, pseed, gseed in (("line", 31, 41), ("horizon", 32, 42)):
        P = inputs.make_head_params(kind, pseed)
        for tag, dt in (("f32", torch.float32), ("f64", torch.float64)):
            torch.manual_seed(0)
            m = ns.LSQ_layer.Classification(kind, size=(32, 64), channels_in=128, resize=256)
            sd = m.state_dict()
            for k, v in P.items():
                assert tuple(sd[k].shape) == v.shape, (k, sd[k].shape, v.shape)
                sd[k] = torch.from_numpy(v)
            m.load_state_dict(sd)
            m = m.to(dt).train()
            x = torch.from_numpy(x_np).to(dt).requires_grad_(True)
            y = m(x)
            g = torch.from_numpy(np.random.default_rng(gseed).standard_normal(tuple(y.shape))).to(dt)
            (y * g).sum().backward()
            out["%s/out_%s" % (kind, tag)] = y.detach().double().numpy()
            summarize("%s/dx_%s" % (kind, tag), x.grad, 4096, out)
            for n, p in m.named_parameters():
                summarize("%s/grad_%s/%s" % (kind, tag, n), p.grad, 1024, out)
            for n, b in m.named_buffers():
                if n.endswith("running_mean") or n.endswith("running_var"):
                    out["%s/buf_%s/%s" % (kind, tag, n)] = b.detach().double().numpy()
        out["%s/g" % kind] = np.random.default_rng(gseed).standard_normal(tuple(y.shape))
    return "clas_heads", out


def main():
    if "--only-net-b32" in sys.argv:
        os.makedirs(GOLDEN_DIR, exist_ok=True)
        torch.set_num_threads(max(1, os.cpu_count() or 1))
        name, out = run_net_case(NET_CASE_B32)
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        np.savez_compressed(path, **out)
        print("wrote", path, os.path.getsize(path), "bytes", "loss", out["loss_f32"], out["loss_f64"])
        return 0
    if "--only-clas" in sys.argv:
        os.makedirs(GOLDEN_DIR, exist_ok=True)
        name, out = run_clas_heads()
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        np.savez_compressed(path, **out)
        print("wrote", path, os.path.getsize(path), "bytes")
        return 0
    if "--only-area" in sys.argv:      # add the A12 fixture without touching the (bit-identical) existing ones
        os.makedirs(GOLDEN_DIR, exist_ok=True)
        name, out = run_area_loss()
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        np.savez_compressed(path, **out)
        print("wrote", path, os.path.getsize(path), "bytes")
        return 0
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    jobs = [run_homography(), run_area_loss(), run_clas_heads()]
    for i, c in enumerate(LSQ_CASES):
        name, out = run_lsq_case(c)
        if c[0] not in ("bp_l2_d2", "bev_l2_d2"):
            out.pop("grid0")            # one BP grid + one BEV grid are enough (1 MB each)
        jobs.append(("lsq_" + name, out))
        print("lsq", name, "beta32-beta64 max", np.abs(out["beta_f32"] - out["beta_f64"]).max(), flush=True)
    for c in NET_CASES:
        name, out = run_net_case(c)
        jobs.append((name, out))
        print("net", name, "loss", out["loss_f32"], out["loss_f64"], flush=True)
    for name, out in jobs:
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        np.savez_compressed(path, **out)
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    sys.exit(main())
