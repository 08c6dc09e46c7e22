"""engine.GraphedTrainStep -- the whole training step as one CUDA-graph replay, what bench.py times -- against the
reference's goldens and against eager steps of the same model:

  * one replay at the benchmark workload passes the whole-path golden gates of oracle/golden_check.py;
  * a plain user training loop (optimizer, set_to_none zero_grad, new batches through load() and the double-buffered
    prefetch()/swap_in(), Dropout2d on) stays bit-identical to the same loop run eagerly;
  * eager forwards and steps on the same model between replays (another conv mode, eval, another batch size) do not free
    anything the graph reads, and the next replay still equals an eager step.

Inputs are 256x512 so the kernels dispatch as in the benchmark (tcgen05 vs CUDA-core fallback, split counts).
"""
import weakref

import numpy as np
import pytest
import torch

from oracle import golden_check, inputs

pytestmark = pytest.mark.gpu
TOL = 1e-4


@pytest.fixture(autouse=True)
def _no_active_packs():
    yield
    from lanedetection_end2end_b200 import ops_net
    ops_net.ACTIVE_PACKS = None


def _model(L, B, seed=11, dropout=True):
    model, args = golden_check.build_net(L, 2, 0.3, B)
    sd = model.state_dict()
    for k, v in inputs.make_erfnet_params(3, L, seed=seed).items():
        sd[k] = torch.from_numpy(v)
    model.load_state_dict(sd)
    model = model.cuda().train()
    model.defer_status_check = True
    if not dropout:
        for m in model.modules():
            if hasattr(m, "dropout"):
                m.dropout.p = 0
    return model, args


def _batch(B, seed):
    """(x, xgt, valid) on the host."""
    xgt, valid = inputs.make_loss_targets(B, 4, seed=seed)
    return torch.from_numpy(inputs.make_images(B, 256, 512, seed=seed)), torch.from_numpy(xgt), torch.from_numpy(valid)


def _eager_step(model, crit, L, x, xgt, valid):
    """The plain eager step with the loss routine GraphedTrainStep uses."""
    from lanedetection_end2end_b200 import engine
    from lanedetection_end2end_b200.Loss_crit import fused_backprojection_loss
    out = model(x, torch.zeros(x.shape[0], 4), True)
    if engine.FUSED_LOSS:
        loss, _ = fused_backprojection_loss(crit, out[:L], xgt, valid)
    else:
        loss, _ = crit.forward_lanes(out[:L], xgt, valid)
    loss.backward()
    return loss.detach()


def _state(model):
    return {n: t.detach().clone() for n, t in list(model.named_parameters()) + list(model.named_buffers())}


def _assert_same_step(mg, me, what):
    """Every gradient, parameter and buffer of the graphed model `mg` equals the eager model's bit for bit."""
    for (n, pg), pe in zip(mg.named_parameters(), me.parameters()):
        if pe.grad is None:
            assert pg.grad is None, (what, "grad", n)
        else:
            assert pg.grad is not None, (what, "grad is None", n)
            assert torch.equal(pg.grad, pe.grad), (what, "grad", n)
        assert torch.equal(pg, pe), (what, "param", n)
    for (n, bg), be in zip(mg.named_buffers(), me.buffers()):
        assert torch.equal(bg, be), (what, "buffer", n)


def _drop_blocks(model):
    from lanedetection_end2end_b200.Networks import ERFNet
    return [m for m in model.modules() if isinstance(m, ERFNet.non_bottleneck_1d) and m.dropout.p > 0]


# ------------------------------------------------------------------------------------------------------------------
# A. one replay vs the reference's goldens
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["tf32x3", "fp32"])
@pytest.mark.parametrize("name", ["net_l2_d2_b32", "net_l4_d3"])       # _b32: batch 32, 2 lanes, order 2 (bench config 2)
def test_graph_replay_matches_reference_golden(name, mode):
    """Construction + one replay is one training step of the reference: the gates of golden_check.run_full_path on the
    replay's activations, beta, loss, every parameter gradient and the BatchNorm running statistics after one step."""
    from lanedetection_end2end_b200 import ops_net
    from lanedetection_end2end_b200.engine import GraphedTrainStep
    from lanedetection_end2end_b200.Loss_crit import backprojection_loss
    ops_net.set_conv_mode(mode)
    case = golden_check.FullPathCase(name)
    # the last call of each hook is the capture: the stored tensors are graph-static and hold each replay's values
    taps, hooks = case.hook_taps()
    gstep = GraphedTrainStep(case.model, backprojection_loss(case.args), case.L, case.x, case.xgt, case.valid)
    for h in hooks:
        h.remove()
    loss = gstep()
    torch.cuda.synchronize()
    assert int(gstep.status.item()) == 0
    betas = [b for b in gstep.out[:4] if b is not None]
    rep = golden_check.compare_full_path(case, taps, betas, loss, tol=TOL, enforce=True)
    print(rep)
    bns = [(n, m) for n, m in case.model.named_modules() if isinstance(m, torch.nn.BatchNorm2d)]
    assert bns
    for n, m in bns:
        assert int(m.num_batches_tracked) == 1, n


# ------------------------------------------------------------------------------------------------------------------
# B. a training loop: graph vs eager, bit for bit
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["tf32x3", "tf32", "fp32"])
def test_training_loop_graph_matches_eager_bitwise(mode, monkeypatch):
    """Two identical models, SGD with momentum and weight decay, four steps on distinct batches, the plain loop
    ``opt.zero_grad(); step; opt.step()`` on both.  Batches 1-2 reach the graph through load(), 3-4 from pinned host
    memory in bench.py's order (prefetch once, then swap_in, prefetch next, replay).  Dropout2d stays on: the masks of
    each replay are recorded and replayed into the eager model.  Exact equality is expected: the kernels are
    deterministic and the only device atomics are integer tickets."""
    from lanedetection_end2end_b200 import ops_net
    from lanedetection_end2end_b200.engine import GraphedTrainStep
    from lanedetection_end2end_b200.Loss_crit import backprojection_loss
    from lanedetection_end2end_b200.Networks import ERFNet
    ops_net.set_conv_mode(mode)
    L, B, steps = 2, 4, 4
    mg, args = _model(L, B)
    me, _ = _model(L, B)

    # record every block's Dropout2d mask of each replay into buffers the test owns (a copy_ captured with the step)
    recorded = []
    draw = ERFNet.fused_dropout_masks

    def recording_draw(blocks, batch, device):
        masks = draw(blocks, batch, device)
        if not recorded:
            recorded.extend(torch.empty_like(m) for m in masks)
        for r, m in zip(recorded, masks):
            r.copy_(m)
        return masks

    monkeypatch.setattr(ERFNet, "fused_dropout_masks", recording_draw)

    batches = [_batch(B, seed=200 + i) for i in range(steps + 1)]       # the last one is only prefetched
    pinned = [tuple(t.pin_memory() for t in b) for b in batches]
    before = _state(mg)
    gstep = GraphedTrainStep(mg, backprojection_loss(args), L, *(t.cuda() for t in batches[0]))
    torch.cuda.synchronize()
    after = _state(mg)
    for n in before:        # construction changes nothing but the contents of .grad
        assert torch.equal(before[n], after[n]), ("changed by construction", n)

    drops_g, drops_e = _drop_blocks(mg), _drop_blocks(me)
    assert len(recorded) == len(drops_g) == len(drops_e) > 0
    crit_e = backprojection_loss(args)
    opt_g = torch.optim.SGD(mg.parameters(), lr=0.0, momentum=0.9, weight_decay=1e-4)
    opt_e = torch.optim.SGD(me.parameters(), lr=0.0, momentum=0.9, weight_decay=1e-4)
    masks_per_step = []
    for i in range(steps):
        opt_g.zero_grad()
        if i < 2:
            gstep.load(*(t.cuda() for t in batches[i]))
        else:
            if i == 2:
                gstep.prefetch(*pinned[2])
            gstep.swap_in()
            gstep.prefetch(*pinned[i + 1])
        loss_g = gstep()
        masks = [m.clone() for m in recorded]
        masks_per_step.append(masks)

        for blk, m in zip(drops_e, masks):
            blk.drop_mask_override = m
        opt_e.zero_grad()
        loss_e = _eager_step(me, crit_e, L, *(t.cuda() for t in batches[i]))
        torch.cuda.synchronize()
        assert np.isfinite(float(loss_e)), (i, float(loss_e))
        assert torch.equal(loss_g, loss_e), (i, float(loss_g), float(loss_e))
        for (n, pg), pe in zip(mg.named_parameters(), me.parameters()):
            # the optimizer reads p.grad: it must be the gradient the replay wrote
            assert (pg.grad is None) == (pe.grad is None), ("step %d" % i, n, pg.grad is None)
        if i == 0:      # a step size that moves the parameters visibly and keeps them in range, the same on both
            lr = 1e-3 / max(float(p.grad.abs().max()) for p in me.parameters() if p.grad is not None)
            for opt in (opt_g, opt_e):
                for group in opt.param_groups:
                    group["lr"] = lr
        opt_g.step()
        opt_e.step()
        _assert_same_step(mg, me, "step %d" % i)
        assert torch.equal(mg.lsq_status, me.lsq_status), i
        if i == 0:
            assert any(not torch.equal(p, before[n]) for n, p in mg.named_parameters()), "SGD did not move"

    # the recorded masks are real Dropout2d draws: fresh per replay, values 0 or 1/(1-p), keep rate ~ 1-p
    for i in range(1, steps):
        assert not torch.equal(torch.cat([m.flatten() for m in masks_per_step[i]]),
                               torch.cat([m.flatten() for m in masks_per_step[i - 1]])), i
    kept, total = {}, {}
    for masks in masks_per_step:
        for blk, m in zip(drops_g, masks):
            p = float(blk.dropout.p)
            scale = torch.tensor(1.0 / (1.0 - p), dtype=torch.float32, device=m.device)
            assert bool(((m == 0) | (m == scale)).all()), p
            kept[p] = kept.get(p, 0) + int((m != 0).sum())
            total[p] = total.get(p, 0) + m.numel()
    for p in kept:
        mean, sd = total[p] * (1 - p), (total[p] * p * (1 - p)) ** 0.5
        assert abs(kept[p] - mean) <= 5 * sd, (p, kept[p], mean, sd)


# ------------------------------------------------------------------------------------------------------------------
# C. eager work on the same model between replays
# ------------------------------------------------------------------------------------------------------------------
def test_eager_work_between_replays_keeps_captured_operands_alive():
    """After capture in tf32x3: two eager fp32 training steps (new operand kinds -> the weight-pack job table is
    rebuilt), an eval forward and a training forward at another batch size.  Everything the graph reads through a
    host-side cache must still be alive -- checked on the host, before any replay -- and the next replay must equal an
    eager tf32x3 step from the same parameters and buffers."""
    from lanedetection_end2end_b200 import ops_lsq, ops_net
    from lanedetection_end2end_b200.engine import GraphedTrainStep
    from lanedetection_end2end_b200.Loss_crit import backprojection_loss
    ops_net.set_conv_mode("tf32x3")
    L, B = 2, 4
    model, args = _model(L, B, dropout=False)
    crit = backprojection_loss(args)
    gstep = GraphedTrainStep(model, crit, L, *(t.cuda() for t in _batch(B, seed=300)))
    packs = model.net.__dict__["_weight_packs"]
    refs = [weakref.ref(packs.jobs)]
    refs += [weakref.ref(t) for e in packs.job_entries for t in (e[1], e[2])]
    refs += [weakref.ref(t) for tab in ops_lsq._TABLE_CACHE.values() for t in (tab.xtab, tab.ytab, tab.yrow)
             if t is not None]
    refs += [weakref.ref(t) for t in ops_lsq._WS_CACHE.values()]
    n_jobs = len(packs.job_entries)

    ops_net.set_conv_mode("fp32")
    for s in (301, 302):
        model.zero_grad()
        _eager_step(model, crit, L, *(t.cuda() for t in _batch(B, seed=s)))
    assert packs.jobs is not refs[0]() and len(packs.job_entries) > n_jobs, "the job table was not rebuilt"
    model.eval()
    with torch.no_grad():
        model(_batch(B, seed=303)[0].cuda(), torch.zeros(B, 4), True)
    model.train()
    model(_batch(2, seed=304)[0].cuda(), torch.zeros(2, 4), True)
    ops_net.set_conv_mode("tf32x3")
    torch.cuda.synchronize()
    dead = [i for i, r in enumerate(refs) if r() is None]
    assert not dead, "tensors the captured step reads were freed (job table = 0): %s" % dead

    ref_model, _ = _model(L, B, dropout=False)
    ref_model.load_state_dict(model.state_dict())
    batch = [t.cuda() for t in _batch(B, seed=305)]
    gstep.load(*batch)
    model.zero_grad()
    loss_g = gstep()
    loss_e = _eager_step(ref_model, backprojection_loss(args), L, *batch)
    torch.cuda.synchronize()
    assert torch.equal(loss_g, loss_e), (float(loss_g), float(loss_e))
    _assert_same_step(model, ref_model, "replay after eager work")
