"""Whole-step CUDA graph for the training hot path.

One step = zero grads -> ``Net.forward`` -> backprojection loss over the lanes -> backward
(-> flat gradient all-reduce when data-parallel): ~600 kernel launches of a few microseconds
each (SURVEY.md 7.2 #6).  Eagerly, the Python/ctypes cost per launch bounds the step once the kernels
are fast; captured once into a ``torch.cuda.CUDAGraph`` the step is a single replay.  Inputs live
in static device buffers (``copy_`` new batches in, asynchronously from pinned host memory); the loss and
the LSQ status word are static outputs the caller reads when it wants to (no sync inside the step).

The graph only contains our C-ABI kernels, a handful of tiny float64 torch ops of the loss, torch's
graph-safe Philox draws for the Dropout2d masks, and (optionally) the NCCL all-reduce.

Contract of ``GraphedTrainStep``:
  * Construction runs a few eager warm-up steps and the capture, then puts every module buffer (BatchNorm running
    statistics, ``num_batches_tracked``) back to its value before construction.  What it leaves changed is the
    contents of the parameters' ``.grad`` tensors and the CUDA RNG offset.
  * Supported loops: the plain ``opt.zero_grad(); step(); opt.step()`` (``set_to_none`` or not: every call re-attaches
    the captured gradient tensors as ``.grad``), and ``load()`` / ``prefetch()`` + ``swap_in()`` for new batches.
    Parameters may be updated in place (any optimizer); the captured weight packing reads their current values.
  * Eager forwards and steps on the same model between replays are allowed: every device tensor the capture reads
    through a host-side cache (weight-pack job table and packed operands, LSQ grid tables and workspace) is held by
    the step object, so a cache that later rebuilds or evicts it cannot free memory the graph still uses.
  * A capture is invalidated by replacing parameter or buffer objects (``load_state_dict`` copies in place and is
    fine; assigning a new ``nn.Parameter`` is not) and by changing the loss homography (its constants are baked
    into the loss launch).  The graph also keeps the batch shape, convolution mode and Dropout2d ``p`` values it was
    captured with.  Build a new step after any of these changes.
"""
import os

import torch

# lf_backproj_loss: one launch for the loss of all lanes + its gradient instead of ~40 tiny float64 torch launches.
# GPU-validated (tests/test_net_gpu.py::test_fused_backprojection_loss_kernel, profiles/r02): on by default;
# LANEFIT_FUSED_LOSS=0 falls back to the torch ops of Loss_crit.backprojection_loss.forward_lanes.
FUSED_LOSS = os.environ.get("LANEFIT_FUSED_LOSS", "1") != "0"


def _cached_operands(model):
    """Device tensors a captured step reads through host-side caches that may later drop or replace them.

    * ``WeightPackCache`` (one per ERFNet): ``refresh()`` builds a new job table once an eager forward registers another
      operand kind (another conv mode, another dispatch), and drops entries whose parameter went away.
    * ``ops_lsq._TABLE_CACHE`` clears itself past 16 grids; ``ops_lsq._WS_CACHE`` replaces a workspace that is too small.
    Safe without pinning: ``ERFNet._DROP_PLANS``, ``ops_net._TCG_WGRAD_IDX`` and ``ops_net._SUPER_IDX`` never evict; the
    loss ticket lives on the criterion (held by the step) and the loss constants are passed by value into the launch."""
    from . import ops_lsq
    refs = []
    for m in model.modules():
        packs = m.__dict__.get("_weight_packs")
        if packs is not None and packs.jobs is not None:
            refs.append((packs.jobs, list(packs.job_entries)))
    refs.append(list(ops_lsq._TABLE_CACHE.values()))
    refs.append(list(ops_lsq._WS_CACHE.values()))
    return refs


class GraphedTrainStep:
    """One training step (zero grads -> forward -> loss -> backward [-> all-reduce]) captured into a CUDA graph.

    Calling the object replays it and returns the static float64 loss; ``out`` holds the forward's outputs of the replay
    (detached 9-tuple as ``Net.forward`` returns it: beta0..3, masked, output, ...), ``status`` the LSQ status word.

    Construction leaves the model's parameters and buffers as they were (only the ``.grad`` contents change).  Before
    every replay the captured gradient tensors are re-attached as ``p.grad`` wherever ``.grad`` was set to None
    (``optimizer.zero_grad()`` defaults to ``set_to_none=True``) or replaced, so the plain
    ``opt.zero_grad(); step(); opt.step()`` loop trains; with a data-parallel reducer these are the views of its flat
    buffer that ``attach()`` installed.  See the module docstring for what invalidates a capture."""

    def __init__(self, model, criterion, nclasses, example_x, example_xgt, example_valid, reducer=None, warmup=3,
                 capture_error_mode="global", extra_loss=None, global_valid=False):
        self.model = model
        self.global_valid = global_valid  # batch-global sum(valid) normaliser across ranks (ddp.lane_valid_scale)
        self.extra_loss = extra_loss      # callable(forward 9-tuple) -> scalar added to the loss (e.g. the --clas head losses)
        self.crit = criterion
        self.L = nclasses
        self.reducer = reducer
        dev = example_x.device
        self.x = example_x.clone()
        self.xgt = example_xgt.clone()
        self.valid = example_valid.clone()
        self.gt_line = torch.zeros(example_x.shape[0], 4)
        model.defer_status_check = True
        self.params = [p for p in model.parameters() if p.requires_grad]
        # the warm-up steps update the BatchNorm running statistics and step counters: restored after the capture
        buffers = list(model.buffers())
        saved = [b.clone() for b in buffers]

        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):
                self._eager_step(first=True)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        # gradients now exist as persistent tensors; the captured step zeroes and re-accumulates them
        if reducer is not None and hasattr(reducer, "attach"):
            reducer.attach()          # gradients become views of the flat all-reduce buffer: no pack / unpack copies
        self._grad_slots = [(p, p.grad) for p in self.params if p.grad is not None]
        self.grads = [g for _, g in self._grad_slots]
        self.graph = torch.cuda.CUDAGraph()
        # with NCCL in the graph use capture_error_mode="thread_local": the process group's watchdog thread polls CUDA
        # events, which the default "global" mode treats as a capture violation
        with torch.cuda.graph(self.graph, capture_error_mode=capture_error_mode):
            self.loss, out = self._eager_step(first=False)
        self.out = tuple(t.detach() if torch.is_tensor(t) else t for t in out)
        self.status = model.lsq_status
        self._cache_refs = _cached_operands(model)
        with torch.no_grad():
            for b, v in zip(buffers, saved):     # into the same storage the graph updates
                b.copy_(v)

    def _eager_step(self, first):
        if first:
            self.model.zero_grad(set_to_none=True)
        else:
            torch._foreach_zero_(self.grads)
        out = self.model(self.x, self.gt_line, True)
        scale = None
        if self.global_valid:
            from .ddp import lane_valid_scale
            scale = lane_valid_scale(self.valid, self.L)
        if FUSED_LOSS and hasattr(self.crit, "_fused_host_constants"):
            from .Loss_crit import fused_backprojection_loss
            loss, _ = fused_backprojection_loss(self.crit, out[:self.L], self.xgt, self.valid, lane_scale=scale)
        elif hasattr(self.crit, "forward_lanes"):
            loss, _ = self.crit.forward_lanes(out[:self.L], self.xgt, self.valid, lane_scale=scale)    # all lanes in one pass
        else:
            loss = 0
            for l in range(self.L):
                ll, _ = self.crit(out[l], self.xgt[:, l], self.valid[:, l])
                loss = loss + ll
            loss = loss / self.L
        if self.extra_loss is not None:
            loss = loss + self.extra_loss(out)
        loss.backward()
        if self.reducer is not None:
            self.reducer()
        return loss.detach(), out

    def load(self, x, xgt, valid):
        """Stage a new batch (device or pinned-host tensors) into the static input buffers."""
        self.x.copy_(x, non_blocking=True)
        self.xgt.copy_(xgt, non_blocking=True)
        self.valid.copy_(valid, non_blocking=True)

    # -- double-buffered input pipeline: the H2D copy of batch i+1 runs on a copy stream while step i computes
    def prefetch(self, x, xgt, valid):
        """Start copying the NEXT batch (pinned host tensors) into the staging buffers on the copy stream."""
        if not hasattr(self, "_copy_stream"):
            dev = self.x.device
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._stage = [torch.empty_like(self.x), torch.empty_like(self.xgt), torch.empty_like(self.valid)]
            self._ready = torch.cuda.Event()
            self._consumed = torch.cuda.Event()
            self._consumed.record(torch.cuda.current_stream(dev))
        self._copy_stream.wait_event(self._consumed)     # staging buffers were drained by swap_in()
        with torch.cuda.stream(self._copy_stream):
            for dst, src in zip(self._stage, (x, xgt, valid)):
                dst.copy_(src, non_blocking=True)
            self._ready.record(self._copy_stream)

    def swap_in(self):
        """Move the prefetched batch into the graph's static inputs (device-to-device, on the compute stream)."""
        cur = torch.cuda.current_stream(self.x.device)
        cur.wait_event(self._ready)
        self.x.copy_(self._stage[0], non_blocking=True)
        self.xgt.copy_(self._stage[1], non_blocking=True)
        self.valid.copy_(self._stage[2], non_blocking=True)
        self._consumed.record(cur)

    def __call__(self):
        for p, g in self._grad_slots:     # zero_grad(set_to_none=True) or a new .grad: hand the captured tensor back
            if p.grad is not g:
                p.grad = g
        self.graph.replay()
        return self.loss


class GraphedInference:
    """Eval-mode forward (BatchNorm-folded launches, ops_eval.py) captured once into a CUDA graph and replayed per batch:
    what the reference's validate() / test_model() loops do per batch (BP/main.py:452, BP/test.py:53-55), without the ~25 us
    of ctypes / Python per launch.  ``infer(x)`` copies the batch into the static input and replays; the returned 9-tuple
    (beta0..3, masked, output, line, horizon, output_seg) aliases static buffers that the next call overwrites.
    The BatchNorm-folded weights are cached at capture time: after an optimizer step they are stale, so capture again.
    ``model.lsq_status`` (device int32, OR-ed) reports singular systems; `check()` reads it (one sync)."""

    def __init__(self, model, example_x, warmup=2):
        self.model = model.eval()
        model.defer_status_check = True
        self.x = example_x.clone()
        self.gt_line = torch.zeros(example_x.shape[0], 4)
        dev = example_x.device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(max(1, warmup)):             # builds and caches the folded operands outside the capture
                model(self.x, self.gt_line, True)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.no_grad(), torch.cuda.graph(self.graph):
            self.out = model(self.x, self.gt_line, True)

    def infer(self, x):
        self.x.copy_(x, non_blocking=True)
        self.graph.replay()
        return self.out

    def check(self):
        st = int(self.model.lsq_status.item())
        if st:
            self.model.lsq_status.zero_()
            raise RuntimeError("status word %d (1 singular / 2 non-finite / 4 not positive definite normal matrix)" % st)
