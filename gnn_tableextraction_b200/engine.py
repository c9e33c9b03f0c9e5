"""Train / inference step engine for ``GcnSAGE`` on the sm_100a kernels.

Restates the train-step envelope of the reference
(/root/reference/src/models/model_train.py:297,320-332):

    batch_graph = dgl.batch(train_batch).to(device)      -> H2D of one pinned host batch
    logits = model(batch_graph)                           -> layer kernels (layers.py)
    loss = CrossEntropyLoss(weight)(logits, labels.long())-> gte_cross_entropy_fwd/bwd
    optimizer.zero_grad(); loss.backward(); optimizer.step()
                                                          -> explicit backward kernels writing
                                                             one flat gradient buffer, one
                                                             (optional) all-reduce, fused Adam

without autograd bookkeeping, without the per-step ``.item()`` sync, and replayed
from a CUDA graph -- for fixed-shape batches, or for every batch up to a
``BatchCapacity`` (padded on the device inside the graph).  Data parallel by graph
(pages are independent): every rank runs the same step on its own pages; the
loss statistics ride in the tail of the flat gradient buffer, so ONE SUM
all-reduce per step carries gradients and statistics; Adam divides by the
GLOBAL label-weight sum, which reproduces the single-GPU result (not a mean
of per-rank means).
"""
from __future__ import annotations

import gc
import os
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import layers as L
from . import ops
from ._lib import GteError
from .graph import PageGraphBatch, page_table
from .nn import GcnSAGE, _is_relu
from .pool import PagePool


def _dropout_p(d) -> float:
    """dropout attribute of the reference modules: nn.Dropout or the float 0. (models.py:30-33)"""
    return float(d.p) if isinstance(d, nn.Dropout) else float(d or 0.0)


@dataclass(frozen=True)
class BatchCapacity:
    """The largest page batch a capacity-captured step accepts: total nodes, total edges, page count, and the largest
    page in nodes and in edges.  The reference batches shuffled real pages (model_train.py:283-297) and streams pages
    for prediction (model_predict.py:130-154), so the totals change from batch to batch; a step captured for a
    capacity replays one CUDA graph for every batch that fits, padded on the device to the shape ``shape``."""

    nodes: int
    edges: int
    pages: int
    page_nodes: int
    page_edges: int

    def __post_init__(self):
        for k in ("nodes", "edges", "pages", "page_nodes", "page_edges"):
            v = getattr(self, k)
            if not isinstance(v, (int, np.integer)) or isinstance(v, bool):
                raise GteError(f"BatchCapacity: {k} must be an int, got {v!r}")
            object.__setattr__(self, k, int(v))
        if self.nodes < 1 or self.pages < 1 or self.edges < 0 or self.page_edges < 1:
            raise GteError(f"BatchCapacity: need nodes >= 1, pages >= 1, edges >= 0, page_edges >= 1 (got {self})")
        if self.page_nodes < 2:  # every padding page needs room for more than one node (see shape)
            raise GteError(f"BatchCapacity: page_nodes={self.page_nodes} < 2")
        if self.page_nodes > PAGE_NODES_MAX:
            raise GteError(f"BatchCapacity: page_nodes={self.page_nodes} > {PAGE_NODES_MAX}, the largest page the page "
                           "kernels stage")
        n_cap, e_cap, _ = self.shape
        if e_cap >= 2 ** 31 or n_cap >= 2 ** 31:
            raise GteError(f"BatchCapacity: {n_cap} nodes / {e_cap} edges after padding exceed int32 ids")

    @property
    def shape(self) -> Tuple[int, int, int]:
        """(N_cap, E_cap, P_cap) of the captured batch.  K = max(ceil(nodes / (page_nodes - 1)), ceil(edges /
        page_edges)) padding slots: any fitting batch leaves at least K free page slots and K padding nodes, and
        K slots carry all padding nodes and edges without exceeding the page caps."""
        k = max(-(-self.nodes // (self.page_nodes - 1)), -(-self.edges // self.page_edges))
        return self.nodes + k, self.edges, self.pages + k

    def check(self, batch_num_nodes: Sequence[int], batch_num_edges: Sequence[int]) -> None:
        """Raise a GteError naming the limit a batch with these page sizes breaks."""
        bn, be = list(batch_num_nodes), list(batch_num_edges)
        if len(bn) != len(be):
            raise GteError(f"batch: {len(bn)} page node counts but {len(be)} page edge counts")
        if not bn:
            raise GteError("batch: no pages")
        if min(bn) < 0 or min(be) < 0:
            raise GteError("batch: negative page size")
        pre = "batch does not fit the captured capacity:"
        if len(bn) > self.pages:
            raise GteError(f"{pre} {len(bn)} pages > pages={self.pages}")
        if sum(bn) > self.nodes:
            raise GteError(f"{pre} {sum(bn)} nodes > nodes={self.nodes}")
        if sum(be) > self.edges:
            raise GteError(f"{pre} {sum(be)} edges > edges={self.edges}")
        if max(bn) > self.page_nodes:
            raise GteError(f"{pre} a page of {max(bn)} nodes > page_nodes={self.page_nodes}")
        if max(be) > self.page_edges:
            raise GteError(f"{pre} a page of {max(be)} edges > page_edges={self.page_edges}")

    def fits(self, batch_num_nodes: Sequence[int], batch_num_edges: Sequence[int]) -> bool:
        try:
            self.check(batch_num_nodes, batch_num_edges)
        except GteError:
            return False
        return True


PAGE_NODES_MAX = 1600  # graph.page_table: larger pages get no page table (generic kernels)


def padded_page_table(capacity: BatchCapacity, batch_num_nodes: Sequence[int], batch_num_edges: Sequence[int]):
    """Page table (node offsets, edge offsets: int32 [P_cap + 1] each) of a batch padded to ``capacity.shape``: the
    real pages as given, then s = min(P_cap - P, N_cap - n) padding pages sharing the N_cap - n padding nodes and the
    E_cap - e padding edges evenly (each gets at least one node and at most page_nodes / page_edges), then empty
    pages.  gte_pad_batch makes every padding edge a weight-0 self-loop on a node of its own padding page."""
    capacity.check(batch_num_nodes, batch_num_edges)
    n_cap, e_cap, p_cap = capacity.shape
    bn = np.asarray(list(batch_num_nodes), dtype=np.int64)
    be = np.asarray(list(batch_num_edges), dtype=np.int64)
    p, n, e = len(bn), int(bn.sum()), int(be.sum())
    s = min(p_cap - p, n_cap - n)  # >= K >= 1
    j = np.arange(1, s + 1, dtype=np.int64)
    po = np.full(p_cap + 1, n_cap, dtype=np.int64)
    eo = np.full(p_cap + 1, e_cap, dtype=np.int64)
    po[0] = eo[0] = 0
    np.cumsum(bn, out=po[1:p + 1])
    np.cumsum(be, out=eo[1:p + 1])
    po[p + 1:p + 1 + s] = n + j * (n_cap - n) // s
    eo[p + 1:p + 1 + s] = e + j * (e_cap - e) // s
    return po.astype(np.int32), eo.astype(np.int32)


# ------------------------------------------------------------------ resident passes: epochs planned over a PagePool --
@dataclass(frozen=True)
class PlannedBatch:
    """One slice of an epoch plan (``plan_epoch``): its page ids, whether it fits the captured capacity -- then the
    next ``replay()`` runs it; otherwise run it eagerly on ``pool.batch(ids)`` --, and its node and page counts."""

    ids: np.ndarray
    fits: bool
    nodes: int
    pages: int


def _plan_words(ids: np.ndarray, starts: np.ndarray, batch_pages: int) -> np.ndarray:
    """int32 plan buffer contents (gte.h): [cursor 0, flag 0, nfit, B, L, 0, 0, 0 | ids | starts]"""
    words = np.zeros(ops.PLAN_HEADER + ids.size + starts.size, dtype=np.int32)
    words[2:5] = (starts.size, min(batch_pages, ids.size), ids.size)
    words[ops.PLAN_HEADER:ops.PLAN_HEADER + ids.size] = ids
    words[ops.PLAN_HEADER + ids.size:] = starts
    return words


def plan_slices(capacity: BatchCapacity, n_i: np.ndarray, e_i: np.ndarray, page_ids, batch_pages: int):
    """Host side of ``plan_epoch`` over a pool with per-page node / edge counts ``n_i`` / ``e_i``: ``page_ids`` cut
    into consecutive slices of ``batch_pages`` (the last may be short), each decided against ``capacity`` exactly as
    ``capacity.fits`` decides (vectorised over the slices).  Returns (list of PlannedBatch, int32 plan words)."""
    num_pages = len(n_i)
    if isinstance(batch_pages, bool) or not isinstance(batch_pages, (int, np.integer)) or batch_pages < 1:
        raise GteError(f"plan_epoch: batch_pages must be a positive int, got {batch_pages!r}")
    ids = np.asarray(page_ids)
    if ids.ndim != 1 or ids.size == 0 or not np.issubdtype(ids.dtype, np.integer):
        raise GteError(f"plan_epoch: page_ids must be a non-empty 1-D integer sequence, got {ids.dtype} {ids.shape}")
    if ids.size > num_pages:
        raise GteError(f"plan_epoch: {ids.size} page ids > the pool's {num_pages} pages (the device plan holds at most "
                       "one epoch over the pool)")
    if int(ids.min()) < 0 or int(ids.max()) >= num_pages:
        raise GteError(f"plan_epoch: page ids must lie in [0, {num_pages}), got [{int(ids.min())}, {int(ids.max())}]")
    ids = ids.astype(np.int64)
    b = int(batch_pages)
    starts = np.arange(0, ids.size, b, dtype=np.int64)
    pn, pe = n_i[ids], e_i[ids]
    nodes, edges = np.add.reduceat(pn, starts), np.add.reduceat(pe, starts)
    pages = np.minimum(b, ids.size - starts)
    fits = ((pages <= capacity.pages) & (nodes <= capacity.nodes) & (edges <= capacity.edges)
            & (np.maximum.reduceat(pn, starts) <= capacity.page_nodes)
            & (np.maximum.reduceat(pe, starts) <= capacity.page_edges))
    batches = [PlannedBatch(ids[s:s + p], bool(f), int(n), int(p)) for s, p, f, n in zip(starts, pages, fits, nodes)]
    return batches, _plan_words(ids, starts[fits], b)


def check_resident_capture(pool, capacity: Optional[BatchCapacity], world: int, in_feats: int) -> None:
    """Refuse a pass captured on a PagePool that cannot run: no capacity, data parallel, a feature width other than
    the model's input."""
    if capacity is None:
        raise GteError("capture: a pass on a PagePool needs a capacity (capacity=BatchCapacity(...))")
    if world > 1:
        raise GteError("capture: data parallel with a resident PagePool is not supported (each rank would need its own "
                       "pool shard); feed host batches on every rank")
    if pool.feat_width != in_feats:
        raise GteError(f"capture: the pool's features are {pool.feat_width} wide, the model takes {in_feats}")


def resident_warmup_ids(pool, capacity: BatchCapacity) -> np.ndarray:
    """The pool's first pages that fit ``capacity`` together (the capture's warm-up batch): pages no larger than the
    page caps, in pool order, as many as the page / node / edge totals allow."""
    ok = np.flatnonzero((pool.n_i <= capacity.page_nodes) & (pool.e_i <= capacity.page_edges))[:capacity.pages]
    k = int(np.count_nonzero((np.cumsum(pool.n_i[ok]) <= capacity.nodes) & (np.cumsum(pool.e_i[ok]) <= capacity.edges)))
    if k == 0:
        raise GteError("capture: no page of the pool fits the capacity")
    return ok[:k]


# ---------------------------------------------------------------------- the trainer's optimizer as torch.optim.Adam --
def check_adam_group(group: dict, where: str) -> Tuple[float, float, float, float, float]:
    """(lr, beta1, beta2, eps, weight_decay) of an Adam param group the trainer's kernels can run, validated by
    torch.optim.Adam's rules; a GteError names what they cannot run (a tensor value, AMSGrad, maximize, AdamW)."""
    for k in ("amsgrad", "maximize", "decoupled_weight_decay"):
        if group.get(k, False):
            raise GteError(f"{where}: {k}=True is not supported (plain Adam with L2 weight decay only)")
    lr, betas, eps, wd = group["lr"], group["betas"], group["eps"], group["weight_decay"]
    if not isinstance(betas, (tuple, list)) or len(betas) != 2:
        raise GteError(f"{where}: betas must be a pair, got {betas!r}")
    vals = (lr, betas[0], betas[1], eps, wd)
    for name, v in zip(("lr", "beta1", "beta2", "eps", "weight_decay"), vals):
        if isinstance(v, torch.Tensor):
            raise GteError(f"{where}: {name} as a tensor is not supported; assign a Python number")
        if isinstance(v, bool) or not isinstance(v, (int, float, np.integer, np.floating)):
            raise GteError(f"{where}: {name} must be a number, got {v!r}")
    lr, b1, b2, eps, wd = (float(v) for v in vals)
    # torch.optim.Adam.__init__'s checks (written so that NaN fails them)
    if not 0.0 <= lr:
        raise GteError(f"{where}: invalid learning rate: {lr}")
    if not 0.0 <= eps:
        raise GteError(f"{where}: invalid epsilon value: {eps}")
    if not 0.0 <= b1 < 1.0 or not 0.0 <= b2 < 1.0:
        raise GteError(f"{where}: invalid beta parameters: {(b1, b2)}")
    if not 0.0 <= wd:
        raise GteError(f"{where}: invalid weight_decay value: {wd}")
    return lr, b1, b2, eps, wd


def loaded_adam_step(state_dict: dict, shapes: Sequence[torch.Size]) -> int:
    """The step count of an Adam state dict for parameters of these shapes, in flat-buffer order (0: no state yet).
    Raises a GteError when the trainer cannot load it: other than one param group, a parameter count or shape other
    than the model's, per-parameter steps that differ, or a group the kernels cannot run (``check_adam_group``)."""
    groups = state_dict.get("param_groups")
    if not isinstance(groups, list) or len(groups) != 1:
        raise GteError(f"optimizer.load_state_dict: expected one param group, got "
                       f"{len(groups) if isinstance(groups, list) else groups!r}")
    group = groups[0]
    check_adam_group(group, "optimizer.load_state_dict")
    ids = list(group["params"])
    if len(ids) != len(shapes):
        raise GteError(f"optimizer.load_state_dict: {len(ids)} parameters, the model has {len(shapes)}")
    state = state_dict.get("state", {})
    if not any(i in state for i in ids):
        return 0
    steps = set()
    for j, (i, shape) in enumerate(zip(ids, shapes)):
        st = state.get(i)
        if not st:
            raise GteError(f"optimizer.load_state_dict: parameter {j} has no state while others have")
        for k in ("exp_avg", "exp_avg_sq"):
            t = st.get(k)
            if not isinstance(t, torch.Tensor) or tuple(t.shape) != tuple(shape):
                raise GteError(f"optimizer.load_state_dict: parameter {j}: {k} of shape "
                               f"{tuple(t.shape) if isinstance(t, torch.Tensor) else t!r}, expected {tuple(shape)}")
        step = st.get("step")  # a tensor since torch 1.12, an int before
        steps.add(float(step.item() if isinstance(step, torch.Tensor) else step))
    if len(steps) != 1:
        raise GteError(f"optimizer.load_state_dict: the parameters have different step counts {sorted(steps)}; the "
                       "trainer keeps one")
    step = steps.pop()
    if not (step >= 0 and step == int(step)):
        raise GteError(f"optimizer.load_state_dict: step {step} is not a count")
    return int(step)


class TrainerAdam(torch.optim.Adam):
    """``SageTrainer.optimizer``: a ``torch.optim.Adam`` over the model's parameters, in flat-buffer order, whose state
    lives in the trainer's device buffers.  Its one param group holds the hyper-parameters every update path of the
    trainer reads -- torch's schedulers change them through it -- and ``state_dict()`` / ``load_state_dict()`` speak
    torch's format, so checkpoints move between the trainer and a plain ``torch.optim.Adam`` over the same model.
    ``step()`` and ``zero_grad()`` are refused: the trainer's own steps update the parameters."""

    def __init__(self, trainer: "SageTrainer", params, lr, betas, eps, weight_decay):
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        self._trainer = trainer
        self._loaded_step = 0
        self.register_state_dict_pre_hook(TrainerAdam._state_from_device)
        self.register_load_state_dict_pre_hook(TrainerAdam._check_load)
        self.register_load_state_dict_post_hook(TrainerAdam._state_to_device)

    def step(self, closure=None):
        raise GteError("SageTrainer.optimizer.step(): the trainer applies Adam in its own steps (train_step / replay); "
                       "drive only the learning-rate schedule through the optimizer")

    def zero_grad(self, set_to_none: bool = True):
        raise GteError("SageTrainer.optimizer.zero_grad(): the trainer's backward overwrites its gradient buffer every "
                       "step (and set_to_none would detach the parameters' gradient views)")

    def add_param_group(self, param_group):
        if self.param_groups:
            raise GteError("SageTrainer.optimizer: one param group only (the trainer's flat parameter buffer)")
        super().add_param_group(param_group)

    def _views(self):
        tr = self._trainer
        return [(p, tr.exp_avg[o:o + p.numel()].view_as(p), tr.exp_avg_sq[o:o + p.numel()].view_as(p))
                for p, o in zip(self.param_groups[0]["params"], tr._offs)]

    def _set_state(self, step: int):
        """per-parameter state as torch.optim.Adam keeps it: empty before the first step, else a float32 CPU ``step``
        and views of the flat moment buffers"""
        self.state.clear()
        if step > 0:
            for p, m, v in self._views():
                self.state[p] = {"step": torch.tensor(float(step), dtype=torch.float32), "exp_avg": m, "exp_avg_sq": v}

    def _state_from_device(self):
        self._set_state(int(self._trainer.step_dev.item()))

    def _check_load(self, state_dict):
        self._loaded_step = loaded_adam_step(state_dict, [p.shape for p in self.param_groups[0]["params"]])

    def _state_to_device(self):
        # torch has cast the loaded moments to the parameters' device; copy them into the buffers captured graphs read
        tr, step = self._trainer, self._loaded_step
        with torch.no_grad():
            if step == 0:
                tr.exp_avg.zero_()
                tr.exp_avg_sq.zero_()
            else:
                for p, m, v in self._views():
                    m.copy_(self.state[p]["exp_avg"])
                    v.copy_(self.state[p]["exp_avg_sq"])
            tr.step_dev.fill_(step)
        self._set_state(step)


class SageTrainer:
    def __init__(self, model: GcnSAGE, lr: float = 0.01, weight_decay: float = 5e-4, betas=(0.9, 0.999),
                 eps: float = 1e-8, class_weights: Optional[torch.Tensor] = None, process_group=None):
        self.model = model
        params = list(model.parameters())
        if not params or not params[0].is_cuda:
            raise GteError("SageTrainer: move the model to a CUDA device first (no CPU path)")
        self.device = params[0].device
        for layer in model.layers:
            if layer.activation is not None and not _is_relu(layer.activation):
                raise GteError("SageTrainer: only activation=F.relu/None is fused; use the nn.Module path otherwise")
        self.class_w = None if class_weights is None else class_weights.to(self.device, torch.float32).contiguous()
        self.pg = process_group
        self.world = 1
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)

        # Dropout (models.py:30-33,60-61,113): masks come from Philox keyed by (seed, offset) held on the DEVICE, so a
        # captured step draws fresh masks on every replay: every call site of a step uses base offset + its own share,
        # and the base advances once per step (gte_rng_advance, captured with the step).
        self._drop_p = [_dropout_p(model.dropout)] + [_dropout_p(layer.dropout) for layer in model.layers]
        self.has_dropout = any(p > 0 for p in self._drop_p)
        gen = torch.cuda.default_generators[self.device.index if self.device.index is not None else torch.cuda.current_device()]
        rank = torch.distributed.get_rank(process_group) if self.world > 1 else 0
        # ranks share the seed (torch.manual_seed) but must not share masks: disjoint regions of the counter space
        self.rng_dev = torch.tensor([int(gen.initial_seed()) & (2 ** 63 - 1), rank << 44], dtype=torch.int64, device=self.device)
        # one flat fp32 buffer for parameters, gradients and both Adam moments;
        # the nn.Parameters become views, so state_dict()/load_state_dict() keep working
        total = sum(p.numel() for p in params)
        # every tensor starts on a 16-byte boundary so the kernels can vectorise
        offs, o = [], 0
        for p in params:
            offs.append(o)
            o += (p.numel() + 3) // 4 * 4
        # Data parallel: ONE all-reduce per step.  The loss statistics [sum w*nll, sum w, #correct] live in the tail of
        # the flat gradient buffer, every rank back-propagates the UN-normalised sum, the single SUM all-reduce carries
        # gradients and statistics together, and Adam divides by the global label-weight sum it finds in the tail
        # (gte_adam_step grad_den).  GTE_DP_FUSED=1 forces this path on one GPU (tests).
        self.dp_fused = self.world > 1 or os.environ.get("GTE_DP_FUSED", "0") == "1"
        self._flat_len = o
        self.flat_param = torch.zeros(o, dtype=torch.float32, device=self.device)
        self.flat_grad = None
        self._dp_peer = None
        if self.world > 1 and os.environ.get("GTE_DP_PEER", "1") != "0":
            self._setup_peer_exchange(o + 4)
        if self.flat_grad is None:
            self.flat_grad = torch.zeros(o + 4, dtype=torch.float32, device=self.device)
        self.exp_avg = torch.zeros(o, dtype=torch.float32, device=self.device)
        self.exp_avg_sq = torch.zeros(o, dtype=torch.float32, device=self.device)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.num_params = total
        self._offs = offs
        self._grad_views: Dict[int, torch.Tensor] = {}
        with torch.no_grad():
            for p, off in zip(params, offs):
                view = self.flat_param[off:off + p.numel()].view_as(p)
                view.copy_(p.data)
                p.data = view
                gv = self.flat_grad[off:off + p.numel()].view_as(p)
                p.grad = gv
                self._grad_views[id(p)] = gv
        self.stats = self.flat_grad[o:o + 3] if self.dp_fused else torch.zeros(3, dtype=torch.float32, device=self.device)
        # peer exchange: the tail of flat_grad keeps the LOCAL statistics, the fused kernel writes the global ones here
        self.stats_global = torch.zeros(4, dtype=torch.float32, device=self.device) if self._dp_peer else None
        self._one = torch.ones(1, dtype=torch.float32, device=self.device)
        if self.world > 1:
            # every rank must start from the same parameters / optimiser state (DDP broadcasts from rank 0 too):
            # do not rely on identical seeding
            for t in (self.flat_param, self.exp_avg, self.exp_avg_sq, self.step_dev):
                torch.distributed.broadcast(t, src=torch.distributed.get_global_rank(self.pg, 0) if self.pg is not None else 0,
                                            group=self.pg)
        self.num_classes = int(model.layers[-1].linear.weight.shape[0])
        self._train: Optional[_CapturedPass] = None  # the captured train or predict step
        self._mode = "train"
        # Adam's hyper-parameters [lr, beta1, beta2, eps, weight_decay] in device memory: every update path reads them
        # when it runs, so a learning-rate schedule reaches captured replays (a graph freezes by-value kernel
        # arguments).  optimizer.param_groups[0] is where they are set; _sync_hparams writes them here when they change.
        # Data parallel: every rank holds its own copy, so every rank must apply the same schedule.
        self.hparams = torch.zeros(5, dtype=torch.float32, device=self.device)
        self._hp_key = None
        self.optimizer = TrainerAdam(self, model.parameters(), lr, betas, eps, weight_decay)
        self._sync_hparams()

    # ------------------------------------------------------- optimiser -----
    @property
    def lr(self):
        """the learning rate of ``optimizer.param_groups[0]`` (the next step uses what is assigned here)"""
        return self.optimizer.param_groups[0]["lr"]

    @lr.setter
    def lr(self, value):
        self.optimizer.param_groups[0]["lr"] = value

    def _sync_hparams(self):
        """Called before every path that can run an update (train_step, replay, replay_set, replay_prefetched and the
        capture warm-up; the split tail runs inside the replays).  When the param group changed since the last call,
        validate it and write ``hparams`` with one copy, ordered on the current stream before the update; else this
        is one tuple comparison."""
        groups = self.optimizer.param_groups
        g = groups[0]
        key = (len(groups), g["lr"], g["betas"], g["eps"], g["weight_decay"], g["amsgrad"], g["maximize"],
               g.get("decoupled_weight_decay", False))
        if key != self._hp_key or isinstance(key[1], torch.Tensor):  # a tensor equal to the number compares equal
            if len(groups) != 1:
                raise GteError("SageTrainer.optimizer: one param group only (the trainer's flat parameter buffer)")
            vals = check_adam_group(g, "SageTrainer.optimizer")
            with torch.cuda.device(self.device):
                if torch.cuda.is_current_stream_capturing():
                    raise GteError("SageTrainer: Adam's hyper-parameters changed while a CUDA graph is being captured; "
                                   "the copy would be replayed with the graph.  Change them before or after the capture")
                # a fresh pinned staging tensor per write: the caching host allocator keeps it until the copy has run
                staging = torch.tensor(vals, dtype=torch.float32).pin_memory()
                self.hparams.copy_(staging, non_blocking=True)
            self._hp_key = key
        # LR schedulers warn about `scheduler.step()` before `optimizer.step()` unless the optimizer's `_opt_called`
        # (torch's private flag, set by the wrapper a scheduler puts around optimizer.step) is true.  optimizer.step()
        # is refused here, so the trainer's own updates count as the optimizer's steps.
        self.optimizer._opt_called = True

    # ----------------------------------------------------------- pieces ----
    def _layer_args(self, layer):
        has_ln = isinstance(layer.lynorm, nn.LayerNorm)
        return (layer.linear.weight.data, None if layer.linear.bias is None else layer.linear.bias.data,
                layer.lynorm.weight.data if has_ln else None, layer.lynorm.bias.data if has_ln else None, has_ln,
                layer.lynorm.eps if has_ln else 1e-5, _is_relu(layer.activation))

    def forward(self, g: PageGraphBatch, keep_ctx: bool = True, layer_outputs: Optional[list] = None,
                training: bool = False):
        """Layer loop of ``GcnSAGE.forward`` (models.py:105-116).  ``layer_outputs`` (tests): a list that receives every
        layer's output tensor (the parity tests read the ReLU on/off patterns from it).  ``training``: dropout active."""
        h = g.ndata["feat"]
        w_edge = g.edata["feat"]
        ctxs: List[L.LayerCtx] = []
        used = 0  # Philox counters consumed so far in this step
        drop_on = training and self.has_dropout
        if drop_on and self._drop_p[0] > 0:  # models.py:113: dropout on the input features (they need no gradient)
            h, _ = ops.dropout_concat(h, None, self._drop_p[0], rng_dev=self.rng_dev, offset=used)
            used += ops.dropout_counters(h.shape[0], h.shape[1])
        # tf32 hi / lo tiles of every layer's W in ONE launch (the layers would otherwise pack one by one)
        packs: Dict[int, torch.Tensor] = {}
        n_rows = h.shape[0]
        todo = [(li, layer.linear.weight.data, layer.linear.weight.shape[1] // 2)
                for li, layer in enumerate(self.model.layers)
                if L.wants_pack(n_rows, layer.linear.weight.shape[1] // 2, layer.linear.weight.shape[0], layer.use_pp)]
        if len(todo) > 1:
            for (li, _, _), pk in zip(todo, ops.umma_pack_weights_batch([(W, fin, 2) for _, W, fin in todo])):
                packs[li] = pk
        for li, layer in enumerate(self.model.layers):
            W, b, gamma, beta, has_ln, eps, relu = self._layer_args(layer)
            drop = None
            if drop_on and self._drop_p[1 + li] > 0:
                drop = L.DropoutSpec(self._drop_p[1 + li], 0, used, self.rng_dev)
                used += ops.dropout_counters(h.shape[0], W.shape[1])
            h, ctx = L.sage_layer_forward(g, h, w_edge, W, b, gamma, beta, ln=has_ln, relu=relu, eps=eps, agg=L.GCN,
                                          use_pp=layer.use_pp, save_for_backward=keep_ctx, dropout=drop,
                                          pack=packs.get(li))
            ctxs.append(ctx if keep_ctx else None)
            if layer_outputs is not None:
                layer_outputs.append(h)
        self._rng_used = used
        return h, ctxs

    def backward(self, g: PageGraphBatch, ctxs: List[L.LayerCtx], dlogits: torch.Tensor,
                 dy_comb: Optional[torch.Tensor] = None):
        dy = dlogits
        layers = list(self.model.layers)
        for i in range(len(layers) - 1, -1, -1):
            layer = layers[i]
            W, b, gamma, beta, has_ln, eps, relu = self._layer_args(layer)
            gv = self._grad_views
            dy = L.sage_layer_backward(
                g, ctxs[i], dy, W, gamma, beta, gv[id(layer.linear.weight)],
                None if layer.linear.bias is None else gv[id(layer.linear.bias)],
                gv[id(layer.lynorm.weight)] if has_ln else None, gv[id(layer.lynorm.bias)] if has_ln else None,
                need_dh=(i > 0), accumulate=False, dy_comb=dy_comb if i == len(layers) - 1 else None,
                dh_agg_first=True)

    def _all_reduce(self, t: torch.Tensor):
        if self.world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.SUM, group=self.pg)

    # The step in kernel-only stages (forward + loss, backward, exchange + update): with the peer-memory exchange they
    # are ONE CUDA graph; with the NCCL fallback the first two are captured and the collective + Adam run eagerly.
    def _stage_forward(self, g: PageGraphBatch, labels: torch.Tensor):
        logits, ctxs = self.forward(g, training=self.model.training)
        ops.cross_entropy_fwd(logits, labels, self.class_w, stats=self.stats)
        return logits, ctxs

    def _stage_backward(self, g: PageGraphBatch, labels: torch.Tensor, logits, ctxs):
        den = self._one if self.dp_fused else self.stats[1:2]
        dc = None
        if L.wants_class_grad_comb(ctxs[-1], logits.shape[0]):
            # the class layer consumes [d logits | A_hat^T d logits] as one operand: the loss backward writes its half in place
            dc = ops.cross_entropy_bwd_comb(logits, labels, self.class_w, den)
            dlogits = ops.comb_views(dc, logits.shape[1])[0]
        else:
            dlogits = ops.cross_entropy_bwd(logits, labels, self.class_w, den)
        self.backward(g, ctxs, dlogits, dy_comb=dc)
        if getattr(self, "_rng_used", 0) > 0:
            ops.rng_advance(self.rng_dev, self._rng_used)  # the next step (or graph replay) draws new masks

    def _stage_update(self):
        ops.adam_step(self.flat_param, self.flat_grad, self.exp_avg, self.exp_avg_sq, hparams=self.hparams,
                      step_dev=self.step_dev, grad_den=self.stats[1:2] if self.dp_fused else None, count=self._flat_len)

    def _setup_peer_exchange(self, numel: int):
        """Flat gradient buffer in symmetric memory (every rank can load every other rank's buffer over NVLink) for the
        fused all-reduce + Adam kernel.  Falls back to NCCL + gte_adam_step when the ranks cannot map each other."""
        try:
            import torch.distributed._symmetric_memory as symm_mem

            group = self.pg if self.pg is not None else torch.distributed.group.WORLD
            buf = symm_mem.empty(numel, dtype=torch.float32, device=self.device)
            buf.zero_()
            hdl = symm_mem.rendezvous(buf, group)
            if int(getattr(hdl, "offset", 0)) != 0 or hdl.world_size != self.world or hdl.signal_pad_size < 2048:
                raise RuntimeError("unexpected symmetric-memory layout")
            # this library's words of every rank's signal pad: 1 KB into the pad (torch's own barriers use its first words)
            pads = torch.tensor([int(p) + 1024 for p in hdl.signal_pad_ptrs], dtype=torch.int64, device=self.device)
            torch.cuda.synchronize(self.device)
            torch.distributed.barrier(group)
            self.flat_grad = buf
            self._dp_peer = {"hdl": hdl, "grad_ptrs": int(hdl.buffer_ptrs_dev), "pads": pads, "rank": int(hdl.rank),
                             "local": torch.zeros(4, dtype=torch.int32, device=self.device)}
        except Exception as exc:  # no P2P mapping (or an older torch): the NCCL path still works
            import warnings

            warnings.warn(f"SageTrainer: peer-memory gradient exchange unavailable ({type(exc).__name__}: {exc}); using NCCL")
            self.flat_grad, self._dp_peer = None, None

    def _stage_exchange_update(self):
        """gradient all-reduce + Adam: ONE kernel over NVLink peer memory when the ranks share symmetric memory, else one
        NCCL all-reduce (gradients + loss statistics in one buffer) + gte_adam_step"""
        if self._dp_peer is not None:
            d = self._dp_peer
            ops.dp_allreduce_adam(d["grad_ptrs"], d["pads"].data_ptr(), d["rank"], self.world, self._flat_len, self._flat_len,
                                  self.flat_param, self.exp_avg, self.exp_avg_sq, self.stats_global,
                                  hparams=self.hparams, step_dev=self.step_dev, local_words=d["local"])
        else:
            self._all_reduce(self.flat_grad)  # dp_fused: gradients + [sum w*nll, sum w, #correct] in one collective
            self._stage_update()

    def _result(self) -> torch.Tensor:
        return self.stats_global[:3] if self._dp_peer is not None else self.stats

    def step_stats(self) -> torch.Tensor:
        """device tensor [sum w*nll, sum w, #correct] of the last step (global over ranks)"""
        return self._result()

    def _stage_local(self, g: PageGraphBatch, labels: torch.Tensor):
        """the step up to the gradient exchange: forward + loss + backward"""
        logits, ctxs = self._stage_forward(g, labels)
        self._stage_backward(g, labels, logits, ctxs)
        return logits

    def _step_impl(self, g: PageGraphBatch, labels: torch.Tensor):
        logits = self._stage_local(g, labels)
        self._stage_exchange_update()
        return logits

    # ------------------------------------------------------------- API -----
    def train_step(self, g: PageGraphBatch, labels: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One optimisation step.  Returns the device tensor
        ``[sum w*nll, sum w, #correct]`` (global over ranks); loss = [0]/[1].
        No host synchronisation happens here."""
        if labels is None:
            labels = g.ndata["label"]
        with torch.cuda.device(self.device):
            self._sync_hparams()
            self._step_impl(g, labels)
        return self._result()

    @torch.no_grad()
    def predict(self, g: PageGraphBatch) -> torch.Tensor:
        """Batched inference logits (model_predict.py:144-146 does this page by page)."""
        with torch.cuda.device(self.device):
            logits, _ = self.forward(g, keep_ctx=False)
        return logits

    def _predict_impl(self, g: PageGraphBatch, labels: Optional[torch.Tensor]):
        """forward (nothing saved for a backward pass) + argmax + per-page correct counts, all on the device"""
        pages = g.pages()
        if pages is None:
            raise GteError("captured predict pass needs a page table (batch_num_nodes / batch_num_edges)")
        logits, _ = self.forward(g, keep_ctx=False)
        return ops.page_predictions(logits, pages[0], pages[1], labels)

    @torch.no_grad()
    def predict_pages(self, g: PageGraphBatch, labels: Optional[torch.Tensor] = None):
        """The predict loop of model_predict.py:130-154 for a whole batch of pages in one pass:
        returns (preds int32 [N] on device, per-page accuracy float64 tensor [P] on device or None).
        ``all_pred.extend(preds.tolist())`` and ``mean_test_acc += acc`` of the reference become
        ``preds.tolist()`` and ``acc.sum()`` over the batches."""
        if labels is None:
            labels = g.ndata.get("label")
        pages = g.pages()
        if pages is None:  # one huge graph: a single "page"
            pages = page_table([g.num_nodes()], [g.num_edges()], g.num_nodes(), g.device)
            if pages is None:
                off = torch.tensor([0, g.num_nodes()], dtype=torch.int32, device=g.device)
                pages = (off, 1, g.num_nodes(), g.num_edges())
        with torch.cuda.device(self.device):
            logits, _ = self.forward(g, keep_ctx=False)
            preds, correct = ops.page_predictions(logits, pages[0], pages[1], labels)
        acc = None
        if correct is not None:
            sizes = (pages[0][1:] - pages[0][:-1]).to(torch.float64)
            acc = correct.to(torch.float64) / sizes
        return preds, acc

    # ------------------------------------------------------- evaluation -----
    def _eval_impl(self, g: PageGraphBatch, labels: torch.Tensor, totals: torch.Tensor):
        """forward without dropout and without saved activations + gte_eval_accumulate into ``totals``: reads the
        parameters, writes nothing the train step reads (not rng_dev, not self.stats / the flat-gradient tail)"""
        logits, _ = self.forward(g, keep_ctx=False)
        ops.eval_accumulate(logits, labels, self.class_w, totals)

    def eval_totals(self) -> torch.Tensor:
        """A zeroed float64 device buffer [2 + C*C] for ``evaluate``: [sum w*nll, sum w, confusion counts C x C]."""
        return torch.zeros(2 + self.num_classes ** 2, dtype=torch.float64, device=self.device)

    @torch.no_grad()
    def evaluate(self, g: PageGraphBatch, labels: Optional[torch.Tensor] = None,
                 totals: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The validation step of model_train.py:349-364 on the device: forward (always without dropout, nothing saved
        for a backward pass), then the weighted CE statistics and the confusion matrix of ``torch.argmax`` ADDED to
        ``totals`` (a fresh ``eval_totals()`` when None), which is returned.  Rows with a label outside [0, C) are
        skipped.  ``EvalCapture.result`` shows how to read the totals.  No host synchronisation happens here."""
        if labels is None:
            labels = g.ndata["label"]
        if totals is None:
            totals = self.eval_totals()
        with torch.cuda.device(self.device):
            self._eval_impl(g, labels, totals)
        return totals

    def capture_eval(self, host_batch, capacity: Optional[BatchCapacity] = None) -> "EvalCapture":
        """Capture ``evaluate`` as a pass of its own, beside the captured train step (which stays): without a capacity
        for batches of this shape -- ``host_batch`` stays resident and ``replay()`` copies nothing, the fixed
        validation batch of model_train.py:242-249 --, with one for every batch that fits it (see ``capture``), or on
        a ``PagePool`` with a capacity (``plan_epoch`` + ``replay``, see ``capture``).  The pass has its own memory
        pool and totals buffer and reads the live parameters, so after a train replay it sees the updated weights."""
        return EvalCapture(self, host_batch, capacity)

    def _check_resident(self, pool: PagePool, capacity: Optional[BatchCapacity]):
        check_resident_capture(pool, capacity, self.world, int(self.model.layers[0].linear.weight.shape[1]) // 2)

    # ----------------------------------------------------- CUDA graphs -----
    @property
    def _static(self) -> Optional[Dict[str, torch.Tensor]]:
        """static input set 0 of the captured train / predict step"""
        return None if self._train is None else self._train.statics[0]

    @property
    def _statics(self) -> Optional[List[Dict[str, torch.Tensor]]]:
        return None if self._train is None else self._train.statics

    @property
    def _graph(self):
        return None if self._train is None else self._train.graphs[0]

    def capture_predict(self, host_batch, capacity: Optional[BatchCapacity] = None):
        """Capture the batched predict pass of model_predict.py:130-154 (format build + forward without saved
        activations + argmax + per-page correct counts) for batches of this shape, or for every batch that fits
        ``capacity`` (see ``capture``).  Feed batches with ``load_batch`` / ``prefetch_batch`` (on a ``PagePool``:
        ``plan_epoch``); ``replay()`` / ``replay_prefetched()`` then return ``(preds int32 [N], page_correct int32
        [P])`` -- views of static device tensors of the input set that ran, sized for the batch in it, valid until
        that set runs again."""
        return self.capture(host_batch, capacity=capacity, split=False, mode="predict")

    def capture(self, host_batch, capacity: Optional[BatchCapacity] = None, split: Optional[bool] = None,
                mode: str = "train"):
        """Capture the whole step (format build + forward + loss + backward +
        optimiser) for batches with exactly this node / edge count.  Later
        batches are fed with ``load_batch`` + ``replay``.  ``split`` (default: data-parallel
        runs) captures the kernels in one graph and leaves the all-reduce and Adam outside it.

        ``capacity``: capture once for every batch that fits it (``fits()``), e.g. the shuffled batches of real pages
        of model_train.py:283-297.  The static inputs have the capacity's padded shape; a batch is copied as it is and
        ``gte_pad_batch``, the first kernel of the graph, pads it on the device with zero-feature, label -1 nodes and
        weight-0 self-loops in pages of their own, which change no loss statistic and no gradient.  ``host_batch``
        must fit; it gives the feature width and the warm-up contents.

        ``host_batch`` may be a ``PagePool`` instead (``capacity`` required, one GPU): the pass then gathers its
        batches from the pool on the device -- its first kernels plan the next batch of an epoch plan and copy its
        pages into the static inputs --, so an epoch costs one upload of page ids (``plan_epoch``) and one
        ``replay()`` per fitting batch, with no host batching and no per-batch copy.  The warm-up runs on the pool's
        first pages that fit.

        A trainer holds one captured step: a new capture replaces the previous one.  A pass captured by
        ``capture_eval`` is separate and stays."""
        if split is None:
            split = self.world > 1 and self._dp_peer is None  # the peer-memory exchange is an ordinary kernel: one graph
        if mode not in ("train", "predict"):
            raise GteError(f"capture: unknown mode {mode}")
        if isinstance(host_batch, PagePool):
            self._check_resident(host_batch, capacity)
        if mode == "predict":
            body, tail = self._predict_impl, None
        elif split:  # [graph: batch assembly + forward + CE + backward] -> ONE all-reduce -> Adam (eager, 2 launches)
            body, tail = self._stage_local, self._stage_exchange_update
        else:
            body, tail = self._step_impl, None
        if mode == "train":
            self._sync_hparams()  # the warm-up steps run with the current hyper-parameters
        # the warm-up steps train: restore the optimiser state afterwards
        snap = (self.flat_param.clone(), self.exp_avg.clone(), self.exp_avg_sq.clone(), self.step_dev.clone())
        self._train = _CapturedPass(self.device, host_batch, capacity, body, tail)
        self._mode = mode
        self.flat_param.copy_(snap[0])
        self.exp_avg.copy_(snap[1])
        self.exp_avg_sq.copy_(snap[2])
        self.step_dev.copy_(snap[3])
        return self._graph

    def _captured(self, what: str) -> "_CapturedPass":
        if self._train is None:
            raise GteError(f"{what}: call capture() first")
        return self._train

    def _before_replay(self):
        if self._mode == "train":
            self._sync_hparams()

    def fits(self, host_batch: Dict[str, torch.Tensor]) -> bool:
        """True when ``host_batch`` can run through the captured step (``load_batch`` / ``prefetch_batch`` accept it).
        Route a batch that does not fit to ``train_step`` / ``predict_pages``."""
        return self._captured("fits").fits(host_batch)

    def plan_epoch(self, page_ids, batch_pages: int) -> List[PlannedBatch]:
        """Plan an epoch of a step captured on a ``PagePool``: ``page_ids`` (at most ``pool.num_pages`` ids, in the
        caller's order -- e.g. a permutation, trimmed by a loop that drops the last short batch) is cut into
        consecutive batches of ``batch_pages`` pages, the last possibly short.  One copy uploads the ids and the
        batches that fit the capacity; every later ``replay()`` runs the next of them.  Returns the batches in
        order; run one that does not fit eagerly: ``train_step(pool.batch(b.ids))`` / ``predict_pages(...)``."""
        return self._captured("plan_epoch").plan_epoch(page_ids, batch_pages)

    def load_batch(self, host_batch: Dict[str, torch.Tensor]):
        """Copy a host batch into static input set 0.  The batch must have the captured node / edge totals and page
        count and no page larger than the captured maxima; page ORDER and SIZES may differ (the page table is
        refreshed with the batch).  Capacity capture: any batch that fits the capacity; one that does not is refused
        with a GteError before anything is copied."""
        self._captured("load_batch").load_batch(host_batch)

    def _outputs(self, which: int):
        if self._mode == "predict":
            preds, correct = self._train.outs[which]
            if self._train.capacity is not None:  # the batch that ran, without its padding
                n, p = self._train.rows[which]
                return preds[:n], correct[:p]
            return preds, correct
        return self._result()

    def replay(self):
        """Run the captured step on input set 0 -- on a ``PagePool``: on the next planned batch that fits --; returns
        the statistics (train) or ``(preds, page_correct)`` of the batch (predict)."""
        self._captured("replay")
        self._before_replay()
        self._train.replay_next()
        return self._outputs(0)

    def prefetch_batch(self, host_batch: Dict[str, torch.Tensor]):
        """Start the H2D copy of the NEXT batch on a side stream.  Two static input sets alternate, each with its own
        captured graph (sharing one memory pool), so the step reads the batch where the copy engine put it: no
        device-to-device staging copy.  ``replay_prefetched()`` consumes the sets in order."""
        self._captured("prefetch_batch").prefetch_batch(host_batch)

    def replay_set(self, which: int) -> torch.Tensor:
        """Run one captured step on static input set ``which`` (0 or 1) as it is: inputs resident in HBM, no copy.
        The sets are filled by ``prefetch_batch`` / ``load_batch``; the caller keeps track of what is in them."""
        self._captured("replay_set")
        self._before_replay()
        self._train.replay_set(which)
        return self._outputs(which)

    def replay_prefetched(self):
        """Run one captured step on the oldest prefetched batch."""
        if self._train is None:
            raise GteError("replay_prefetched: no prefetched batch")
        self._before_replay()
        return self._outputs(self._train.replay_prefetched())


class _CapturedPass:
    """One captured pass: the CUDA graph of ``body(g, labels)`` over static input sets, and everything that feeds it --
    the static inputs of the batch shape or of a ``BatchCapacity`` (padded on the device by gte_pad_batch, the first
    kernel of the graph), the validation and page layout of a fed batch, its host->device copies and the two-set
    prefetch pipeline.  ``outs[i]`` keeps what ``body`` returned while capturing over input set i.  ``tail`` (may be
    None) runs eagerly after every replay: the data-parallel all-reduce + Adam of a split train step.

    Captured on a ``PagePool`` (a resident pass; capacity capture with one input set), the graph starts with
    gte_gather_plan + gte_gather_pages, which assemble the next batch of the device epoch plan ``plan`` from the pool;
    the host keeps the same plan's (n, P) per fitting batch to cut the outputs and to refuse a replay past it."""

    def __init__(self, device, source, capacity: Optional[BatchCapacity], body, tail=None):
        self.pool = source if isinstance(source, PagePool) else None
        host_batch = None if self.pool is not None else source
        if self.pool is not None:
            self._check_capacity(capacity, None)
            warm = resident_warmup_ids(self.pool, capacity)
        elif capacity is not None:
            self._check_capacity(capacity, host_batch)
        self.device, self.capacity, self.body, self.tail = device, capacity, body, tail
        dev = device
        if capacity is None:
            n, e = int(host_batch["num_nodes"]), int(host_batch["src"].numel())
            f = self.feat_width = int(host_batch["feat"].shape[1])
            st = {
                "src": torch.empty(e, dtype=torch.int32, device=dev),
                "dst": torch.empty(e, dtype=torch.int32, device=dev),
                "weight": torch.empty(e, dtype=torch.float32, device=dev),
                "feat": torch.empty((n, f), dtype=torch.float32, device=dev),
                "label": torch.empty(n, dtype=torch.float32, device=dev),
            }
            bn, be = list(host_batch["batch_num_nodes"]), list(host_batch["batch_num_edges"])
            self.meta = (n, e, bn, be)
            # The page table (node / edge offsets of the pages) is part of the INPUT: a later batch with the same totals
            # may order or size its pages differently, so every static input set owns device copies of the two offset
            # arrays and load_batch / prefetch_batch refresh them.  Only the maxima (shared-memory sizing of the page
            # kernels) and the page count are fixed at capture time.
            pages = page_table(bn, be, n, dev)
            if pages is not None:
                st["page_off"], st["edge_off"] = pages[0], pages[4]
                self.caps = (pages[1], pages[2], pages[3])  # page count, max page nodes, max page edges
            else:
                self.caps = None
        else:
            n_cap, e_cap, p_cap = capacity.shape
            if self.pool is not None:
                self.feat_width = self.pool.feat_width
                bn, be = self.pool.n_i[warm], self.pool.e_i[warm]
            else:
                self.feat_width = int(host_batch["feat"].shape[1])
                bn, be = host_batch["batch_num_nodes"], host_batch["batch_num_edges"]
            st = self._capacity_set()
            # the structure the captured kernels see: P_cap pages, none larger than the capacity's page caps (the
            # page lists only size the batch; the offsets come from st["page_off"] / st["edge_off"] every replay)
            po, eo = padded_page_table(capacity, bn, be)
            self.meta = (n_cap, e_cap, np.diff(po).tolist(), np.diff(eo).tolist())
            self.caps = (p_cap, capacity.page_nodes, capacity.page_edges)
        self.rows = [None, None]  # capacity capture: (n, P) of the batch in each input set
        self.loaded_layout = [None, None]
        self.statics = [st]
        self.stage_sets = None
        if self.pool is None:
            self.load_batch(host_batch)
        else:
            # the device plan holds one epoch over the pool: its pointer is captured, so it is sized once, here
            self.plan = torch.zeros(ops.PLAN_HEADER + 2 * self.pool.num_pages, dtype=torch.int32, device=dev)
            # a plan of the one warm-up batch (nfit = 1 <= L = len(warm) for any warm-up, as the plan kernel requires),
            # uploaded again before each warm-up run
            warm_words = _plan_words(warm, np.zeros(1, dtype=np.int64), len(warm))

        # warm-up on a side stream (allocator + lazy module state)
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            for _ in range(2):
                if self.pool is not None:
                    self._upload_plan(warm_words)
                self.run_eager(st)
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize(dev)
        self._check_static_structure(st)
        self.outs = [None, None]
        self.graphs = [self._capture_over(0)]
        self._plan_rows, self._plan_next, self._plan_checked = [], 0, True  # no epoch planned yet

    def run_eager(self, st):
        """the captured pass over static input set ``st``, launched eagerly (warm-up)"""
        self._pad(st)
        out = self.body(self.graph_of(st), st["label"])
        if self.tail is not None:
            self.tail()
        return out

    def graph_of(self, st) -> PageGraphBatch:
        n = self.meta[0]
        g = PageGraphBatch(st["src"], st["dst"], n, self.meta[2], self.meta[3])
        caps = self.caps
        g._cache["pages"] = None if caps is None else (st["page_off"], caps[0], caps[1], caps[2], st["edge_off"])
        g.edata["feat"] = st["weight"]
        g.ndata["feat"] = st["feat"]
        return g

    def _check_static_structure(self, st):
        """Host check (one synchronisation, capture time only) that the batch in ``st`` honours its page table: the
        one-kernel batch assembly raises a device flag when an edge leaves its page (results would be undefined)."""
        g = self.graph_of(st)
        if g.prepare(st["weight"]):
            g.check_page_structure()
        if "pad_bad" in st and int(st["pad_bad"].item()) != 0:
            raise GteError("capture: gte_pad_batch flagged the padded batch (word outside the capacity or bad page table)")
        if self.pool is not None:
            self._check_plan_flag("capture")

    # -- capacity capture: one graph for every batch that fits a BatchCapacity ------------------------------------
    @classmethod
    def _check_capacity(cls, capacity: BatchCapacity, host_batch):
        if not isinstance(capacity, BatchCapacity):
            raise GteError(f"capture: capacity must be a BatchCapacity, got {type(capacity).__name__}")
        _, _, p_cap = capacity.shape
        if not ops.page_formats_supported((None, p_cap, capacity.page_nodes, capacity.page_edges)):
            raise GteError(f"capture: pages of {capacity.page_nodes} nodes / {capacity.page_edges} edges do not fit the "
                           "one-kernel batch assembly (shared memory); lower page_nodes / page_edges")
        if host_batch is not None:
            cls._check_fit(capacity, host_batch, int(host_batch["feat"].shape[1]))

    @staticmethod
    def _check_fit(capacity: BatchCapacity, host_batch, f: int):
        bn, be = list(host_batch["batch_num_nodes"]), list(host_batch["batch_num_edges"])
        capacity.check(bn, be)
        n, e = int(host_batch["num_nodes"]), int(host_batch["src"].numel())
        if sum(bn) != n or sum(be) != e:
            raise GteError("captured step: page sizes do not add up to the batch's node / edge totals")
        feat = host_batch["feat"]
        if feat.dim() != 2 or int(feat.shape[0]) != n or int(feat.shape[1]) != f:
            raise GteError(f"captured step: features {tuple(feat.shape)}, expected [{n}, {f}]")
        if host_batch["label"].numel() != n or host_batch["dst"].numel() != e or host_batch["weight"].numel() != e:
            raise GteError("captured step: label / dst / weight sizes do not match the batch totals")

    def _capacity_set(self) -> Dict[str, torch.Tensor]:
        """One static input set of the capacity shape.  ``meta`` = [n, e, P, 0 | page_off (P_cap + 1) | edge_off
        (P_cap + 1)] travels in ONE copy; ``word``, ``page_off`` and ``edge_off`` are views of it."""
        dev = self.device
        n_cap, e_cap, p_cap = self.capacity.shape
        meta = torch.zeros(4 + 2 * (p_cap + 1), dtype=torch.int32, device=dev)
        return {
            "src": torch.zeros(e_cap, dtype=torch.int32, device=dev),
            "dst": torch.zeros(e_cap, dtype=torch.int32, device=dev),
            "weight": torch.zeros(e_cap, dtype=torch.float32, device=dev),
            "feat": torch.zeros((n_cap, self.feat_width), dtype=torch.float32, device=dev),
            "label": torch.zeros(n_cap, dtype=torch.float32, device=dev),
            "meta": meta, "word": meta[:4], "page_off": meta[4:5 + p_cap], "edge_off": meta[5 + p_cap:],
            "pad_bad": torch.zeros(1, dtype=torch.int32, device=dev),
        }

    def _pad(self, st):
        """first kernels of a capacity-captured pass: (resident: plan the next batch and gather it from the pool,) pad
        the batch in ``st`` to the capacity shape"""
        if self.pool is not None:
            pool = self.pool
            ops.gather_plan(self.plan, pool.n_dev, pool.e_dev, self.capacity, st["meta"])
            ops.gather_pages(self.plan, st["meta"], self.capacity, pool.node_off, pool.edge_off, pool.coo[0], pool.coo[1],
                             pool.w_coo, pool.feat, pool.label, st["src"], st["dst"], st["weight"], st["feat"],
                             st["label"])
        if self.capacity is not None:
            ops.pad_batch(st["word"], st["page_off"], st["edge_off"], st["src"], st["dst"], st["weight"], st["feat"],
                          st["label"], bad=st["pad_bad"])

    # -- resident pass: batches planned over the pool, gathered on the device ------------------------------------
    def _host_fed(self, what: str):
        if self.pool is not None:
            raise GteError(f"{what}: this pass gathers its batches from a PagePool; use plan_epoch() + replay()")

    def _upload_plan(self, words: np.ndarray):
        # a fresh pinned staging tensor per upload, as in _copy_inputs: a queued copy never reads a rewritten buffer
        staging = torch.empty(words.size, dtype=torch.int32, pin_memory=True)
        staging.numpy()[:] = words
        self.plan[:words.size].copy_(staging, non_blocking=True)

    def _check_plan_flag(self, what: str):
        flag = int(self.plan[1].item())
        if flag:
            raise GteError(f"{what}: the resident pass's gather kernels flagged the plan ({flag}: 1 = past the plan, "
                           "2 = a batch did not fit or named a page outside the pool, 4 = page table and pool disagree)")

    def plan_epoch(self, page_ids, batch_pages: int) -> List[PlannedBatch]:
        if self.pool is None:
            raise GteError("plan_epoch: the pass was captured on a host batch; capture it on a PagePool")
        batches, words = plan_slices(self.capacity, self.pool.n_i, self.pool.e_i, page_ids, batch_pages)
        self._upload_plan(words)
        self._plan_rows = [(b.nodes, b.pages) for b in batches if b.fits]
        self._plan_next, self._plan_checked = 0, False
        return batches

    def replay_next(self):
        """``replay()`` of the public API: input set 0, or the next planned batch of a resident pass"""
        if self.pool is None:
            self.replay(0)
            return
        if self._plan_next >= len(self._plan_rows):
            raise GteError(f"replay: all {len(self._plan_rows)} fitting batches of the plan have run; call plan_epoch()")
        self.rows[0] = self._plan_rows[self._plan_next]
        self._plan_next += 1
        self.replay(0)
        if not self._plan_checked:  # once per plan: one host read
            self._plan_checked = True
            self._check_plan_flag("replay")

    def fits(self, host_batch: Dict[str, torch.Tensor]) -> bool:
        self._host_fed("fits")
        try:
            self._page_layout(host_batch)
        except GteError:
            return False
        return True

    def _page_layout(self, host_batch):
        """Validated (page_off, edge_off) host int32 tensors of a batch fed to a captured pass, or None when the
        captured pass has no page table.  Raises when the batch cannot run through the captured kernels.  Capacity
        capture: (n, e, P, key) of the batch, the padded page table is built when it is copied."""
        if self.capacity is not None:
            self._check_fit(self.capacity, host_batch, self.feat_width)
            bn, be = tuple(host_batch["batch_num_nodes"]), tuple(host_batch["batch_num_edges"])
            return int(host_batch["num_nodes"]), int(host_batch["src"].numel()), len(bn), (bn, be)
        n, e, bn0, be0 = self.meta
        if int(host_batch["num_nodes"]) != n or int(host_batch["src"].numel()) != e:
            raise GteError("captured step: batch node / edge totals differ from the captured ones")
        feat = host_batch["feat"]
        if feat.dim() != 2 or int(feat.shape[1]) != self.feat_width:
            raise GteError(f"captured step: features {tuple(feat.shape)}, expected [{n}, {self.feat_width}]")
        if self.caps is None:
            return None
        bn, be = list(host_batch["batch_num_nodes"]), list(host_batch["batch_num_edges"])
        p, max_n, max_e = self.caps
        if len(bn) != p or len(be) != p or sum(bn) != n or sum(be) != e:
            raise GteError("captured step: page count / page sizes do not add up to the captured batch shape")
        if max(bn) > max_n or max(be) > max_e:
            raise GteError(f"captured step: largest page ({max(bn)} nodes, {max(be)} edges) exceeds the captured maxima "
                           f"({max_n}, {max_e}) the page kernels were sized for; capture with the largest batch first")
        if "page_off" in host_batch and "edge_off" in host_batch:
            return host_batch["page_off"], host_batch["edge_off"], (bn, be)
        po = np.zeros(p + 1, dtype=np.int32)
        eo = np.zeros(p + 1, dtype=np.int32)
        np.cumsum(np.asarray(bn, dtype=np.int64), out=po[1:])
        np.cumsum(np.asarray(be, dtype=np.int64), out=eo[1:])
        return torch.from_numpy(po), torch.from_numpy(eo), (bn, be)

    def _copy_inputs(self, which: int, host_batch, layout):
        st = self.statics[which]
        if self.capacity is not None:
            # the real prefix only: H2D bytes and host work follow the batch, not the capacity (the graph pads)
            n, e, p, key = layout
            for k, m in (("src", e), ("dst", e), ("weight", e), ("feat", n), ("label", n)):
                st[k][:m].copy_(host_batch[k], non_blocking=True)
            if self.loaded_layout[which] != key:
                # a fresh pinned staging tensor per load: torch's caching host allocator keeps it until its
                # non-blocking copy has run, so a queued copy never reads a rewritten buffer
                po, eo = padded_page_table(self.capacity, key[0], key[1])
                meta = torch.empty(st["meta"].numel(), dtype=torch.int32, pin_memory=True)
                m = meta.numpy()
                m[:4] = (n, e, p, 0)
                m[4:4 + po.size] = po
                m[4 + po.size:] = eo
                st["meta"].copy_(meta, non_blocking=True)
                self.loaded_layout[which] = key
            self.rows[which] = (n, p)
            return
        for k in ("src", "dst", "weight", "feat", "label"):
            st[k].copy_(host_batch[k], non_blocking=True)
        if layout is not None:
            po, eo, key = layout
            if self.loaded_layout[which] != key:  # fixed-size pages: the offsets never change, skip the copies
                st["page_off"].copy_(po, non_blocking=True)
                st["edge_off"].copy_(eo, non_blocking=True)
                self.loaded_layout[which] = key

    def _capture_over(self, which: int, pool=None):
        """Capture the pass reading static input set ``which`` (capturing launches nothing)."""
        st = self.statics[which]
        graph = torch.cuda.CUDAGraph()
        kw = {} if pool is None else {"pool": pool}
        # No cyclic garbage collection while capturing.  Trainers and their passes reference each other, so a discarded
        # trainer's CUDA graphs are freed by the cyclic collector, whenever it happens to run; destroying a graph while
        # a stream captures invalidates the capture.  torch.cuda.graph no longer runs gc.collect() before capturing
        # (torch 2.11), and this showed up as a capture failing with cudaErrorStreamCaptureInvalidated after
        # "operation not permitted when stream is capturing (function reset)" warnings, in a test that ran after
        # others had dropped captured trainers.
        gc_was_on = gc.isenabled()
        gc.disable()
        try:
            with torch.cuda.graph(graph, **kw):
                self._pad(st)
                self.outs[which] = self.body(self.graph_of(st), st["label"])
        finally:
            if gc_was_on:
                gc.enable()
        return (graph,) if self.tail is not None else graph

    def load_batch(self, host_batch: Dict[str, torch.Tensor]):
        self._host_fed("load_batch")
        self._copy_inputs(0, host_batch, self._page_layout(host_batch))

    def replay(self, which: int = 0):
        graph = self.graphs[which]
        if isinstance(graph, tuple):
            graph[0].replay()
            self.tail()
        else:
            graph.replay()

    # -- pipelined input: the host->device copy of batch i+1 overlaps the pass over batch i ----------------------
    def prefetch_batch(self, host_batch: Dict[str, torch.Tensor]):
        self._host_fed("prefetch_batch")
        layout = self._page_layout(host_batch)
        if self.stage_sets is None:
            torch.cuda.synchronize(self.device)
            self._copy_stream = torch.cuda.Stream(device=self.device)
            first = self.statics[0]
            if self.capacity is None:
                second = {k: torch.empty_like(v) for k, v in first.items()}
                for k, v in first.items():
                    second[k].copy_(v)  # valid contents for the capture below (capturing runs nothing)
            else:
                second = self._capacity_set()  # word / page_off / edge_off are views of meta: allocate, do not clone
                for k in ("src", "dst", "weight", "feat", "label", "meta"):
                    second[k].copy_(first[k])
                self.rows[1] = self.rows[0]
            self.loaded_layout[1] = self.loaded_layout[0]
            pool = (self.graphs[0][0] if isinstance(self.graphs[0], tuple) else self.graphs[0]).pool()
            self.statics.append(second)
            self.graphs.append(self._capture_over(1, pool=pool))
            self.stage_sets = self.statics
            self._stage_ready = [torch.cuda.Event(), torch.cuda.Event()]
            self._stage_free = [torch.cuda.Event(), torch.cuda.Event()]
            self._stage_w = self._stage_r = 0
            # set 0 may still be read by work queued before this call
            self._stage_free[0].record(torch.cuda.current_stream(self.device))
            self._stage_free[1].record(torch.cuda.current_stream(self.device))
        if self._stage_w - self._stage_r >= 2:
            raise GteError("prefetch_batch: both input sets hold unconsumed batches; call replay_prefetched() first")
        i = self._stage_w % 2
        cs = self._copy_stream
        cs.wait_event(self._stage_free[i])  # the pass that last read input set i has finished
        with torch.cuda.stream(cs):
            self._copy_inputs(i, host_batch, layout)
            self._stage_ready[i].record(cs)
        self._stage_w += 1

    def replay_set(self, which: int):
        self._host_fed("replay_set")
        if self.stage_sets is None and which != 0:
            raise GteError("replay_set: the second input set exists after the first prefetch_batch()")
        self.replay(which)

    def replay_prefetched(self) -> int:
        """Run the pass on the oldest prefetched batch; returns the input set it read."""
        self._host_fed("replay_prefetched")
        if self.stage_sets is None or self._stage_r >= self._stage_w:
            raise GteError("replay_prefetched: no prefetched batch")
        i = self._stage_r % 2
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(self._stage_ready[i])
        self.replay(i)
        self._stage_free[i].record(cur)
        self._stage_r += 1
        return i


class EvalCapture:
    """A captured evaluation pass (``SageTrainer.capture_eval``): forward without dropout + gte_eval_accumulate into
    one float64 device buffer ``totals`` = [sum w*nll, sum w, confusion counts C x C (rows: true class, columns:
    prediction)].  Replays ADD to the totals, so one ``reset()`` per epoch followed by replays over the validation
    batches sums the epoch; ``result()`` reads it.  Feed batches as for the captured train step: ``load_batch`` +
    ``replay()`` or ``prefetch_batch`` + ``replay_prefetched()``; a batch that does not ``fits()`` goes to ``run(g)``.

    Captured on a ``PagePool`` (with a capacity): ``plan_epoch(ids, B)`` once per epoch, then ``replay()`` per
    planned batch that fits and ``run(pool.batch(b.ids))`` for the others.

    Data parallel: every rank evaluates its own shard; ``all_reduce(totals, SUM)`` once per epoch before
    ``result()`` gives the global numbers."""

    def __init__(self, trainer: SageTrainer, host_batch, capacity: Optional[BatchCapacity]):
        if isinstance(host_batch, PagePool):
            trainer._check_resident(host_batch, capacity)
        self._trainer = trainer
        self.num_classes = trainer.num_classes
        self.totals = trainer.eval_totals()
        totals = self.totals
        self._pass = _CapturedPass(trainer.device, host_batch, capacity,
                                   lambda g, labels: trainer._eval_impl(g, labels, totals))
        self.reset()  # the warm-up passes accumulated into the totals

    def fits(self, host_batch: Dict[str, torch.Tensor]) -> bool:
        """True when ``host_batch`` can run through the captured pass; route one that does not to ``run``."""
        return self._pass.fits(host_batch)

    def load_batch(self, host_batch: Dict[str, torch.Tensor]):
        """Copy a host batch into the pass's static input set 0 (refused with a GteError before anything is copied
        when it does not fit)."""
        self._pass.load_batch(host_batch)

    def prefetch_batch(self, host_batch: Dict[str, torch.Tensor]):
        """Start the H2D copy of the next batch on a side stream (two input sets alternate, as for the train step)."""
        self._pass.prefetch_batch(host_batch)

    def plan_epoch(self, page_ids, batch_pages: int) -> List[PlannedBatch]:
        """Plan the validation batches of a pass captured on a ``PagePool`` (see ``SageTrainer.plan_epoch``)."""
        return self._pass.plan_epoch(page_ids, batch_pages)

    def replay(self) -> torch.Tensor:
        """Evaluate the batch in input set 0 (a resident batch needs no copy) -- on a ``PagePool``: the next planned
        batch that fits --; returns ``totals``."""
        self._pass.replay_next()
        return self.totals

    def replay_prefetched(self) -> torch.Tensor:
        """Evaluate the oldest prefetched batch; returns ``totals``."""
        self._pass.replay_prefetched()
        return self.totals

    def run(self, g: PageGraphBatch, labels: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Eager evaluation of a batch into the same totals (for batches that do not fit the capture)."""
        return self._trainer.evaluate(g, labels, totals=self.totals)

    def reset(self):
        """Zero the totals (once per epoch)."""
        self.totals.zero_()

    def result(self) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """Device tensors (loss = sum w*nll / sum w, accuracy = trace / sum of counts, cm int64 [C, C]) of the
        totals.  ``metrics.precision_recall_f1(cm)`` gives the per-class scores."""
        t = self.totals
        cm = t[2:].view(self.num_classes, self.num_classes).to(torch.int64)
        return t[0] / t[1], cm.trace().to(torch.float64) / cm.sum(), cm
