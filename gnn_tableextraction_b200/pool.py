"""``PagePool`` -- dataset-resident page graphs with pre-built sparse formats.

Replaces the per-step host work of the reference's train loop
(/root/reference/src/models/model_train.py:286-297: slice the page list,
``dgl.batch(train_batch).to(device)``, then two lazy COO->CSC/CSR sorts inside
DGL) for datasets that fit in HBM (180 GB holds ~10^8 word boxes with BBOX
features): every page's COO, edge weights, features and labels live on the GPU
with page-local ids.  Two ways to batch them:
  * ``PagePool.batch`` (eager) assembles a batch with its CSC / CSR by
    ``gte_batch_concat_csx`` -- an offset-concatenation that is bit-identical to a
    stable sort of the batched COO because node ids are page-major; the pool-wide
    CSC / CSR it concatenates are built on its first call;
  * a pass captured on the pool (``SageTrainer.capture(pool, capacity=...)``)
    gathers each planned batch on the device inside its CUDA graph
    (``gte_gather_plan`` + ``gte_gather_pages``).
"""
from __future__ import annotations

from typing import List, Sequence

import numpy as np
import torch

from . import ops
from .graph import PageGraphBatch, batch_pages_host


class PagePool:
    """Every page of a dataset on one device, with page-local node ids: COO, edge weights, features, labels, the
    pages' node / edge offsets (int64) and their node / edge counts (host int64 ``n_i`` / ``e_i`` and device int32).
    ``batch(ids)`` assembles a ``PageGraphBatch`` eagerly; a ``SageTrainer`` pass captured on the pool
    (``capture(pool, capacity=...)``) gathers its batches from it inside the CUDA graph."""

    def __init__(self, pages: Sequence, device="cuda"):
        self.device = torch.device(device)
        dev = self.device
        self.num_pages = len(pages)
        self.n_i = np.array([p.num_nodes for p in pages], dtype=np.int64)
        self.e_i = np.array([int(p.src.shape[0]) for p in pages], dtype=np.int64)
        noff = np.zeros(self.num_pages + 1, dtype=np.int64)
        eoff = np.zeros(self.num_pages + 1, dtype=np.int64)
        np.cumsum(self.n_i, out=noff[1:])
        np.cumsum(self.e_i, out=eoff[1:])
        self.node_off = torch.from_numpy(noff).to(dev)
        self.edge_off = torch.from_numpy(eoff).to(dev)
        self.n_dev = torch.from_numpy(self.n_i.astype(np.int32)).to(dev)
        self.e_dev = torch.from_numpy(self.e_i.astype(np.int32)).to(dev)
        whole = PageGraphBatch.from_host(batch_pages_host(pages, pin=False), dev)
        src, dst = whole.edges()
        n_shift = self.node_off[self._edge_page()].to(torch.int32)
        self.coo = ((src - n_shift).contiguous(), (dst - n_shift).contiguous())
        self.w_coo = whole.edata["feat"]
        self.feat = whole.ndata["feat"]
        self.label = whole.ndata["label"]
        self._formats = None  # (csc, csr, w_csc, w_csr) of the whole pool, built by the first batch()

    @property
    def feat_width(self) -> int:
        return int(self.feat.shape[1])

    def _edge_page(self) -> torch.Tensor:
        """[E_pool]: the page that owns each edge"""
        return torch.repeat_interleave(torch.arange(self.num_pages, device=self.device), self.e_dev.long())

    def _sparse_formats(self):
        """CSC / CSR of every page with page-local ids and the weights in both orders: one GPU format build over the
        whole dataset, done on first use (only ``batch()`` needs them; they would triple the pool's footprint)"""
        if self._formats is None:
            dev = self.device
            P = self.num_pages
            edge_page = self._edge_page()
            n_shift = self.node_off[edge_page].to(torch.int32)
            whole = PageGraphBatch(self.coo[0] + n_shift, self.coo[1] + n_shift, int(self.n_i.sum()))
            slot_page = torch.repeat_interleave(torch.arange(P, device=dev), torch.from_numpy(self.n_i + 1).to(dev))
            slots = torch.arange(int(self.n_i.sum()) + P, device=dev)
            e_shift = self.edge_off[edge_page].to(torch.int32)

            def localise(fmt):
                indptr, indices, eid = fmt
                lp = (indptr[slots - slot_page] - self.edge_off[slot_page].to(torch.int32)).contiguous()
                return lp, (indices - n_shift).contiguous(), (eid - e_shift).contiguous()

            self._formats = (localise(whole.csc()), localise(whole.csr()), whole.weights_csc(self.w_coo),
                             whole.weights_csr(self.w_coo))
        return self._formats

    def batch(self, page_ids: Sequence[int]) -> PageGraphBatch:
        """``dgl.batch([pages[i] for i in page_ids])`` with CSC/CSR/weights ready."""
        dev = self.device
        csc, csr, w_csc, w_csr = self._sparse_formats()
        ids = np.asarray(page_ids, dtype=np.int64)
        bn = np.zeros(len(ids) + 1, dtype=np.int64)
        be = np.zeros(len(ids) + 1, dtype=np.int64)
        np.cumsum(self.n_i[ids], out=bn[1:])
        np.cumsum(self.e_i[ids], out=be[1:])
        n_tot, e_tot = int(bn[-1]), int(be[-1])
        meta = torch.from_numpy(np.concatenate([bn, be, ids])).to(dev, non_blocking=True)
        bno, beo = meta[: len(ids) + 1], meta[len(ids) + 1: 2 * len(ids) + 2]
        pid = meta[2 * len(ids) + 2:].to(torch.int32)

        def cat(fmt, w):
            return ops.batch_concat_csx(fmt[0], fmt[1], fmt[2], w, self.node_off, self.edge_off, pid, bno, beo, n_tot, e_tot)

        cp, ci, ce, cw = cat(csc, w_csc)
        rp, ri, re, rw = cat(csr, w_csr)
        _, src, _, w_coo = cat((csc[0], self.coo[0], None), self.w_coo)
        _, dst, _, _ = cat((csc[0], self.coo[1], None), None)
        g = PageGraphBatch(src, dst, n_tot, self.n_i[ids].tolist(), self.e_i[ids].tolist())
        g.edata["feat"] = w_coo
        g.set_formats(csc=(cp, ci, ce), csr=(rp, ri, re), w_csc=cw, w_csr=rw, w_src=w_coo)
        # node rows of the selected pages (device-side index arithmetic; features stay resident)
        page_of_node = torch.repeat_interleave(torch.arange(len(ids), device=dev), (bno[1:] - bno[:-1]),
                                               output_size=n_tot)
        node_idx = torch.arange(n_tot, device=dev) - bno[page_of_node] + self.node_off[pid.long()[page_of_node]]
        g.ndata["feat"] = self.feat.index_select(0, node_idx)
        g.ndata["label"] = self.label.index_select(0, node_idx)
        return g
