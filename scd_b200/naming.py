"""Image x vocabulary scoring, per-image top-k, per-cluster voting, name assignment and
re-assignment - the reference's inline naming code as functions over ``libscd_b200.so``.

Reference call sites (paths relative to the reference checkout):
  * scoring + top-k      ``main_unsup.py:504-531`` (softmax), ``main_ptsup.py:526-545`` (raw ``100*cos``)
  * whole-vocab argmax   ``main_ptsup.py:78-99`` ``get_clip_preds_fast``
  * top-k accuracy       ``local_utils/clip_lang_util.py:151-154`` ``accuracy``
  * vote                 ``main_unsup.py:572-586``, ``main_ptsup.py:636-648``
  * assign_name          ``local_utils/clip_lang_util.py:156-180`` (+ Hungarian ``gcd/project_utils/cluster_utils.py:234``)
  * re-assignment        ``main_unsup.py:601-614``, ``main_ptsup.py:668-676``
The de-facto signatures are kept: features ``[n, D]`` (tensor or ndarray) and ``zeroshot_weights [D, V]``
in, ``(values [n, k], indices [n, k] int64)`` / ``LongTensor[n]`` / ``(ind, w)`` out.

The contraction runs on the tcgen05 tensor cores in bf16 with fp32 accumulation (upstream CLIP on CUDA
is fp16 end to end): features and vocabulary are rounded to bf16 once, the N x V logits never reach HBM.
"""
from __future__ import annotations

import copy
import ctypes
from collections import Counter

import numpy as np
import torch

from . import _lib

SCALE = 100.0          # the reference's logit scale (``100. *``)


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError('scd_b200 needs a CUDA device (there is no CPU fallback)')


def _feats_bf16(feats) -> torch.Tensor:
    """[n, D] bf16 contiguous on the device (ndarray inputs are uploaded like ``main_unsup.py:522``)."""
    _require_cuda()
    if not torch.is_tensor(feats):
        feats = torch.from_numpy(np.ascontiguousarray(feats))
    feats = feats.to('cuda', non_blocking=True)
    if feats.dtype == torch.bfloat16:
        return feats.contiguous()
    f32 = feats.to(torch.float32).contiguous()
    out = torch.empty(f32.shape, dtype=torch.bfloat16, device=f32.device)
    if f32.numel():
        lib = _lib.load()
        _lib.check(lib.scd_cast_bf16(f32.data_ptr(), f32.numel(), out.data_ptr(), _stream()), 'scd_cast_bf16')
    return out


class Vocabulary:
    """``zeroshot_weights [D, V]`` (V contiguous, ``clip_lang_util.py:107``) re-laid out once as the K-major
    bf16 operand ``Wt [V, D]``.  ``col_offset`` is the global index of column 0 when this rank holds a
    column shard of a larger vocabulary (SURVEY 8e)."""

    def __init__(self, zeroshot_weights, col_offset: int = 0):
        _require_cuda()
        W = zeroshot_weights if torch.is_tensor(zeroshot_weights) else torch.from_numpy(np.asarray(zeroshot_weights))
        if W.dim() != 2:
            raise ValueError('zeroshot_weights must be [D, V]')
        W = W.to('cuda')
        if W.dtype not in (torch.float32, torch.bfloat16):
            W = W.to(torch.float32)
        if W.stride(1) != 1:
            W = W.contiguous()
        self.D, self.V = int(W.shape[0]), int(W.shape[1])
        self.col_offset = int(col_offset)
        self.Wt = torch.empty(self.V, self.D, dtype=torch.bfloat16, device=W.device)
        if self.V:
            lib = _lib.load()
            _lib.check(lib.scd_vocab_prepare(W.data_ptr(), int(W.dtype == torch.bfloat16), self.D, self.V, W.stride(0),
                                             self.Wt.data_ptr(), _stream()), 'scd_vocab_prepare')

    @classmethod
    def from_rows(cls, Wt: torch.Tensor, col_offset: int = 0):
        """Wrap an already K-major ``[V, D]`` bf16 tensor (e.g. gathered voted columns)."""
        self = cls.__new__(cls)
        self.Wt = Wt.contiguous()
        self.V, self.D = int(Wt.shape[0]), int(Wt.shape[1])
        self.col_offset = int(col_offset)
        return self

    def select(self, name_idx) -> 'Vocabulary':
        """The ``[D, K]`` stack of voted columns (``main_unsup.py:601-602``) as a K-row vocabulary."""
        sel = torch.as_tensor(np.asarray(name_idx, dtype=np.int64), device=self.Wt.device)
        out = torch.empty(sel.numel(), self.D, dtype=torch.bfloat16, device=self.Wt.device)
        if sel.numel():
            lib = _lib.load()
            _lib.check(lib.scd_gather_rows_bf16(self.Wt.data_ptr(), sel.data_ptr(), sel.numel(), self.D, self.V,
                                                out.data_ptr(), _stream()), 'scd_gather_rows_bf16')
        return Vocabulary.from_rows(out)


def _as_vocab(w) -> Vocabulary:
    return w if isinstance(w, Vocabulary) else Vocabulary(w)


class TopKPlan:
    """Outputs + workspace of the fused scoring/top-k launch for fixed ``(n, V, k)``: a hot loop (or a CUDA
    graph) re-launches without touching the allocator."""

    def __init__(self, n: int, v: int, k: int, device, want_stats: bool = False, idx_out: torch.Tensor | None = None):
        lib = _lib.load()
        self.n, self.v, self.k = int(n), int(v), int(k)
        self.vals = torch.empty(self.n, self.k, dtype=torch.float32, device=device)
        if idx_out is not None:            # write the indices straight into a caller-owned [n, k] int64 buffer
            assert idx_out.shape == (self.n, self.k) and idx_out.dtype == torch.int64 and idx_out.is_contiguous()
        self.idx = idx_out if idx_out is not None else torch.empty(self.n, self.k, dtype=torch.int64, device=device)
        self.rmax = torch.empty(self.n, dtype=torch.float32, device=device) if want_stats else None
        self.rsum = torch.empty(self.n, dtype=torch.float32, device=device) if want_stats else None
        self.ws = torch.empty(lib.scd_name_topk_workspace_bytes(self.n, self.v, self.k) if self.n else 256,
                              dtype=torch.uint8, device=device)

    def run(self, feats_bf16: torch.Tensor, vocab: 'Vocabulary', softmax: bool, scale: float = SCALE):
        if int(feats_bf16.shape[0]) != self.n or vocab.V != self.v:
            raise ValueError('TopKPlan was built for a different shape')
        if self.n == 0:
            return self.vals, self.idx, self.rmax, self.rsum
        if int(feats_bf16.shape[1]) != vocab.D:
            raise ValueError(f'feature width {int(feats_bf16.shape[1])} != vocabulary width {vocab.D}')
        lib = _lib.load()
        _lib.check(lib.scd_name_topk(feats_bf16.data_ptr(), self.n, vocab.D, vocab.Wt.data_ptr(), vocab.V, float(scale), self.k,
                                     int(bool(softmax)), vocab.col_offset, self.vals.data_ptr(), self.idx.data_ptr(),
                                     _lib.ptr(self.rmax), _lib.ptr(self.rsum), self.ws.data_ptr(), self.ws.numel(), _stream()),
                   'scd_name_topk')
        return self.vals, self.idx, self.rmax, self.rsum


def name_topk_raw(feats_bf16: torch.Tensor, vocab: Vocabulary, k: int, softmax: bool, scale: float = SCALE,
                  want_stats: bool = False, plan: TopKPlan | None = None):
    """One launch of the fused scoring/top-k kernel on device-resident operands."""
    if plan is None:
        plan = TopKPlan(int(feats_bf16.shape[0]), vocab.V, k, feats_bf16.device, want_stats)
    return plan.run(feats_bf16, vocab, softmax, scale)


def score_topk(feats, zeroshot_weights, k: int = 5, softmax: bool = False, scale: float = SCALE):
    """``logits = 100. * feats @ zeroshot_weights`` [+ ``F.softmax``] ``.topk(k, 1, True, True)``
    (``main_unsup.py:519-529`` with ``softmax=True``; ``main_ptsup.py:538-543`` with ``softmax=False``).
    Returns ``(values [n,k] fp32, indices [n,k] int64)``, largest first, ties -> lower index."""
    vocab = _as_vocab(zeroshot_weights)
    if not torch.is_tensor(feats):
        feats = torch.from_numpy(np.ascontiguousarray(feats))
    if not feats.is_cuda and feats.dim() == 2 and int(feats.shape[0]) >= 2 * STREAM_ROWS and feats.dtype == torch.float32:
        return _score_topk_streamed(feats, vocab, k, softmax, scale)
    vals, idx, _, _ = name_topk_raw(_feats_bf16(feats), vocab, k, softmax, scale)
    return vals, idx


STREAM_ROWS = 74 * 256         # one full wave of 256-row blocks over the 74 CTA pairs of a B200


def _score_topk_streamed(feats_host: torch.Tensor, vocab: Vocabulary, k: int, softmax: bool, scale: float):
    """HOST features (the reference's ``clip_all_feats`` is a NumPy array uploaded per 1024-row batch,
    ``main_unsup.py:522``): upload in wave-sized row chunks on a copy stream while the previous chunk is cast and
    scored on the caller's stream, so the PCIe transfer (the bound: 390 MB against 2.8 ms of tensor-core work at C2)
    hides the kernel instead of preceding it.  Rows are independent, so the per-chunk results are the final rows."""
    _require_cuda()
    lib = _lib.load()
    n, d = int(feats_host.shape[0]), int(feats_host.shape[1])
    if d != vocab.D:
        raise ValueError(f'feature width {d} != vocabulary width {vocab.D}')
    feats_host = feats_host.contiguous()
    dev = vocab.Wt.device
    vals = torch.empty(n, k, dtype=torch.float32, device=dev)
    idx = torch.empty(n, k, dtype=torch.int64, device=dev)
    main = torch.cuda.current_stream()
    copy = _lib.upload_stream(dev)
    with torch.cuda.stream(copy):                    # allocated under the upload stream: chunk 0 does not wait for `main`
        stage = [torch.empty(STREAM_ROWS, d, dtype=torch.float32, device=dev) for _ in range(2)]
    half = [torch.empty(STREAM_ROWS, d, dtype=torch.bfloat16, device=dev) for _ in range(2)]
    uploaded = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    plans = {}
    for c, lo in enumerate(range(0, n, STREAM_ROWS)):
        rows = min(STREAM_ROWS, n - lo)
        b = c & 1
        with torch.cuda.stream(copy):
            if c >= 2:
                copy.wait_event(consumed[b])                       # the cast of chunk c-2 has read this staging buffer
            stage[b][:rows].copy_(feats_host[lo:lo + rows], non_blocking=True)
            uploaded[b].record(copy)
        main.wait_event(uploaded[b])
        _lib.check(lib.scd_cast_bf16(stage[b].data_ptr(), rows * d, half[b].data_ptr(), main.cuda_stream), 'scd_cast_bf16')
        consumed[b].record(main)
        if rows not in plans:
            plans[rows] = torch.empty(lib.scd_name_topk_workspace_bytes(rows, vocab.V, k), dtype=torch.uint8, device=dev)
        ws = plans[rows]
        # half[b] is reused by chunk c+2 only after this launch: same stream, program order
        _lib.check(lib.scd_name_topk(half[b].data_ptr(), rows, d, vocab.Wt.data_ptr(), vocab.V, float(scale), int(k),
                                     int(bool(softmax)), vocab.col_offset, vals[lo:lo + rows].data_ptr(),
                                     idx[lo:lo + rows].data_ptr(), None, None, ws.data_ptr(), ws.numel(), main.cuda_stream),
                   'scd_name_topk')
    for t in stage:
        t.record_stream(main)
    return vals, idx


def clip_preds(feats, zeroshot_weights) -> torch.Tensor:
    """``get_clip_preds_fast`` (``main_ptsup.py:78-99``) without the target bookkeeping: ``argmax`` over the
    whole vocabulary, ``LongTensor[n]`` on the device."""
    _, idx = score_topk(feats, zeroshot_weights, k=1)
    return idx.view(-1)


def accuracy(feats, zeroshot_weights, target, topk=(1,)):
    """``accuracy(100. * feats @ W, target, topk)`` (``clip_lang_util.py:151-154``; used by
    ``evaluate_semantic_acc_ub_lb`` ``main_ptsup.py:116-120``): number of rows whose target is in the top-k."""
    _, idx = score_topk(feats, zeroshot_weights, k=max(topk))
    tgt = torch.as_tensor(target, device=idx.device).view(-1, 1)
    hit = idx.eq(tgt)
    return [float(hit[:, :kk].any(dim=1).sum().item()) for kk in topk]


def reassign(feats, zeroshot_weights, cand_name_idx) -> np.ndarray:
    """``argmax(100. * feats @ W[:, cand], -1)`` -> NumPy int64 (``main_unsup.py:601-614`` /
    ``main_ptsup.py:668-676``); positions index ``cand_name_idx``."""
    vocab = _as_vocab(zeroshot_weights)
    sel = vocab.select(cand_name_idx)
    _, idx = score_topk(feats, sel, k=1)
    return idx.view(-1).cpu().numpy()


# ----------------------------------------------------------------------------------------- voting
class VotePlan:
    """Outputs + workspace of the device vote for fixed ``(n, K, M)``.  ``k_used`` sizes the global-memory spill
    tables that clusters with more than 8192 top-k entries build their name histogram in (24 bytes per entry; any
    cluster fits, there is no distinct-name limit); it is only allocated when such a cluster can exist."""

    def __init__(self, n: int, n_clusters: int, num_common: int, device, k_used: int = 5):
        lib = _lib.load()
        self.n, self.K, self.M, self.k_used = int(n), int(n_clusters), int(num_common), int(k_used)
        self.names = torch.empty(self.K, self.M, dtype=torch.int64, device=device)
        self.counts = torch.empty(self.K, self.M, dtype=torch.int32, device=device)
        self.distinct = torch.empty(self.K, dtype=torch.int32, device=device)
        self.rows = torch.empty(self.K, dtype=torch.int32, device=device)
        self.overflow = torch.zeros(1, dtype=torch.int32, device=device)
        self.ws = torch.zeros(lib.scd_vote_workspace_bytes(self.n, self.K), dtype=torch.uint8, device=device)
        self.spill = None
        if self.n * self.k_used > 8192:
            self.spill = torch.empty(lib.scd_vote_spill_bytes(self.n, self.k_used), dtype=torch.uint8, device=device)

    def spill_args(self):
        return (_lib.ptr(self.spill), 0 if self.spill is None else self.spill.numel())


def _vote_plan(plan, n: int, K: int, M: int, k_used: int, device, n_at_least: bool = False) -> VotePlan:
    """``plan`` checked against the vote's shape (``n_at_least``: any ``plan.n >= n``), or a new one when it is None."""
    if plan is None:
        return VotePlan(n, K, M, device, k_used=k_used)
    if (plan.K, plan.M) != (K, M) or plan.k_used < k_used or (plan.n < n if n_at_least else plan.n != n):
        raise ValueError('VotePlan was built for a different shape')
    return plan


def _excluded(known_name_idx, device):
    """``(int64 device tensor, count)`` of the names the vote skips; ``(None, 0)`` when there are none."""
    if known_name_idx is None or not len(known_name_idx):
        return None, 0
    excl = torch.as_tensor(np.asarray(list(known_name_idx), dtype=np.int64), device=device)
    return excl, int(excl.numel())


def vote_device(name_idx_topk: torch.Tensor, cluster_of_row, n_clusters: int, top_k: int, num_common: int,
                known_name_idx=None, plan: VotePlan | None = None, presorted=None):
    """Device vote: per cluster the ``num_common`` most common names of ``name_idx_topk[rows, :top_k]``
    (Python ``Counter.most_common`` order).  Returns device tensors
    ``(names [K,M] int64 (-1 padded), counts [K,M] int32, distinct [K] int32, rows [K] int32, overflow [1])``.

    ``presorted``: a ``kmeans._MStep`` whose ``sums_counts(X, labels)`` has just run on these very labels (the
    k-means labels are what ``main_unsup.py:575`` votes with) - its label sort is reused instead of repeated."""
    _require_cuda()
    idx = name_idx_topk
    if not (torch.is_tensor(idx) and idx.is_cuda and idx.dtype == torch.int64 and idx.is_contiguous()):
        idx = torch.as_tensor(idx).to('cuda').to(torch.int64).contiguous()
    n, kt = int(idx.shape[0]), int(idx.shape[1])
    dev = idx.device
    K, M = int(n_clusters), int(num_common)
    plan = _vote_plan(plan, n, K, M, int(top_k), dev)
    excl, n_excl = _excluded(known_name_idx, dev)
    lib = _lib.load()
    if presorted is not None:
        if (presorted.n, presorted.k) != (n, K):
            raise ValueError('presorted M-step does not match the vote shape')
        _lib.check(lib.scd_vote_presorted(idx.data_ptr(), kt, int(top_k), presorted.ws.data_ptr(), n, K, _lib.ptr(excl), n_excl, M,
                                          plan.names.data_ptr(), plan.counts.data_ptr(), plan.distinct.data_ptr(),
                                          plan.overflow.data_ptr(), *plan.spill_args(), _stream()), 'scd_vote_presorted')
        return plan.names, plan.counts, plan.distinct, presorted.counts, plan.overflow
    cl = cluster_of_row
    if not (torch.is_tensor(cl) and cl.is_cuda and cl.dtype == torch.int64 and cl.is_contiguous()):
        cl = torch.as_tensor(cl).to('cuda').to(torch.int64).contiguous()
    _lib.check(lib.scd_vote(idx.data_ptr(), kt, int(top_k), cl.data_ptr(), n, K, _lib.ptr(excl), n_excl, M, plan.names.data_ptr(),
                            plan.counts.data_ptr(), plan.distinct.data_ptr(), plan.rows.data_ptr(), plan.overflow.data_ptr(),
                            plan.ws.data_ptr(), plan.ws.numel(), *plan.spill_args(), _stream()), 'scd_vote')
    return plan.names, plan.counts, plan.distinct, plan.rows, plan.overflow


def pack_vote_records(labels: torch.Tensor, name_idx_topk: torch.Tensor, top_k: int, out: torch.Tensor | None = None):
    """``[n, 1 + top_k]`` int32 records ``[label, name_0 .. name_(top_k-1)]`` - what a rank contributes to the ONE
    all-gather of the row-sharded vote (SURVEY 8e)."""
    n, kt = int(name_idx_topk.shape[0]), int(name_idx_topk.shape[1])
    if out is None:
        out = torch.empty(n, 1 + int(top_k), dtype=torch.int32, device=name_idx_topk.device)
    lib = _lib.load()
    _lib.check(lib.scd_pack_vote_records(labels.data_ptr(), name_idx_topk.data_ptr(), kt, int(top_k), n, out.data_ptr(), _stream()),
               'scd_pack_vote_records')
    return out


def vote_records(records: torch.Tensor, n_clusters: int, num_common: int, known_name_idx=None, plan: VotePlan | None = None):
    """The vote over gathered ``[N, 1 + top_k]`` int32 records (see ``pack_vote_records``); same outputs as ``vote_device``."""
    n, top_k = int(records.shape[0]), int(records.shape[1]) - 1
    K, M = int(n_clusters), int(num_common)
    plan = _vote_plan(plan, n, K, M, top_k, records.device)
    excl, n_excl = _excluded(known_name_idx, records.device)
    lib = _lib.load()
    _lib.check(lib.scd_vote_records(records.data_ptr(), top_k, n, K, _lib.ptr(excl), n_excl, M,
                                    plan.names.data_ptr(), plan.counts.data_ptr(), plan.distinct.data_ptr(), plan.rows.data_ptr(),
                                    plan.overflow.data_ptr(), plan.ws.data_ptr(), plan.ws.numel(), *plan.spill_args(), _stream()),
               'scd_vote_records')
    return plan.names, plan.counts, plan.distinct, plan.rows, plan.overflow


def vote_segments(records: torch.Tensor, seg_offsets: torch.Tensor, n_clusters: int, num_common: int, known_name_idx=None,
                  plan: VotePlan | None = None, n_total: int | None = None):
    """The vote over gathered SORTED-RUN records (``peer.PeerExchange.gather_sorted_records``): ``records``
    ``[world * per, 1 + top_k]`` int32 = ``[global row id, names]`` in each rank's label-sorted order, ``seg_offsets``
    ``[world, K + 1]`` the ranks' offsets.  No sort of the gathered rows; same outputs as ``vote_device``."""
    world, per = int(seg_offsets.shape[0]), int(records.shape[0]) // int(seg_offsets.shape[0])
    top_k = int(records.shape[1]) - 1
    K, M = int(n_clusters), int(num_common)
    n_total = world * per if n_total is None else int(n_total)
    plan = _vote_plan(plan, n_total, K, M, top_k, records.device, n_at_least=True)
    excl, n_excl = _excluded(known_name_idx, records.device)
    lib = _lib.load()
    _lib.check(lib.scd_vote_segments(records.data_ptr(), top_k, n_total, per, world, seg_offsets.data_ptr(), K, _lib.ptr(excl),
                                     n_excl, M, plan.names.data_ptr(), plan.counts.data_ptr(),
                                     plan.distinct.data_ptr(), plan.rows.data_ptr(), plan.overflow.data_ptr(), *plan.spill_args(), _stream()),
               'scd_vote_segments')
    return plan.names, plan.counts, plan.distinct, plan.rows, plan.overflow


def vote(name_idx_topk, u_preds, cluster_ids, top_k: int, num_common: int, known_name_idx=None):
    """``cluster_to_counter`` of ``main_unsup.py:575-577`` / ``main_ptsup.py:636-638``, truncated to each
    cluster's ``num_common`` most common names (all the loop ever reads: ``most_common(num_common_vote)``
    :582 and ``most_common(num_common)`` in ``assign_name`` with ``num_common <= num_common_vote``).
    Counters are built in most-common order, so ``Counter.most_common(m)`` returns exactly what the
    reference's full Counter returns for any ``m <= num_common``."""
    cluster_ids = [int(c) for c in cluster_ids]
    K = (max(cluster_ids) + 1) if cluster_ids else 1
    preds = np.asarray(u_preds)
    if preds.size and (preds.max() >= K):
        K = int(preds.max()) + 1
    names, counts, _, _, overflow = vote_device(name_idx_topk, preds, K, top_k, num_common, known_name_idx)
    names_h, counts_h, ovf = names.cpu().numpy(), counts.cpu().numpy(), int(overflow.item())
    if ovf:                 # cannot happen with the spill tables VotePlan allocates; kept as a guard for raw-ABI callers
        raise RuntimeError('scd_vote: a cluster exhausted the shared-memory name table and no spill buffer was given')
    out = {}
    for c in cluster_ids:
        ctr = Counter()
        for name, cnt in zip(names_h[c], counts_h[c]):
            if name < 0:
                break
            ctr[np.int64(name)] = int(cnt)
        out[c] = ctr
    return out


def voted_candidates(cluster_to_counter, cluster_ids, num_common_vote: int):
    """``main_unsup.py:579-586``: union of the clusters' ``most_common(num_common_vote)`` names in CPython
    ``list(set(...))`` order (that order fixes the columns of ``w`` and so the Hungarian tie-breaks)."""
    names = []
    for i in cluster_ids:
        for name, _cnt in cluster_to_counter[i].most_common(num_common_vote):
            names += [name]
    return list(set(names))


def linear_assignment(cost) -> np.ndarray:
    """``gcd/project_utils/cluster_utils.py:234``: Munkres with the reference's tie-breaking (host C++)."""
    cost = np.ascontiguousarray(np.atleast_2d(cost), dtype=np.int64)
    r, c = cost.shape
    out = np.zeros((min(r, c), 2), dtype=np.int64)
    n = ctypes.c_int(0)
    lib = _lib.load()
    rc = lib.scd_linear_assignment(cost.ctypes.data, r, c, out.ctypes.data, ctypes.byref(n))
    if rc != 0:
        raise RuntimeError('scd_linear_assignment failed')
    return out[:n.value].astype(int)


def assign_name(unique_name_idx, cluster_to_counter, num_common=4):
    """``local_utils/clip_lang_util.py:156-180`` - same signature and return ``(ind, w)``."""
    col_of = {name: j for j, name in enumerate(unique_name_idx)}
    clusters = list(cluster_to_counter.keys())
    dim = max(len(unique_name_idx), len(clusters))
    w = np.zeros((dim, dim), dtype=int)
    for row, cid in enumerate(clusters):
        for name, cnt in cluster_to_counter[cid].most_common(num_common):
            w[row, col_of[name]] += cnt
    ind = linear_assignment(w.max() - w)
    return ind, w


def naming_loop_unsup(name_idx_topk, u_preds, clip_u_feats, zeroshot_weights, n_cluster, top_k=5,
                      num_common_vote=20, num_common_linear=4, max_rounds=50):
    """The iterative voting loop of ``main_unsup.py:568-614`` (names are vocabulary indices).  Returns the
    per-round trace ``[{voted, u_preds, n_unique}]``; the last entry is the converged naming."""
    vocab = _as_vocab(zeroshot_weights)
    feats = _feats_bf16(clip_u_feats)
    u_preds = np.asarray(u_preds)
    cur, prev, trace = [-1], [-2], []
    while set(cur) != set(prev) and len(trace) < max_rounds:
        cluster_ids = list(set(u_preds))                                            # :573
        c2c = vote(name_idx_topk, u_preds, cluster_ids, top_k, num_common_vote)     # :575-577
        uniq = voted_candidates(c2c, cluster_ids, num_common_vote)                  # :579-586
        ind, _w = assign_name(uniq, c2c, num_common=num_common_linear)              # :588
        prev = copy.deepcopy(cur)
        cur = [int(uniq[x[1]]) for x in ind[:n_cluster]]                            # :594
        u_preds = reassign(feats, vocab, cur)                                       # :601-614
        trace.append(dict(voted=list(cur), u_preds=u_preds.copy(), n_unique=len(uniq)))
    return trace


def naming_loop_ptsup(name_idx_topk, all_preds, mask_lab, clip_u_feats, zeroshot_weights, lab_name_idx, n_cluster,
                      top_k=5, num_common_vote=20, num_common_linear=4, max_rounds=50, nouns=None):
    """``main_ptsup.py:588-676`` including its index-space quirk (from round 2 ``unlab_cluster_idx`` /
    ``known_name_idx`` are positions in ``cand_names`` while ``name_idx_topk`` holds vocabulary indices).

    ``nouns`` (optional, the vocabulary's name strings in column order): the bookkeeping then runs on the strings like
    the reference - ``sorted(cand_names)`` :659 is lexicographic (it fixes ``lab_class_index``, the numbering of the
    re-assigned clusters and the row order of the Hungarian matrix), ``nouns.index`` :601 / :669 maps duplicate names
    to their first column, the loop ends when the SET OF NAMES stops changing, and :664's
    ``list(set(cand_names) - set(lab_names))`` takes the string-set order of the running interpreter (hash-seed
    dependent in the reference too).  Without ``nouns`` a name is its column index - equivalent whenever the
    vocabulary list is duplicate-free and in lexicographic order.  ``voted`` / ``cand`` in the trace are names."""
    vocab = _as_vocab(zeroshot_weights)
    feats = _feats_bf16(clip_u_feats)
    all_preds, mask_lab = np.asarray(all_preds), np.asarray(mask_lab)
    u_preds, l_preds = all_preds[~mask_lab], all_preds[mask_lab]                    # :592-593
    if nouns is None:
        name_of, index_of = (lambda i: i), (lambda s: s)
    else:
        first = {}
        for i, s in enumerate(nouns):
            first.setdefault(s, i)
        name_of, index_of = (lambda i: nouns[i]), (lambda s: first[s])              # nouns.index(s)
    lab_names = [name_of(int(i)) for i in lab_name_idx]                             # :598
    num_unlab = n_cluster - len(lab_names)                                          # :602
    known = [index_of(s) for s in lab_names]                                        # :603
    unlab_clusters = list(set(set(all_preds)) - set(l_preds))                       # :625
    cur, prev, trace = [-1], [-2], []
    while set(cur) != set(prev) and len(trace) < max_rounds:
        c2c = vote(name_idx_topk, u_preds, unlab_clusters, top_k, num_common_vote, known_name_idx=known)   # :636-638
        uniq = voted_candidates(c2c, unlab_clusters, num_common_vote)               # :640-648
        ind, _w = assign_name(uniq, c2c, num_common=num_common_linear)              # :649
        prev = copy.deepcopy(cur)
        cur = [name_of(int(uniq[x[1]])) for x in ind[:num_unlab]]                   # :655
        cand = sorted(set(cur + lab_names))                                         # :657-659
        lab_class_index = [cand.index(n) for n in lab_names]                        # :662
        unlab_clusters = [cand.index(n) for n in list(set(cand) - set(lab_names))]  # :664
        known = copy.deepcopy(lab_class_index)                                      # :666
        u_preds = reassign(feats, vocab, [index_of(s) for s in cand])               # :668-676
        trace.append(dict(voted=list(cur), cand=list(cand), u_preds=u_preds.copy(), n_unique=len(uniq)))
    return trace
