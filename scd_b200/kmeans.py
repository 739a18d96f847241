"""Drop-in (semi-supervised) k-means: the reference's ``K_Means`` / ``pairwise_distance`` signatures
over the sm_100a kernels in ``libscd_b200.so``.

Mirrors ``local_utils/faster_mix_k_means_pytorch.py`` (``K_Means`` :8, ``kpp`` :20, ``fit_once`` :39,
``fit_mix_once`` :77, ``fit`` :129, ``fit_mix`` :153, ``pairwise_distance`` :177) and the copy the drivers
import, ``gcd/methods/clustering/faster_mix_k_means_pytorch.py`` (adds ``mode=`` :49-59).  Same
constructor arguments, methods, result attributes and quirks (labelled rows first in ``labels_``,
``n_iter_ == len(l_targets)`` after ``fit_mix``, post-update centres paired with pre-update labels,
NaN centroid for an empty cluster).  All arithmetic runs on the GPU; inputs on the CPU are moved to
the current CUDA device and results are returned on the input's device.  No CPU fallback.

Sharded use (rows of ``X`` / ``u_feats`` block-sharded over the ranks of a ``torch.distributed``
process group, one process per GPU): pass ``process_group=`` - the M-step then all-reduces one packed
``[K*D sums | K counts | inertia]`` fp32 buffer per iteration over NCCL (SURVEY 8e).  Everything that
decides the result is made identical on every rank: the host RNG is re-seeded from a seed rank 0 draws and
broadcasts, k-means++ draws over the GLOBAL distance mass (all-gathered shard sums pick the owning rank, which
resolves the row on its device and broadcasts it), the 'random' / first-k initialisations take GLOBAL row
indices, and the labelled rows of ``fit_mix`` (``l_feats`` / ``l_targets`` are REPLICATED on every rank) enter
the all-reduced sums once, through rank 0.  ``labels_`` holds the labels of the rank's own rows.
"""
from __future__ import annotations

import numpy as np
import torch
from sklearn.utils import check_random_state

from . import _lib


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dev_f32(t: torch.Tensor) -> torch.Tensor:
    """fp32, contiguous, on the current CUDA device (the reference feeds fp32 CUDA tensors, main_unsup.py:340)."""
    if not torch.cuda.is_available():
        raise RuntimeError('scd_b200 needs a CUDA device (there is no CPU fallback)')
    if not torch.is_tensor(t):
        t = torch.as_tensor(t)
    return t.to(device='cuda', dtype=torch.float32).contiguous()


# ----------------------------------------------------------------------------- thin kernel wrappers
class _EStep:
    """Workspace of the tensor-core E-step for a fixed ``(K, D)``: the centroid hi / lo planes and norms.  One per
    fit (or per cached ``(K, D, device, stream)``), never shared between streams.  ``ready_for`` remembers the
    centre tensor whose operands ``_MStep.finalize(estep=...)`` has already left in the workspace."""

    def __init__(self, k, d, device):
        lib = _lib.load()
        self.k, self.d = int(k), int(d)
        self.ws = torch.empty(lib.scd_estep_workspace_bytes(self.k, self.d), dtype=torch.uint8, device=device)
        self.ready_for = None

    def fusable(self, n):
        """Always False: the one-pass E+M kernel was removed (DESIGN 3.3).  Kept for ``bench.py --fused-em``, its only
        caller, which then runs the two-pass round."""
        return False

    def run(self, X, C, labels_out, inertia_acc, mindist=None, exact=False):
        lib = _lib.load()
        flags = _lib.ESTEP_EXACT if exact else 0
        if self.ready_for is not None and self.ready_for == C.data_ptr():
            flags |= _lib.ESTEP_PLANES_READY
        self.ready_for = None
        _lib.check(lib.scd_estep(X.data_ptr(), X.shape[0], X.shape[1], C.data_ptr(), C.shape[0],
                                 labels_out.data_ptr(), _lib.ptr(mindist), _lib.ptr(inertia_acc), flags,
                                 self.ws.data_ptr(), self.ws.numel(), _stream()), 'scd_estep')


_ESTEP_WS = {}


def _estep(X, C, labels_out, inertia_acc, mindist=None, exact=False):
    """One-off E-step (predict, seeding, tests): workspace cached per (K, D, device, stream)."""
    key = (int(C.shape[0]), int(C.shape[1]), X.device.index, _stream())
    es = _ESTEP_WS.get(key)
    if es is None:
        if len(_ESTEP_WS) > 64:
            _ESTEP_WS.clear()
        es = _ESTEP_WS[key] = _EStep(key[0], key[1], X.device)
    es.ready_for = None
    es.run(X, C, labels_out, inertia_acc, mindist, exact)


class _MStep:
    """Workspace + launches of the M-step for a fixed (N, D, K)."""

    def __init__(self, n, d, k, device, ws=None):
        lib = _lib.load()
        self.n, self.d, self.k = n, d, k
        self.ws = ws if ws is not None else torch.zeros(lib.scd_mstep_workspace_bytes(n, k), dtype=torch.uint8, device=device)
        # one buffer [K*D sums | K counts | inertia] (fp32) so the row-sharded case all-reduces it in one call
        self.packed = torch.zeros(k * d + k + 1, dtype=torch.float32, device=device)
        self.sums = self.packed[:k * d].view(k, d)
        self.counts_f = self.packed[k * d:k * d + k]
        self.counts = torch.empty(k, dtype=torch.int32, device=device)
        self.peer = None                                  # (PeerExchange, block) while the sums live in a peer-mapped block
        self.norms = torch.zeros(max(k, 1), dtype=torch.float32, device=device)     # ||c_new[k] - c_old[k]||
        self.shift = torch.zeros(1, dtype=torch.float32, device=device)
        self.tc = bool(lib.scd_estep_uses_tensor_cores(max(n, 1), d, k))

    def bind_peer(self, px, block):
        """Let the segment sum write straight into this rank's block of a ``peer.PeerExchange`` (sums, counts, inertia)."""
        self.peer = (px, block)
        self.sums, self.counts = block[0], block[1]

    def sums_counts(self, X, labels):
        lib = _lib.load()
        _lib.check(lib.scd_mstep_sums(X.data_ptr(), labels.data_ptr(), self.n, self.d, self.k, self.sums.data_ptr(),
                                      self.counts.data_ptr(), self.ws.data_ptr(), self.ws.numel(), _stream()), 'scd_mstep_sums')

    def finalize_peer(self, c_old, c_new, inertia_out, estep: '_EStep | None' = None):
        """The row-sharded M-step's all-reduce + divide in one launch over peer memory (``scd_finalize_centers_peer``);
        the reduced inertia lands in ``inertia_out``, the reduced counts in ``counts_f``, move norms in ``norms``."""
        px, block = self.peer
        px.finalize(block, c_old, c_new, self.norms, self.counts_f, inertia_out, estep)

    def finalize(self, c_old, c_new, counts_f=None, estep: '_EStep | None' = None, shift=True):
        """divide (+ per-cluster move norms when ``c_old`` is given; ``shift=True`` also sums them on the device into
        ``self.shift``).  ``estep``: leave the next E-step's operands of ``c_new`` in that plan's workspace."""
        lib = _lib.load()
        want_shift = shift and c_old is not None
        _lib.check(lib.scd_finalize_centers(self.sums.data_ptr(), None if counts_f is not None else self.counts.data_ptr(),
                                            _lib.ptr(counts_f), _lib.ptr(c_old), c_new.data_ptr(),
                                            self.shift.data_ptr() if want_shift else None, self.k, self.d,
                                            self.norms.data_ptr(), self.norms.numel() * 4,
                                            estep.ws.data_ptr() if estep is not None else None,
                                            estep.ws.numel() if estep is not None else 0, _stream()), 'scd_finalize_centers')
        if estep is not None:
            estep.ready_for = c_new.data_ptr()


PANEL_ROWS = 16384          # rows per upload panel of assign_from_host (50 MB of fp32 at D = 768: ~0.9 ms of PCIe, ~12 us of E-step)


def assign_from_host(X_host: torch.Tensor, centers: torch.Tensor, panel_rows: int = PANEL_ROWS, mstep=None):
    """E-step of one iteration (``faster_mix_k_means_pytorch.py:58-60``) on HOST features: ``torch.from_numpy(x).cuda()``
    (``main_unsup.py:340``) and the assignment pipelined - the rows go up in panels on a copy stream and each panel is
    assigned (fused distance + argmin + inertia) while the next one is on the wire, so only the last panel's ~12 us of
    E-step are left after the transfer.  Rows are independent: labels equal the resident launch bit for bit.
    ``mstep`` must be None: the one-pass E+M that accumulated the M-step's sums per panel was removed (DESIGN 3.3).
    Returns ``(X on the device, labels int64 [N], inertia fp64 [1])``."""
    if mstep is not None:
        raise ValueError('assign_from_host: mstep= must be None - the one-pass E+M was removed (DESIGN 3.3)')
    if not torch.is_tensor(X_host):
        X_host = torch.from_numpy(np.ascontiguousarray(X_host))
    if X_host.is_cuda or X_host.dtype != torch.float32 or X_host.dim() != 2:
        raise ValueError('assign_from_host expects a 2-D float32 host tensor')
    X_host = X_host.contiguous()
    Cd = _dev_f32(centers)
    dev = Cd.device
    n, d = int(X_host.shape[0]), int(X_host.shape[1])
    labels = torch.empty(n, dtype=torch.int64, device=dev)
    inertia = torch.zeros(1, dtype=torch.float64, device=dev)
    es = _EStep(int(Cd.shape[0]), d, dev)
    main = torch.cuda.current_stream()
    copy = _lib.upload_stream(dev)
    with torch.cuda.stream(copy):                    # allocated under the upload stream: the first panel does not wait for `main`
        X = torch.empty(n, d, dtype=torch.float32, device=dev)
    for lo in range(0, n, panel_rows):
        hi = min(lo + panel_rows, n)
        with torch.cuda.stream(copy):
            X[lo:hi].copy_(X_host[lo:hi], non_blocking=True)
            up = torch.cuda.Event()
            up.record(copy)
        main.wait_event(up)
        if lo:
            es.ready_for = Cd.data_ptr()             # the centroid planes of the first panel's launch are still in place
        es.run(X[lo:hi], Cd, labels[lo:hi], inertia)
    X.record_stream(main)
    return X, labels, inertia


def update_centers(X: torch.Tensor, labels: torch.Tensor, k: int, c_old: torch.Tensor | None = None, mstep: '_MStep | None' = None):
    """M-step (``faster_mix_k_means_pytorch.py:61-64``): ``centers[j] = mean(X[labels == j])`` on device-resident rows,
    NaN row for an empty cluster.  ``mstep``: an ``_MStep`` whose ``sums_counts`` has already run on ``(X, labels)`` -
    only the divide is left.  Returns ``(centers [K, D], counts int32 [K], move norms or None, the _MStep)``."""
    Xd = _dev_f32(X)
    ms = mstep
    if ms is None:
        ms = _MStep(int(Xd.shape[0]), int(Xd.shape[1]), int(k), Xd.device)
        ms.sums_counts(Xd, labels)
    c_new = torch.empty(int(k), int(Xd.shape[1]), dtype=torch.float32, device=Xd.device)
    ms.finalize(c_old, c_new, shift=False)
    return c_new, ms.counts, (ms.norms if c_old is not None else None), ms


def pairwise_distance(data1, data2, batch_size=None, *, out_device=None):
    """Reference signature (``local_utils/faster_mix_k_means_pytorch.py:177``): squared Euclidean distance
    matrix ``[N, K]``, direct form, fp32.  Like the reference, the result lives on the **CPU** when
    ``batch_size`` is given (its buffer is ``torch.zeros(N, K)``, :197) and on the input's device
    otherwise; ``out_device`` (extension) overrides that.  ``batch_size`` itself is irrelevant here: the
    kernel tiles internally and never materialises the ``B x K x D`` temporary."""
    src_device = data1.device if torch.is_tensor(data1) else torch.device('cpu')
    X, Cm = _dev_f32(data1), _dev_f32(data2)
    if X.dim() != 2 or Cm.dim() != 2 or X.shape[1] != Cm.shape[1]:
        raise ValueError(f'pairwise_distance expects [N,D] and [K,D], got {tuple(X.shape)} and {tuple(Cm.shape)}')
    out = torch.empty(X.shape[0], Cm.shape[0], dtype=torch.float32, device=X.device)
    if X.shape[0] and Cm.shape[0]:
        lib = _lib.load()
        _lib.check(lib.scd_pairwise_distance(X.data_ptr(), X.shape[0], X.shape[1], Cm.data_ptr(), Cm.shape[0],
                                             out.data_ptr(), None, _stream()), 'scd_pairwise_distance')
    target = out_device if out_device is not None else (torch.device('cpu') if batch_size is not None else src_device)
    return out.to(target)


def constrained_int_costs(data1, data2):
    """int32 ``round(1000 * sqrt(dist))`` cost matrix the size-constrained variant hands to its flow solver
    (``local_utils/sskm_constrained.py:116`` + ``:324``), produced directly by the distance kernel."""
    X, Cm = _dev_f32(data1), _dev_f32(data2)
    out = torch.empty(X.shape[0], Cm.shape[0], dtype=torch.int32, device=X.device)
    if X.shape[0] and Cm.shape[0]:
        lib = _lib.load()
        _lib.check(lib.scd_pairwise_distance(X.data_ptr(), X.shape[0], X.shape[1], Cm.data_ptr(), Cm.shape[0],
                                             None, out.data_ptr(), _stream()), 'scd_pairwise_distance')
    return out


def predict(X, cluster_centers, batch_size=None):
    """The reference has no ``K_Means.predict``; its predict-equivalent is
    ``pairwise_distance(X, centers, bs).argmin(-1)`` (``gcd/methods/clustering/k_means.py:185-186``).
    Here: the fused E-step kernel (no [N,K] matrix)."""
    src_device = X.device if torch.is_tensor(X) else torch.device('cpu')
    Xd, Cd = _dev_f32(X), _dev_f32(cluster_centers)
    labels = torch.empty(Xd.shape[0], dtype=torch.int64, device=Xd.device)
    if Xd.shape[0]:
        _estep(Xd, Cd, labels, None)
    return labels.to(src_device)


class K_Means:
    """Same constructor as the reference (``faster_mix_k_means_pytorch.py:9``; gcd copy appends ``mode``).
    ``process_group`` is the only extension (row-sharded multi-GPU)."""

    def __init__(self, k=3, tolerance=1e-4, max_iterations=100, init='k-means++', n_init=10, random_state=None,
                 n_jobs=None, pairwise_batch_size=None, mode=None, *, process_group=None):
        self.k = k
        self.tolerance = tolerance
        self.max_iterations = max_iterations
        self.init = init
        self.n_init = n_init
        self.random_state = random_state
        self.n_jobs = n_jobs                      # accepted for signature parity; restarts run sequentially on the GPU
        self.pairwise_batch_size = pairwise_batch_size
        self.mode = mode
        self.process_group = process_group

    # ------------------------------------------------------------------ sharding helpers
    def _world(self):
        if self.process_group is None:
            return 1, 0
        import torch.distributed as dist
        return dist.get_world_size(self.process_group), dist.get_rank(self.process_group)

    def _shard_layout(self, n_local, device):
        """Global row offsets of every rank's shard (``[world + 1]`` Python ints) - one all-gather of the local sizes."""
        world, _ = self._world()
        if world == 1:
            return [0, n_local]
        from . import dist as sdist
        sizes = torch.zeros(world, dtype=torch.int64, device=device)
        sdist.all_gather_into(sizes, torch.tensor([n_local], dtype=torch.int64, device=device), self.process_group)
        offs = [0]
        for v in sizes.tolist():
            offs.append(offs[-1] + int(v))
        return offs

    def _global_rows(self, Xd, global_idx):
        """``X_global[global_idx]`` on every rank when the rows of X are block-sharded: the owner of each index fills
        its row of a zero buffer, one all-reduce (sum) replicates the lot."""
        world, rank = self._world()
        idx = [int(i) for i in np.asarray(global_idx).reshape(-1)]
        if world == 1:
            return Xd[torch.as_tensor(idx, device=Xd.device, dtype=torch.int64)].clone()
        import torch.distributed as dist
        offs = self._shard_layout(int(Xd.shape[0]), Xd.device)
        out = torch.zeros(len(idx), Xd.shape[1], dtype=torch.float32, device=Xd.device)
        mine = [(j, g - offs[rank]) for j, g in enumerate(idx) if offs[rank] <= g < offs[rank + 1]]
        if mine:
            dst = torch.as_tensor([j for j, _ in mine], device=Xd.device, dtype=torch.int64)
            src = torch.as_tensor([r for _, r in mine], device=Xd.device, dtype=torch.int64)
            out[dst] = Xd[src]
        dist.all_reduce(out, op=dist.ReduceOp.SUM, group=self.process_group)
        return out

    def _peer_exchange(self, k, d, device):
        """The NVLink peer-memory exchange of this fit's (K, D), or None (single rank, a non-NCCL group such as the gloo
        CPU tests, symmetric memory unavailable, or SCD_B200_EXCHANGE=nccl): then the packed NCCL all-reduce is used."""
        import os
        if self.process_group is None or os.environ.get('SCD_B200_EXCHANGE', 'peer') == 'nccl':
            return None
        from . import peer
        cache = self.__dict__.setdefault('_px_cache', {})
        key = (int(k), int(d))
        if key not in cache:
            px = None
            if peer.available(self.process_group):
                try:
                    px = peer.PeerExchange(self.process_group, k, d, device=device)
                except Exception as e:                         # every rank fails alike (same driver, same allocator)
                    import warnings
                    warnings.warn(f'scd_b200: peer-memory exchange unavailable ({e}); using the NCCL all-reduce')
            cache[key] = px
        return cache[key]

    def _allreduce(self, mstep: _MStep, inertia_acc: torch.Tensor):
        """SURVEY 8e: one packed all-reduce of [K*D sums | K counts | inertia] when rows are sharded."""
        if self.process_group is None:
            return None
        from . import dist as sdist
        lib = _lib.load()
        _lib.check(lib.scd_pack_counts_inertia(mstep.counts.data_ptr(), inertia_acc.data_ptr(), mstep.k,
                                               mstep.counts_f.data_ptr(), _stream()), 'scd_pack_counts_inertia')
        sdist.allreduce_packed(mstep.packed, self.process_group)
        inertia_acc.copy_(mstep.packed[-1:])
        return mstep.counts_f

    def _assign(self, X, centers, labels_out, inertia_acc, estep: '_EStep | None' = None):
        """E-step of one iteration: ``labels_out[i] = argmin_k ||X_i - c_k||^2`` and ``inertia_acc += sum of the
        minima``.  (The size-constrained subclass overrides this with the min-cost-flow assignment.)"""
        if estep is not None:
            estep.run(X, centers, labels_out, inertia_acc)
        else:
            _estep(X, centers, labels_out, inertia_acc)

    def _lloyd(self, X_assign, X_all, labels, l_num, centers, l_feats=None):
        """The iteration loop shared by fit_once (:56-74) and fit_mix_once (:102-126).

        X_assign: rows that get (re)assigned each iteration (all of X, or u_feats); X_all: rows the M-step
        averages (X, or cat(l_feats, u_feats)); labels: int64 [len(X_all)], first l_num entries fixed."""
        dev = X_all.device
        k, d = self.k, X_all.shape[1]
        mstep = _MStep(X_all.shape[0], d, k, dev)
        estep = _EStep(k, d, dev)
        inertia_acc = torch.zeros(1, dtype=torch.float64, device=dev)
        px = self._peer_exchange(k, d, dev)
        inertia_red = torch.zeros(1, dtype=torch.float64, device=dev) if px is not None else None
        c_cur = centers.clone().contiguous()
        c_new = torch.empty_like(c_cur)
        # inertia and the K move norms leave the device as two small pinned copies: the one host sync per iteration
        host_i = torch.empty(1, dtype=torch.float64).pin_memory()
        host_n = torch.empty(mstep.norms.numel(), dtype=torch.float32).pin_memory()
        best_labels = best_inertia = best_centers = None
        n_done = 0
        u_view = labels[l_num:]
        for it in range(self.max_iterations):
            n_done = it + 1
            if px is not None:                      # this iteration's [sums | counts | inertia] block, mapped by every rank
                block = px.next_mstep_block()
                mstep.bind_peer(px, block)
                inertia_acc = block[2]
            inertia_acc.zero_()
            if X_assign.shape[0]:
                self._assign(X_assign, c_cur, u_view, inertia_acc, estep)          # :58-60 / :105-107,:111
            if l_num:
                lib = _lib.load()
                _lib.check(lib.scd_labelled_inertia(l_feats.data_ptr(), labels.data_ptr(), l_num, d, c_cur.data_ptr(), k,
                                                    inertia_acc.data_ptr(), _stream()), 'scd_labelled_inertia')   # :108-110
            mstep.sums_counts(X_all, labels)                                       # :61-64 / :113-116
            if px is not None:                      # all-reduce over peer loads + divide + :71 / :123, one launch
                mstep.finalize_peer(c_cur, c_new, inertia_red, estep=estep if mstep.tc else None)
            else:
                counts_f = self._allreduce(mstep, inertia_acc)
                mstep.finalize(c_cur, c_new, counts_f, estep=estep if mstep.tc else None, shift=False)   # divide + :71 / :123
            host_i.copy_(inertia_red if px is not None else inertia_acc, non_blocking=True)
            host_n.copy_(mstep.norms, non_blocking=True)
            torch.cuda.current_stream().synchronize()                              # the one host sync per iteration
            inertia = float(host_i[0])
            # :71 / :123 torch.sum(torch.sqrt(...)) in fp32: the K norms are added in a fixed order on the host
            shift = np.float32(0.0)
            for v in host_n.numpy()[:k]:
                shift = np.float32(shift + v)
            inertia32 = float(np.float32(inertia))
            if best_inertia is None or inertia32 < best_inertia:                   # :66-69 / :118-121
                best_labels, best_centers, best_inertia = labels.clone(), c_new.clone(), inertia32
            c_cur, c_new = c_new, c_cur
            if np.float32(shift) ** 2 < self.tolerance:                            # :72 / :124
                break
        return best_labels, torch.tensor(best_inertia, dtype=torch.float32, device=dev), best_centers, n_done

    # ------------------------------------------------------------------ reference API
    def kpp(self, X, pre_centers=None, k=10, random_state=None):
        """k-means++ seeding, ``faster_mix_k_means_pytorch.py:20-36`` (gcd copy :82-110 with the "no
        candidate" guard).  Keeps a running min-distance vector and only measures the newly added centre
        (``scd_kpp_update``: one N x D pass per centre instead of the reference's N x c x D); draws
        ``r = random_state.rand()`` from the same host RNG stream, one draw per centre, and resolves
        ``first index with cumsum(d2 / sum(d2)) >= r`` on the device (``scd_kpp_select``).  The picked row index
        stays on the device, so the whole seeding is a stream of launches with a single host sync at the end.
        With ``process_group`` the rows of ``X`` are this rank's shard and the draw runs over the global distance
        mass (``_kpp_sharded``); ``pre_centers`` must then be identical on every rank."""
        rs = check_random_state(random_state)
        Xd = _dev_f32(X)
        if self._world()[0] > 1:
            return self._kpp_sharded(Xd, pre_centers, k, rs)
        n, d = int(Xd.shape[0]), int(Xd.shape[1])
        dev = Xd.device
        if pre_centers is not None:
            Cc = _dev_f32(pre_centers).view(-1, d)
        else:
            Cc = Xd[rs.randint(0, len(Xd))].view(1, -1)                            # :25
        centers = torch.empty(max(k, Cc.shape[0]), d, dtype=torch.float32, device=dev)
        n_have = int(Cc.shape[0])
        centers[:n_have] = Cc
        if n_have >= k or n == 0:
            return centers[:n_have]
        lib = _lib.load()
        ws = torch.empty(lib.scd_kpp_workspace_bytes(n), dtype=torch.uint8, device=dev)
        d2 = torch.empty(n, dtype=torch.float32, device=dev)
        pick = torch.full((1,), -1, dtype=torch.int64, device=dev)
        no_hit = torch.zeros(1, dtype=torch.int32, device=dev)
        # distances to the centres we start from (:28-30): fused fp32 E-step, min-distance output only
        scratch_labels = torch.empty(n, dtype=torch.int64, device=dev)
        _estep(Xd, centers[:n_have].contiguous(), scratch_labels, None, mindist=d2, exact=True)
        sums_valid = 0
        while n_have < k:
            r = float(rs.rand())                                                   # :33 (one host draw per added centre)
            _lib.check(lib.scd_kpp_select(d2.data_ptr(), n, sums_valid, r, pick.data_ptr(), no_hit.data_ptr(), ws.data_ptr(),
                                          ws.numel(), _stream()), 'scd_kpp_select')                          # :31-34
            _lib.check(lib.scd_kpp_update(Xd.data_ptr(), n, d, pick.data_ptr(), None, 0, d2.data_ptr(), centers[n_have].data_ptr(),
                                          ws.data_ptr(), ws.numel(), _stream()), 'scd_kpp_update')           # :35 + next :28-30
            sums_valid = 1
            n_have += 1
        if int(no_hit.item()) & 2:                                                 # the one host sync of the seeding
            # gcd copy :104-107 silently reuses the previous index; with none yet, both copies fail
            raise IndexError('kpp: no cumulative probability reached the draw (reference :34)')
        return centers[:n_have]

    def _kpp_sharded(self, Xd, pre_centers, k, rs):
        """k-means++ over block-sharded rows (SURVEY 8e).  Every rank holds the same RNG state.  Per added centre: the
        shard sums of the min-distance vector are all-gathered (fp64), the draw ``r * total`` falls into exactly one
        shard, that rank resolves the row on its device with the remaining mass as its local draw and broadcasts the
        row; every rank then updates its own min-distance vector against the broadcast vector.  One small host sync
        per centre (the reference syncs per centre as well, :34 ``.nonzero()[0][0]``)."""
        import torch.distributed as dist
        from . import dist as sdist
        lib = _lib.load()
        group = self.process_group
        world, rank = self._world()
        n, d = int(Xd.shape[0]), int(Xd.shape[1])
        dev = Xd.device
        offs = self._shard_layout(n, dev)
        if pre_centers is not None:
            Cc = _dev_f32(pre_centers).view(-1, d)
        else:
            Cc = self._global_rows(Xd, [rs.randint(0, offs[-1])]).view(1, -1)      # :25 over the global row range
        centers = torch.empty(max(k, Cc.shape[0]), d, dtype=torch.float32, device=dev)
        n_have = int(Cc.shape[0])
        centers[:n_have] = Cc
        if n_have >= k:
            return centers[:n_have]
        ws = torch.empty(lib.scd_kpp_workspace_bytes(max(n, 1)), dtype=torch.uint8, device=dev)
        d2 = torch.zeros(max(n, 1), dtype=torch.float32, device=dev)
        pick = torch.full((1,), -1, dtype=torch.int64, device=dev)
        no_hit = torch.zeros(1, dtype=torch.int32, device=dev)
        if n:
            _estep(Xd, centers[:n_have].contiguous(), torch.empty(n, dtype=torch.int64, device=dev), None, mindist=d2, exact=True)
        sums = torch.zeros(world, dtype=torch.float64, device=dev)
        row = torch.empty(d, dtype=torch.float32, device=dev)
        while n_have < k:
            r = float(rs.rand())                                                   # :33, the same value on every rank
            local = d2[:n].double().sum().view(1) if n else torch.zeros(1, dtype=torch.float64, device=dev)
            sdist.all_gather_into(sums, local, group)
            shard = sums.tolist()
            total = float(sum(shard))
            if not total > 0.0:
                raise IndexError('kpp: no cumulative probability reached the draw (reference :34)')
            target, run, owner = r * total, 0.0, world - 1
            for q in range(world):
                if shard[q] > 0.0 and run + shard[q] >= target:
                    owner = q
                    break
                run += shard[q]
            if rank == owner:
                r_local = min(max((target - run) / shard[owner], 0.0), 1.0)
                pick.fill_(-1)
                _lib.check(lib.scd_kpp_select(d2.data_ptr(), n, 0, r_local, pick.data_ptr(), no_hit.data_ptr(), ws.data_ptr(),
                                              ws.numel(), _stream()), 'scd_kpp_select')
                p_host = int(pick.item())
                row.copy_(Xd[p_host if p_host >= 0 else n - 1])                    # rounding at the shard's far end: its last row
            src = dist.get_global_rank(group, owner) if group is not None else owner
            dist.broadcast(row, src=src, group=group)
            centers[n_have] = row
            if n:
                _lib.check(lib.scd_kpp_update(Xd.data_ptr(), n, d, None, row.data_ptr(), 0, d2.data_ptr(), None,
                                              ws.data_ptr(), ws.numel(), _stream()), 'scd_kpp_update')
            n_have += 1
        return centers[:n_have]

    def fit_once(self, X, random_state):
        Xd = _dev_f32(X)
        k = self.k
        if self.init == 'k-means++':
            centers = self.kpp(Xd, k=k, random_state=random_state)                 # :44
        elif self.init == 'random':
            rs = check_random_state(self.random_state)                             # :46 (self.random_state, as the reference)
            if self._world()[0] > 1 and not isinstance(self.random_state, (int, np.integer)):
                rs = random_state                                                   # the shared stream of _best_of: same draw on every rank
            n_total = self._shard_layout(int(Xd.shape[0]), Xd.device)[-1]
            idx = rs.choice(n_total, k, replace=False)
            centers = self._global_rows(Xd, idx)                                   # :47-49
        else:
            centers = self._global_rows(Xd, list(range(k))) if self._world()[0] > 1 else Xd[:k].clone()   # :50-52
        labels = torch.empty(Xd.shape[0], dtype=torch.int64, device=Xd.device)
        return self._lloyd(Xd, Xd, labels, 0, centers)

    def fit_mix_once(self, u_feats, l_feats, l_targets, random_state):
        U, L = _dev_f32(u_feats), _dev_f32(l_feats)
        tg = l_targets if torch.is_tensor(l_targets) else torch.as_tensor(l_targets)
        tg = tg.to(U.device)
        l_classes, remapped = torch.unique(tg, return_inverse=True)                # :80, :93-95 (sorted unique -> 0..C_l-1)
        l_num, n_lab_classes = int(tg.numel()), int(l_classes.numel())
        lab_labels = remapped.view(-1).long().contiguous()
        # labelled class means (:78-82) with the M-step kernels (labelled rows are replicated: no exchange)
        ms = _MStep(l_num, L.shape[1], n_lab_classes, U.device)
        ms.sums_counts(L, lab_labels)
        l_centers = torch.empty(n_lab_classes, L.shape[1], dtype=torch.float32, device=U.device)
        ms.finalize(None, l_centers)
        centers = self.kpp(U, l_centers, k=self.k, random_state=random_state)      # :98
        world, rank = self._world()
        if world > 1 and rank != 0:
            # the replicated labelled rows enter the all-reduced sums / inertia once, through rank 0
            u_labels = torch.full((U.shape[0],), -1, dtype=torch.int64, device=U.device)
            best_u, best_inertia, best_centers, _ = self._lloyd(U, U, u_labels, 0, centers)
            best_labels = torch.cat((lab_labels, best_u))
        else:
            cat_feats = torch.cat((L, U)).contiguous()                             # :83
            labels = torch.full((cat_feats.shape[0],), -1, dtype=torch.int64, device=U.device)     # :88
            labels[:l_num] = lab_labels
            best_labels, best_inertia, best_centers, _ = self._lloyd(U, cat_feats, labels, l_num, centers, l_feats=L)
        # :127 returns the stale loop variable of :94 + 1, i.e. the number of labelled rows
        return best_labels, best_inertia, best_centers, l_num

    def _best_of(self, run, src_device):
        rs = check_random_state(self.random_state)
        if self._world()[0] > 1:
            # one RNG stream for all ranks: rank 0 draws a seed from its own state (random_state=None included) and
            # broadcasts it - every rank then takes identical draws, so centres, labels and the `break` agree
            import torch.distributed as dist
            seed = torch.tensor([int(rs.randint(0, 2 ** 31 - 1))], dtype=torch.int64, device='cuda')
            src = dist.get_global_rank(self.process_group, 0) if self.process_group is not None else 0
            dist.broadcast(seed, src=src, group=self.process_group)
            rs = np.random.RandomState(int(seed.item()))
        best = None
        for _ in range(self.n_init):                                               # :133-140 / :157-164
            labels, inertia, centers, n_iters = run(rs)
            if best is None or float(inertia) < best:
                self.labels_ = labels.clone().to(src_device)
                self.cluster_centers_ = centers.clone().to(src_device)
                best = float(inertia)
                self.inertia_ = inertia.to(src_device)
                self.n_iter_ = n_iters

    def fit(self, X):
        src = X.device if torch.is_tensor(X) else torch.device('cpu')
        Xd = _dev_f32(X)
        self._best_of(lambda rs: self.fit_once(Xd, rs), src)

    def fit_mix(self, u_feats, l_feats, l_targets):
        src = u_feats.device if torch.is_tensor(u_feats) else torch.device('cpu')
        U, L = _dev_f32(u_feats), _dev_f32(l_feats)
        self._best_of(lambda rs: self.fit_mix_once(U, L, l_targets, rs), src)
