"""Drop-in size-constrained (semi-supervised) k-means: ``local_utils/sskm_constrained.py`` ``K_Means``
(imported by the drivers as ``ConSemiSupKMeans``, ``main_unsup.py:24`` / ``main_ptsup.py:24``; constructed at
``main_unsup.py:339`` / ``main_ptsup.py:358``) over the sm_100a kernels and the host flow solver of
``libscd_b200.so``.

Same constructor (``size_min`` / ``size_max`` after ``max_iterations``, :16), methods and result attributes as
the reference.  Per iteration the reference computes the full ``N x K`` distance matrix on the GPU, copies
``sqrt(dist)`` to the host, builds an explicit ``N*K``-arc flow graph and hands it to OR-Tools (:66-67 /
:115-116, :226-356).  Here:

  1. the fused fp32 E-step (no ``N x K`` matrix) gives the plain argmin and a device histogram gives the
     cluster sizes; a monotone transform of the distances keeps the argmin optimal, so when every size already
     lies in ``[size_min, size_max]`` - the common case with the drivers' loose defaults 50 / 1000-1200 - that
     IS an optimum of the flow problem and nothing else happens;
  2. otherwise the distance kernel emits the solver's int32 costs ``round(1000 * sqrt(dist))`` (:116 + :324)
     directly, they are copied to the host (as in the reference) and ``scd_constrained_assign`` repairs the size
     violations by successive shortest augmenting paths (exact optimum; ``csrc/constrained.cpp``).

Optimal labellings are not unique under tied integer costs, and OR-Tools is not available to compare with:
parity is on the optimal total cost and the size bounds (SURVEY 8c).  Multi-GPU: replicas only (a global
combinatorial solve, SURVEY 8e).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from .kmeans import K_Means as _K_Means, _dev_f32, _estep, _stream


def labels_constrained(cost_x1000, size_min: int, size_max: int):
    """``solve_min_cost_flow_graph`` (:331-356) on a HOST int32 cost matrix ``[N, K]``: returns
    ``(labels int32 [N], total_cost int, n_augment int)``; raises the reference's exception when the bounds are
    infeasible (``K * size_min > N`` or ``K * size_max < N``)."""
    cost = np.ascontiguousarray(cost_x1000, dtype=np.int32)
    if cost.ndim != 2:
        raise ValueError('cost matrix must be [N, K]')
    n, k = cost.shape
    labels = np.empty(n, dtype=np.int32)
    total, aug = ctypes.c_int64(0), ctypes.c_int64(0)
    rc = _lib.load().scd_constrained_assign(cost.ctypes.data, n, k, int(size_min), int(size_max), labels.ctypes.data,
                                            ctypes.byref(total), ctypes.byref(aug))
    if rc == 2:
        raise Exception('There was an issue with the min cost flow input.')        # :349-350
    if rc != 0:
        raise RuntimeError('scd_constrained_assign: bad arguments')
    return labels, int(total.value), int(aug.value)


class K_Means(_K_Means):
    """Constructor of ``local_utils/sskm_constrained.py:16``."""

    def __init__(self, k=3, tolerance=1e-4, max_iterations=100, size_min=100, size_max=1000, init='k-means++', n_init=10,
                 random_state=None, n_jobs=None, pairwise_batch_size=None):
        super().__init__(k=k, tolerance=tolerance, max_iterations=max_iterations, init=init, n_init=n_init,
                         random_state=random_state, n_jobs=n_jobs, pairwise_batch_size=pairwise_batch_size)
        self.size_min = size_min
        self.size_max = size_max
        self.n_flow_solves_ = 0          # iterations whose size bounds were active (diagnostic, not in the reference)

    def _assign(self, X, centers, labels_out, inertia_acc, estep=None):
        """``_labels_constrained`` (:226-274) for the rows of ``X``: labels into ``labels_out`` (int64, device),
        ``inertia_acc += sum_i D[i, label_i]**2`` (:271-272)."""
        lib = _lib.load()
        n, d = int(X.shape[0]), int(X.shape[1])
        k = int(centers.shape[0])
        # (1) plain argmin with the same fp32 direct-form arithmetic the cost matrix uses + cluster sizes
        plain_inertia = torch.zeros(1, dtype=torch.float64, device=X.device)
        _estep(X, centers, labels_out, plain_inertia, exact=True)
        counts = torch.empty(k, dtype=torch.int32, device=X.device)
        _lib.check(lib.scd_label_histogram(labels_out.data_ptr(), n, k, counts.data_ptr(), _stream()), 'scd_label_histogram')
        sizes = counts.cpu()
        if int(sizes.min()) >= self.size_min and int(sizes.max()) <= self.size_max:
            inertia_acc += plain_inertia
            return
        # (2) bounds active: int32 costs from the distance kernel -> host -> augmenting-path solver
        self.n_flow_solves_ += 1
        cost = torch.empty(n, k, dtype=torch.int32, device=X.device)
        _lib.check(lib.scd_pairwise_distance(X.data_ptr(), n, d, centers.data_ptr(), k, None, cost.data_ptr(), _stream()),
                   'scd_pairwise_distance')
        labels, _total, _aug = labels_constrained(cost.cpu().numpy(), self.size_min, self.size_max)
        labels_out.copy_(torch.from_numpy(labels).to(X.device, dtype=torch.int64))
        _lib.check(lib.scd_labelled_inertia(X.data_ptr(), labels_out.data_ptr(), n, d, centers.data_ptr(), k,
                                            inertia_acc.data_ptr(), _stream()), 'scd_labelled_inertia')

    def fit(self, X):
        """:141-163.  The reference's unsupervised path yields int32 labels (``labels.astype(np.int32)`` :265,
        ``torch.from_numpy`` :68) and a NumPy float32 inertia."""
        super().fit(X)
        self.labels_ = self.labels_.to(torch.int32)
        self.inertia_ = np.float32(self.inertia_.item())
