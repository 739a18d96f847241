"""Peer-memory (NVLink) exchange buffers of the sharded path (SURVEY 8e): the two exchange steps the path has - the
M-step's sum over row shards and the replication of the vote records - are done by the kernels that produce / consume
the data, through buffers every rank maps into its address space, instead of NCCL launches between them.

  * ``PeerExchange.mstep_block(parity)``: this rank's ``[K*D sums | K counts | inertia]`` block.  ``scd_mstep_sums`` and the
    E-step's inertia accumulator write straight into it; ``finalize()`` = ``scd_finalize_centers_peer``: flag barrier, peer
    loads of all G blocks added in rank order, divide, move norms, next E-step operands - one launch.
  * ``PeerExchange.gather_records()``: ``scd_pack_vote_records_peer`` stores the rank's ``[label, names]`` int32 records into
    every rank's gathered array, ``scd_peer_barrier`` orders the stores against the vote.

Buffers are torch symmetric memory (cuMem allocations exchanged once per ``PeerExchange``); blocks are double-buffered by
parity so a rank may run one exchange ahead of a slow peer (kernel docs in ``csrc/peer_kernel.cuh``).  All ranks of the
group must construct the object and call its methods in the same order.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib

MSTEP_CHANNEL, RECORD_CHANNEL = 0, 1


def _align(x: int, a: int = 256) -> int:
    return (x + a - 1) // a * a


def available(group=None) -> bool:
    """True when the group runs over NCCL on CUDA devices and torch exposes symmetric memory."""
    try:
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) < 2:
            return False
        if 'nccl' not in str(dist.get_backend(group)):
            return False
        import torch.distributed._symmetric_memory as symm_mem     # noqa: F401
        return True
    except Exception:
        return False


class PeerExchange:
    def __init__(self, group, k: int, d: int, n_total: int = 0, k_used: int = 0, device=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        self.group = group if group is not None else dist.group.WORLD
        self.world = dist.get_world_size(self.group)
        if self.world > 16:
            raise ValueError('PeerExchange supports up to 16 ranks of one NVLink domain')
        dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        buf = symm_mem.empty(self.buffer_bytes(self.world, k, d, n_total, k_used), dtype=torch.uint8, device=dev)
        buf.zero_()
        self.handle = symm_mem.rendezvous(buf, self.group.group_name)
        torch.cuda.synchronize(dev)
        dist.barrier(group=self.group)                      # every pad is zero before anybody signals
        self._carve(self.world, dist.get_rank(self.group), k, d, n_total, k_used, buf, [int(p) for p in self.handle.buffer_ptrs])

    @classmethod
    def buffer_bytes(cls, world: int, k: int, d: int, n_total: int = 0, k_used: int = 0) -> int:
        """Bytes of one rank's exchange buffer."""
        return cls.__new__(cls)._layout(world, k, d, n_total, k_used)

    def _layout(self, world: int, k: int, d: int, n_total: int, k_used: int) -> int:
        """Sizes and byte offsets of the exchange buffer - flag pad | 2 x M-step block | 2 x record array | 2 x offsets
        table - set on ``self``; returns the buffer's size in bytes."""
        lib = _lib.load()
        self.world = int(world)
        self.k, self.d, self.n_total, self.k_used = int(k), int(d), int(n_total), int(k_used)
        self.mstep_bytes = _align(lib.scd_peer_mstep_bytes(self.k, self.d))
        self.per = (self.n_total + self.world - 1) // self.world if self.n_total else 0      # rows per rank (dist.shard_bounds)
        self.rec_w = 1 + self.k_used
        self.rec_bytes = _align(self.world * self.per * self.rec_w * 4) if self.n_total else 0
        self.seg_bytes = _align(self.world * (self.k + 1) * 4) if self.n_total else 0      # [world, K + 1] offsets of the sorted runs
        self.off_mstep = _align(lib.scd_peer_flag_bytes())
        self.off_rec = self.off_mstep + 2 * self.mstep_bytes
        self.off_seg = self.off_rec + 2 * self.rec_bytes
        return self.off_seg + 2 * self.seg_bytes

    def _carve(self, world: int, rank: int, k: int, d: int, n_total: int, k_used: int, buf: torch.Tensor, ptrs):
        """Lays out this rank's exchange buffer ``buf`` (``buffer_bytes`` long, zeroed) and takes its views; ``ptrs[r]`` is
        rank r's buffer as this rank addresses it.  Needs no process group: the tests run the exchange kernels on one GPU
        with ordinary allocations standing in for the ranks' mapped buffers."""
        if buf.numel() < self._layout(world, k, d, n_total, k_used):
            raise ValueError('exchange buffer smaller than its layout')
        self.rank = int(rank)
        self.buf = buf
        self.table = (C.c_void_p * self.world)(*ptrs)       # rank -> base of its exchange buffer, mapped here
        self._mstep_parity = 0
        self._rec_parity = 0
        kd = self.k * self.d
        iw = (kd + self.k + 1) // 2 * 2                     # peer_mstep_inertia_word
        self._blocks = []
        for p in range(2):
            base = self.off_mstep + p * self.mstep_bytes
            words = self.buf[base:base + self.mstep_bytes].view(torch.float32)
            sums = words[:kd].view(self.k, self.d)
            counts = self.buf[base + 4 * kd:base + 4 * (kd + self.k)].view(torch.int32)
            inertia = self.buf[base + 4 * iw:base + 4 * iw + 8].view(torch.float64)
            self._blocks.append((sums, counts, inertia, base))
        self._records = []
        for p in range(2):
            base = self.off_rec + p * self.rec_bytes
            if self.n_total:
                rec = self.buf[base:base + self.world * self.per * self.rec_w * 4].view(torch.int32).view(self.world * self.per, self.rec_w)
                sbase = self.off_seg + p * self.seg_bytes
                seg = self.buf[sbase:sbase + self.world * (self.k + 1) * 4].view(torch.int32).view(self.world, self.k + 1)
                self._records.append((rec, base, seg, sbase))

    # ------------------------------------------------------------------ M-step
    def next_mstep_block(self):
        """(sums [K, D] fp32, counts [K] int32, inertia [1] fp64, byte offset) of the block the NEXT iteration fills."""
        blk = self._blocks[self._mstep_parity]
        self._mstep_parity ^= 1
        return blk

    def finalize(self, block, c_old, c_new, norms, counts_out, inertia_out, estep=None):
        """``scd_finalize_centers_peer`` on the block ``next_mstep_block`` returned (all ranks, same order)."""
        lib = _lib.load()
        _lib.check(lib.scd_finalize_centers_peer(self.table, self.table, self.world, self.rank, MSTEP_CHANNEL, block[3],
                                                 _lib.ptr(c_old), c_new.data_ptr(), _lib.ptr(norms) if c_old is not None else None,
                                                 _lib.ptr(counts_out), _lib.ptr(inertia_out), self.k, self.d,
                                                 estep.ws.data_ptr() if estep is not None else None,
                                                 estep.ws.numel() if estep is not None else 0,
                                                 torch.cuda.current_stream().cuda_stream), 'scd_finalize_centers_peer')
        if estep is not None:
            estep.ready_for = c_new.data_ptr()

    # ------------------------------------------------------------------ vote records
    def gather_records(self, labels_local: torch.Tensor, idx_local: torch.Tensor, k_used: int):
        """Replicates this rank's ``[label, name_0 .. name_(k-1)]`` records: returns the gathered ``[N_total, 1 + k]`` int32
        array (valid on the current stream once the barrier kernel has run)."""
        if not self.n_total or k_used != self.k_used:
            raise ValueError('PeerExchange was not sized for these vote records')
        lib = _lib.load()
        rec, base = self._records[self._rec_parity][:2]
        self._rec_parity ^= 1
        n = int(labels_local.shape[0])
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(lib.scd_pack_vote_records_peer(self.table, self.world, self.rank, base, labels_local.data_ptr(), idx_local.data_ptr(),
                                                  int(idx_local.shape[1]), k_used, n, self.rank * self.per, st), 'scd_pack_vote_records_peer')
        _lib.check(lib.scd_peer_barrier(self.table, self.world, self.rank, RECORD_CHANNEL, st), 'scd_peer_barrier')
        return rec[:self.n_total]

    def gather_sorted_records(self, mstep, idx_local: torch.Tensor, k_used: int):
        """The exchange without a second sort: ``mstep`` is the ``kmeans._MStep`` whose ``sums_counts`` has just sorted this
        rank's rows by label.  Records ``[global row id, names]`` leave in that order together with the rank's offsets;
        returns ``(records [world * per, 1 + k] int32, offsets [world, K + 1] int32)`` for ``naming.vote_segments`` - every
        cluster is then ``world`` sorted runs."""
        if not self.n_total or k_used != self.k_used or mstep.k != self.k:
            raise ValueError('PeerExchange was not sized for these vote records')
        lib = _lib.load()
        rec, base, seg, sbase = self._records[self._rec_parity]
        self._rec_parity ^= 1
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(lib.scd_pack_sorted_records_peer(self.table, self.world, self.rank, base, sbase, idx_local.data_ptr(),
                                                    int(idx_local.shape[1]), k_used, int(idx_local.shape[0]), self.rank * self.per,
                                                    mstep.ws.data_ptr(), self.k, st), 'scd_pack_sorted_records_peer')
        _lib.check(lib.scd_peer_barrier(self.table, self.world, self.rank, RECORD_CHANNEL, st), 'scd_peer_barrier')
        return rec, seg

    def unpack_sorted(self, rec: torch.Tensor, seg: torch.Tensor):
        """(labels [N_total] int64, top-k names [N_total, k] int64) in ROW order from gathered sorted-run records (tests / parity)."""
        labels = torch.full((self.n_total,), -1, dtype=torch.int64, device=rec.device)
        names = torch.full((self.n_total, self.k_used), -1, dtype=torch.int64, device=rec.device)
        seg_h = seg.cpu()
        for r in range(self.world):
            n_r = int(seg_h[r, self.k])
            block = rec[r * self.per:r * self.per + n_r].long()
            lab_r = torch.repeat_interleave(torch.arange(self.k, device=rec.device), (seg_h[r, 1:] - seg_h[r, :-1]).to(rec.device))
            labels[block[:, 0]] = lab_r
            names[block[:, 0]] = block[:, 1:]
        return labels, names

    def barrier(self, channel: int = 7):
        lib = _lib.load()
        _lib.check(lib.scd_peer_barrier(self.table, self.world, self.rank, channel, torch.cuda.current_stream().cuda_stream), 'scd_peer_barrier')
