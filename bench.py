#!/usr/bin/env python
"""Benchmark of the SCD naming round (BASELINE.json metric: ms per naming round = one k-means iteration
+ full-vocabulary scoring with per-image top-k + per-cluster vote).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config C2] [--dump-outputs DIR]

* default arm: the B200 path.  `value` = ms per round of the HEADLINE config (C2, the 1-GPU configuration the metric is
  quoted on) with all inputs resident in HBM (CUDA events, max over ranks, rounds replayed as CUDA graphs); `e2e` = the same
  round through the public Python API with HOST (pinned) buffers, H2D/D2H inside the timed region; `roofline` = the dominant
  kernel (fused scoring/top-k, tensor-core bound, timed by event nodes inside the graphs) against MEASURED_PEAKS.json;
  `split.phases_us_rank0` = event nodes at every phase boundary of the round; `cpu_baseline` = the reference's CPU path
  (kind "reference" where the checkout is importable, else the oracle port) on this box's host cores on a bounded row
  sample; `torch_cuda_baseline` = the reference's own PyTorch expressions on CUDA tensors on the same GPU (N=1 only);
  `sustained` = the same graph replayed for >= 2 s.
* N > 1 (launched by torch.distributed.run, one rank per GPU): STRONG scaling of the same workload.  Image rows are
  block-sharded for BOTH contractions - k-means and naming (vocabulary replicated, no exchange).  The two exchange steps
  run inside the kernels over NVLink peer memory (scd_b200/peer.py): the divide kernel sums the ranks' [K*D sums | K counts
  | inertia] blocks with peer loads, and the pack kernel stores each rank's [label, top-k names] int32 records into every
  rank, after which the exact vote runs replicated.  `--exchange nccl` does both with NCCL launches (packed all-reduce,
  all-gather) instead.  `--naming-shard vocab` switches naming to the vocabulary-column-sharded scheme of BASELINE.json
  configs[3] (all rows x V/N columns per rank, all-gather of the [N, k] lists, k-way merge kernel); `--vocab-ways G` makes it
  a (N/G) x G rows x vocabulary process grid.
* every line also carries (unless --no-extra): `c5` - the 1.28M x 768, K=1000, V=100k stress config (configs[4]) on
  the same N GPUs, rows sharded; `c4_vocab_shard` - the V=82k sweep config (configs[3]) with the vocabulary
  column-sharded, next to the same config row-sharded (`c4_rows`; `c4_grid_2d` at N >= 4); and `parity` - sha1 hashes of
  labels / top-k indices / voted names of one round from the initial centroids, and whether the N-rank result equals a
  1-rank recomputation of the whole workload on rank 0 (`equals_n1`).
* --impl reference: the reference's own CPU implementation of the path (its k-means distance function imported from the
  checkout where present, the inline script blocks restated by the oracle - the reference is Python/PyTorch, there is
  nothing to compile into oracle/_ref) with all host threads, on a bounded sample of the same workload, extrapolated
  linearly in rows.  Rank 0 only.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

METRIC = 'ms per naming round (k-means iter + vocab top-k + vote)'
CPU_SAMPLE_ROWS = int(os.environ.get('SCD_BENCH_CPU_ROWS', '8192'))      # rows of the bounded CPU sample (tests shrink it)
TOPK, NUM_COMMON = 5, 20
CPU_KIND_DETAIL = {'reference': "k-means E-step = the reference's own pairwise_distance imported from the checkout; M-step loop, inline "
                                'scoring/top-k block and vote = the oracle restatement (script code, not importable)',
                   'port': 'oracle restatement of the reference (the checkout is absent on this box)'}


# ------------------------------------------------------------------------------------------ helpers
def load_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p.get('hbm_gbs', 6650.0), tflops=p.get('bf16_tflops', 1590.0),
                    tflops_sustained=p.get('bf16_tflops_sustained', 1400.0), source='measured')
    return dict(hbm_gbs=6650.0, tflops=1590.0, tflops_sustained=1400.0, source='fallback')


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU while the timed region runs: a background
    `nvidia-smi -lms 100` process (the profiling recipe's clocks line) - a separate process, so the
    queries never contend with this process's launch path (in-process NVML polling did: it doubled the
    measured step time)."""

    FIELDS = ['clocks.sm', 'clocks.max.sm', 'power.draw', 'clocks_event_reasons.hw_slowdown',
              'clocks_event_reasons.hw_thermal_slowdown', 'clocks_event_reasons.sw_thermal_slowdown',
              'clocks_event_reasons.sw_power_cap']

    def __init__(self, index, enabled=True):
        self.proc, self.t_start, self.t_stop = None, None, None
        if not enabled:
            return
        try:
            import subprocess
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=timestamp,' + ','.join(self.FIELDS),
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.35)           # let it print its first line before the region starts
        except Exception:
            self.proc = None

    def start(self):
        self.t_start = time.time()

    def result(self):
        self.t_stop = time.time()
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            text, _ = self.proc.communicate(timeout=2)
        except Exception:
            self.proc.kill()
            return out
        import datetime
        sm, reasons, mx, power = [], set(), None, []
        for line in text.strip().splitlines():
            parts = [x.strip() for x in line.split(',')]
            if len(parts) != 1 + len(self.FIELDS):
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], '%Y/%m/%d %H:%M:%S.%f').timestamp()
                clk, mxc = float(parts[1]), float(parts[2])
            except Exception:
                continue
            mx = mxc
            if self.t_start - 0.05 <= ts <= self.t_stop + 0.05:
                sm.append(clk)
                try:
                    power.append(float(parts[3]))
                except Exception:
                    pass
                for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), parts[4:]):
                    if val.lower().startswith('active'):
                        reasons.add(name)
        out.update(sm_mhz=(float(np.median(sm)) if sm else None), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm),
                   power_w_max=(max(power) if power else None))
        return out


def physical_gpu_index(local_rank):
    vis = os.environ.get('CUDA_VISIBLE_DEVICES')
    if vis:
        try:
            return int(vis.split(',')[local_rank])
        except Exception:
            return local_rank
    return local_rank


def sha(t: torch.Tensor) -> str:
    """sha1 of a tensor's bytes (moved to the host), first 16 hex digits."""
    return hashlib.sha1(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()[:16]


DUMP_BYTES = 60 << 20              # array data of --dump-outputs: with the .npy headers the files stay under 64 MB
PER_ROW_OUTPUTS = ('labels', 'topk_vals', 'topk_idx')


def dump_outputs(out_dir, outputs, n_rows):
    """Writes `outputs` (Round.outputs) as `out_dir/<name>.npy`, so that two builds run with the same arguments can be
    compared array by array: float32 results stay float32, everything else becomes float64, which holds every integer
    result exactly.  If the per-row arrays would take the total past DUMP_BYTES, the same rows are kept of each: a
    sample drawn with a fixed seed, whose row numbers are written as row_index.npy."""
    arrays = {k: a.astype(np.float32 if a.dtype == np.float32 else np.float64) for k, a in outputs.items()}
    fixed = sum(a.nbytes for k, a in arrays.items() if k not in PER_ROW_OUTPUTS)
    row_bytes = sum(arrays[k].nbytes for k in PER_ROW_OUTPUTS) // n_rows
    if fixed + row_bytes * n_rows > DUMP_BYTES:
        keep = (DUMP_BYTES - fixed) // (row_bytes + 8)
        if keep < 1:
            raise ValueError(f'--dump-outputs: the per-cluster arrays alone take {fixed} bytes, over the {DUMP_BYTES}-byte limit')
        rows =np.sort(np.random.default_rng(0).choice(n_rows, keep, replace=False))
        arrays.update({k: arrays[k][rows] for k in PER_ROW_OUTPUTS}, row_index=rows.astype(np.float64))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


# ------------------------------------------------------------------------------------------ CPU legs
_CPU_DATA = {}
_REF_PD = []


def reference_dir():
    """The checkout of the reference project named by SCD_REFERENCE_DIR, or None (it is not part of this repository)."""
    ref = os.environ.get('SCD_REFERENCE_DIR', '')
    return ref if ref and os.path.isdir(os.path.join(ref, 'local_utils')) else None


def reference_pairwise_distance():
    """The reference's own `pairwise_distance` (local_utils/faster_mix_k_means_pytorch.py:177), imported unmodified when
    SCD_REFERENCE_DIR names a checkout; None otherwise, and the CPU legs run the oracle port.  The inline naming / vote
    blocks of main_*.py are script code and are always the oracle's restatement."""
    if not _REF_PD:
        fn = None
        ref = reference_dir()
        if ref is not None:
            try:
                import importlib.util
                spec = importlib.util.spec_from_file_location('_scd_ref_kmeans', os.path.join(ref, 'local_utils', 'faster_mix_k_means_pytorch.py'))
                mod = importlib.util.module_from_spec(spec)
                spec.loader.exec_module(mod)
                fn = mod.pairwise_distance
            except Exception as e:
                sys.stderr.write(f'[bench] reference checkout present but not importable ({e}); using the oracle port\n')
        _REF_PD.append(fn)
    return _REF_PD[0]


def cpu_kind():
    return 'reference' if reference_pairwise_distance() is not None else 'port'


def cpu_round_ms(cfg, sample_rows, threads, repeats=2):
    """One naming round of the reference's CPU path (oracle port) on `sample_rows` rows of the workload,
    extrapolated linearly to cfg.n rows.  Returns (ms_per_round_full, detail dict)."""
    from oracle import kmeans_oracle, naming_oracle
    from scd_b200 import synth
    torch.set_num_threads(threads)
    ref_pd = reference_pairwise_distance()
    n = min(sample_rows, cfg.n)
    if (cfg.name, n) not in _CPU_DATA:
        _CPU_DATA[(cfg.name, n)] = synth.make(cfg, n_rows=n)
    data = _CPU_DATA[(cfg.name, n)]
    X, Xc, W, C0 = data['X'], data['Xc'], data['W'], data['C0']
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        if ref_pd is not None:                                              # the reference's own function, unmodified
            mind, labels = torch.min(ref_pd(X, C0, 1024), dim=1)           # faster_mix_k_means_pytorch.py:58-59
            mind.sum()
        else:
            labels, _, _ = kmeans_oracle.estep(X, C0, 1024)                 # pairwise_distance(X, C, 1024) + torch.min
        kmeans_oracle.mstep(X, labels, C0.clone())                          # the :61-64 loop
        t1 = time.perf_counter()
        idx, _ = naming_oracle.score_topk(Xc, W, 5, variant='ptsup')        # main_ptsup.py:526-545 restated
        t2 = time.perf_counter()
        c2c = naming_oracle.vote(idx, labels.numpy(), list(range(cfg.k)), 5)
        naming_oracle.voted_candidates(c2c, list(range(cfg.k)), 20)
        t3 = time.perf_counter()
        cur = dict(kmeans=t1 - t0, naming=t2 - t1, vote=t3 - t2, total=t3 - t0)
        if best is None or cur['total'] < best['total']:
            best = cur
    scale = cfg.n / n
    detail = {k: round(v * 1e3 * scale, 1) for k, v in best.items()}
    return best['total'] * 1e3 * scale, detail, n


# ------------------------------------------------------------------------------------------ reference torch path on CUDA
def torch_cuda_round(X, Xc, W, C, k, dtype):
    """The reference's OWN PyTorch expressions on CUDA tensors (what a user of the reference runs on this GPU),
    restated here - bench.py may not import oracle/ outside the CPU legs:
      * E-step   local_utils/faster_mix_k_means_pytorch.py:177-212 pairwise_distance in 1024-row batches (broadcast
                 (A - B) ** 2 .sum(-1); the result buffer is on the CPU there, :197 - kept on the device here, which
                 only helps the baseline), torch.min :59, mindist.sum() :60
      * M-step   :61-64 per-cluster nonzero -> index_select -> mean
      * naming   main_ptsup.py:538-543 per 1024-row batch: 100. * feats @ zeroshot_weights, topk(5) twice
      * vote     main_unsup.py:575-582 Counter per cluster on the host (after ONE copy of the indices, not K)
    Returns (labels, idx, per-part CUDA-event ms)."""
    from collections import Counter
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    n = X.shape[0]
    ev[0].record()
    dist = torch.empty(n, k, device=X.device)
    for lo in range(0, n, 1024):
        a = X[lo:lo + 1024].unsqueeze(1)
        dist[lo:lo + 1024] = ((a - C.unsqueeze(0)) ** 2.0).sum(dim=-1)
    mindist, labels = torch.min(dist, dim=1)
    inertia = mindist.sum()
    centers = C.clone()
    for idx in range(k):
        selected = torch.nonzero(labels == idx).squeeze()
        selected = torch.index_select(X, 0, selected)
        centers[idx] = selected.mean(dim=0)
    ev[1].record()
    feats, Wd = Xc.to(dtype), W.to(dtype)
    top_i, top_v = [], []
    for lo in range(0, n, 1024):
        logits = 100. * feats[lo:lo + 1024] @ Wd
        top_v.append(logits.topk(TOPK, 1, True, True)[0])
        top_i.append(logits.topk(TOPK, 1, True, True)[1])
    idx5 = torch.cat(top_i)
    torch.cat(top_v)
    ev[2].record()
    idx_h, lab_h = idx5.cpu().numpy(), labels.cpu().numpy()
    t0 = time.perf_counter()
    for c in range(k):
        Counter(x for x in idx_h[lab_h == c, :TOPK].reshape(-1)).most_common(NUM_COMMON)
    vote_ms = (time.perf_counter() - t0) * 1e3
    ev[3].record()
    torch.cuda.synchronize()
    float(inertia)
    return labels, idx5, dict(kmeans=ev[0].elapsed_time(ev[1]), naming=ev[1].elapsed_time(ev[2]), vote=vote_ms)


def torch_cuda_baseline(rnd, repeats=3):
    """Times `torch_cuda_round` on the headline workload, inputs resident in HBM (same tensors the B200 arm uses)."""
    cfg = rnd.cfg
    X, C = rnd.X, rnd.C0
    Xc32 = rnd.Xc.float()
    W32 = rnd.vocab.Wt.float().t().contiguous()                   # the reference's [D, V] layout
    out = {}
    for name, dtype in (('bf16', torch.bfloat16), ('fp32', torch.float32)):
        best = None
        for _ in range(repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, _, parts = torch_cuda_round(X, Xc32, W32, C, cfg.k, dtype)
            total = (time.perf_counter() - t0) * 1e3
            if best is None or total < best['total']:
                best = dict(total=total, **parts)
        out[name] = {k: round(v, 3) for k, v in best.items()}
    return dict(value=out['bf16']['total'], unit='ms', gemm_dtype='bf16 (cuBLAS); fp32 variant beside it', split_ms=out,
                what='reference PyTorch expressions on CUDA tensors (1024-row batches, [1024, V] logits in HBM, topk twice, '
                     'K-launch M-step, host Counter vote), wall clock incl. its own host syncs, best of %d' % repeats)


# ------------------------------------------------------------------------------------------ GPU arm
def device_data(cfg, device, d):
    """Synthetic inputs of one config generated ON THE DEVICE (the extra C4 / C5 blocks: 1.28M x 768 rows would take
    minutes with the host generator): unit-norm fp32 image features with K-class structure, bf16 CLIP-like features,
    bf16-rounded unit-norm vocabulary [d, V], centroids = K distinct rows.  Deterministic for a given (config, GPU type)."""
    g = torch.Generator(device=device).manual_seed(cfg.seed)
    mu = torch.randn(cfg.k, d, generator=g, device=device)
    mu = mu / mu.norm(dim=1, keepdim=True)
    y = torch.randint(0, cfg.k, (cfg.n,), generator=g, device=device)
    X = torch.empty(cfg.n, d, device=device)
    Xc = torch.empty(cfg.n, d, dtype=torch.bfloat16, device=device)
    mu2 = torch.randn(cfg.k, d, generator=g, device=device)
    mu2 = mu2 / mu2.norm(dim=1, keepdim=True)
    for lo in range(0, cfg.n, 131072):
        hi = min(lo + 131072, cfg.n)
        x = torch.randn(hi - lo, d, generator=g, device=device) + 4.0 * mu[y[lo:hi]]
        X[lo:hi] = x / x.norm(dim=1, keepdim=True)
        x = torch.randn(hi - lo, d, generator=g, device=device) + 4.0 * mu2[y[lo:hi]]
        Xc[lo:hi] = (x / x.norm(dim=1, keepdim=True)).to(torch.bfloat16)
    W = torch.empty(d, cfg.v, dtype=torch.bfloat16, device=device)
    for lo in range(0, cfg.v, 16384):
        hi = min(lo + 16384, cfg.v)
        w = torch.randn(hi - lo, d, generator=g, device=device)
        W[:, lo:hi] = (w / w.norm(dim=1, keepdim=True)).to(torch.bfloat16).t()
    pick = torch.randperm(cfg.n, generator=g, device=device)[:cfg.k]
    return dict(X=X, Xc=Xc, W=W, C0=X[pick].clone())


class Round:
    """Device-resident state of one rank and the launches of one naming round.

    N = 1: everything local.  N > 1: image rows block-sharded over the ranks for BOTH contractions - k-means (one
    packed NCCL all-reduce of [K*D sums | K counts | inertia] per iteration) and naming (every rank holds the whole
    vocabulary, so its rows' top-k needs no exchange) - then the rank's [label, top-k names] int32 records (24 bytes
    per row) are all-gathered once and the exact vote runs replicated on the gathered records.
    `naming_shard='vocab'`: a (world / vocab_ways) x vocab_ways process grid - a rank scores the rows of its row group
    against its vocabulary-column shard, the partial [rows, k] lists are all-gathered inside the group and merged by
    the k-way merge kernel (vocab_ways = world: every rank scores all rows, BASELINE.json configs[3]).

    Every round is one k-means iteration from the initial centroids C0, so its inputs, and with them its results, are
    the same from round to round and from run to run (the fp32 M-step sums vary in their last bits from run to run;
    iterated, that would change labels).  The round still does the work of an iteration of K_Means._lloyd:
    scd_finalize_centers leaves the new centres' E-step operands in `estep_next`, while the planes of C0 stay in
    `estep`."""

    def __init__(self, cfg, rank, world, group, naming_shard='rows', vocab_ways=None, data=None, host_data=None, exchange='peer',
                 fused_em=False):
        from scd_b200 import dist as sdist, kmeans, naming, synth
        self.cfg, self.rank, self.world, self.group = cfg, rank, world, group
        self.kmeans, self.naming, self.sdist = kmeans, naming, sdist
        self.naming_shard = naming_shard if world > 1 else 'rows'
        dev = torch.device('cuda')
        d = synth.D
        self.host = host_data
        if data is None:
            data = {k: host_data[k] for k in ('X', 'Xc', 'W', 'C0')}
        self.row_lo, self.row_hi = sdist.shard_bounds(cfg.n, world, rank)
        n_local = self.row_hi - self.row_lo
        own = lambda t: t.clone() if t.is_cuda else t.to(dev).contiguous()       # never keep a view of the whole config alive
        self.X = own(data['X'][self.row_lo:self.row_hi])
        self.C0 = data['C0'].to(dev).contiguous()
        self.centers = torch.empty_like(self.C0)
        self.inertia = torch.zeros(1, dtype=torch.float64, device=dev)
        self.mstep = kmeans._MStep(n_local, d, cfg.k, dev)
        self.estep = kmeans._EStep(cfg.k, d, dev)
        self.estep_next = kmeans._EStep(cfg.k, d, dev)
        self.fused_em = fused_em and self.estep.fusable(n_local)
        self.km = kmeans.K_Means(k=cfg.k, process_group=group if world > 1 else None)
        self.labels = torch.empty(n_local, dtype=torch.int64, device=dev)
        # the two exchange steps: NVLink peer memory (the fused kernels of scd_b200/peer.py) unless --exchange nccl
        self.px = None
        if world > 1 and exchange == 'peer':
            from scd_b200 import peer
            import torch.distributed as dist
            ok = 1
            try:
                self.px = peer.PeerExchange(group, cfg.k, d, n_total=cfg.n, k_used=TOPK, device=dev)
            except Exception as e:                                  # symmetric memory unavailable on this box: every rank fails alike
                sys.stderr.write(f'[bench] rank {rank}: peer-memory exchange unavailable ({e}); using the NCCL collectives\n')
                ok = 0
            flag = torch.tensor([ok], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)   # one path for all ranks
            if not bool(flag.item()):
                self.px = None
            self.inertia_red = torch.zeros(1, dtype=torch.float64, device=dev)
        self.exchange = 'peer' if self.px is not None else ('nccl' if world > 1 else None)
        self.g_rec = sdist.RowGather(cfg.n, (1 + TOPK,), torch.int32, dev, group) if world > 1 and self.px is None else None
        self.records = None
        self.subgroup = None
        if self.naming_shard == 'rows':
            self.name_rows = (self.row_lo, self.row_hi)
            self.Xc = naming._feats_bf16(own(data['Xc'][self.row_lo:self.row_hi]))
            self.vocab = naming.Vocabulary(data['W'].to(dev))
            self.topk = naming.TopKPlan(n_local, cfg.v, TOPK, dev)
            self.name_flops = 2.0 * n_local * cfg.v * d
        else:
            import torch.distributed as dist
            ways = world if not vocab_ways else int(vocab_ways)
            row_groups = world // ways
            rg, vg = sdist.grid_2d(world, rank, ways)
            # every rank must create every subgroup, in the same order
            for q in range(row_groups):
                ranks = list(range(q * ways, (q + 1) * ways))
                grp = dist.new_group(ranks=ranks) if ways < world else group
                if q == rg:
                    self.subgroup = grp
            self.ways, self.vg = ways, vg
            # a row group's rows = the union of the k-means shards of its ranks
            lo, hi = sdist.shard_bounds(cfg.n, world, rg * ways)[0], sdist.shard_bounds(cfg.n, world, rg * ways + ways - 1)[1]
            self.name_rows = (lo, hi)
            self.col_lo, self.col_hi = sdist.shard_bounds(cfg.v, ways, vg)
            self.Xc = naming._feats_bf16(own(data['Xc'][lo:hi]))
            self.vocab = naming.Vocabulary(data['W'][:, self.col_lo:self.col_hi].to(dev), col_offset=self.col_lo)
            self.topk = naming.TopKPlan(hi - lo, self.col_hi - self.col_lo, TOPK, dev, want_stats=True)
            self.name_flops = 2.0 * (hi - lo) * (self.col_hi - self.col_lo) * d
            # every rank of the group ends up with the merged lists of all the group's rows; its vote records take
            # the slice that belongs to its own k-means rows
        self.vote_plan = naming.VotePlan(cfg.n, cfg.k, NUM_COMMON, dev, k_used=TOPK)
        self.launches_per_round = 0
        self.graphs = None
        self.last = None

    # -- one round; `ev_name`: optional (start, stop) events around the scoring/top-k launches
    PHASES = ('estep', 'mstep_sums', 'reduce_divide', 'scoring_topk', 'record_exchange', 'vote')

    def run(self, ev_name=None, ev_phase=None):
        cfg, nm = self.cfg, self.naming
        launches = 0
        mark = (lambda i: ev_phase[i].record()) if ev_phase is not None else (lambda i: None)
        mark(0)
        c_old, c_new = self.C0, self.centers
        # ---- k-means iteration: E-step, M-step sums, (all-reduce), divide (+ next E-step's operands)
        inertia = self.inertia
        if self.px is not None:                     # this round's [sums | counts | inertia] block, mapped by every rank
            self.mstep.bind_peer(self.px, self.px.next_mstep_block())
            inertia = self.mstep.peer[1][2]
        inertia.zero_()
        ready = self.estep.ready_for == c_old.data_ptr()
        if self.fused_em:                           # E-step + M-step sums in ONE pass over X (rows re-read from L2 after the argmin)
            self.estep.run(self.X, c_old, self.labels, inertia, mstep=self.mstep); launches += 1 if ready else 2
            mark(1)
        else:
            self.estep.run(self.X, c_old, self.labels, inertia); launches += 1 if ready else 2     # (centroid split +) E-step
            mark(1)
            self.mstep.sums_counts(self.X, self.labels); launches += 3                # hist+scan, scatter, segment sum
        self.estep.ready_for = c_old.data_ptr()     # the planes of C0 stay in `estep`: the next round starts from C0 too
        mark(2)
        if self.px is not None:                     # all-reduce over peer loads + divide + next E-step operands: one launch
            self.mstep.finalize_peer(c_old, c_new, self.inertia_red, estep=self.estep_next); launches += 1
        else:
            counts_f = self.km._allreduce(self.mstep, self.inertia)
            launches += 1 if counts_f is not None else 0                              # pack (the all-reduce is NCCL's)
            self.mstep.finalize(c_old, c_new, counts_f, estep=self.estep_next, shift=False); launches += 1
        mark(3)
        # ---- full-vocabulary scoring + per-image top-5
        if ev_name is not None:
            ev_name[0].record()
        if self.naming_shard == 'rows':
            vals, idx, _, _ = self.topk.run(self.Xc, self.vocab, False); launches += 2
        else:
            vals, idx = self.sdist.sharded_score_topk(self.Xc, self.vocab, TOPK, False, self.subgroup, plan=self.topk); launches += 3
            lo = self.row_lo - self.name_rows[0]
            vals, idx = vals[lo:lo + (self.row_hi - self.row_lo)], idx[lo:lo + (self.row_hi - self.row_lo)]
        if ev_name is not None:
            ev_name[1].record()
        mark(4)
        # ---- per-cluster vote over all rows
        if self.world == 1:
            mark(5)
            if self.fused_em:                       # no label sort was needed for the M-step: the vote does its own
                out = nm.vote_device(idx, self.labels, cfg.k, TOPK, NUM_COMMON, plan=self.vote_plan); launches += 3
            else:
                out = nm.vote_device(idx, None, cfg.k, TOPK, NUM_COMMON, plan=self.vote_plan, presorted=self.mstep); launches += 1
        elif self.px is not None and not self.fused_em:
            # the M-step has just sorted this rank's rows by label: the sorted runs + offsets go to every rank (pack kernel =
            # the all-gather, + flag barrier) and the vote walks them - no sort of the gathered records
            records, seg = self.px.gather_sorted_records(self.mstep, idx, TOPK); launches += 2
            mark(5)
            out = nm.vote_segments(records, seg, cfg.k, NUM_COMMON, plan=self.vote_plan, n_total=cfg.n); launches += 1
            self.records = (records, seg)
        elif self.px is not None:
            records = self.px.gather_records(self.labels, idx, TOPK); launches += 2
            mark(5)
            out = nm.vote_records(records, cfg.k, NUM_COMMON, plan=self.vote_plan); launches += 3
            self.records = records
        else:
            nm.pack_vote_records(self.labels, idx, TOPK, out=self.g_rec.local); launches += 1
            records = self.g_rec.gather()
            mark(5)
            out = nm.vote_records(records, cfg.k, NUM_COMMON, plan=self.vote_plan); launches += 3
            self.records = records
        mark(6)
        self.launches_per_round = launches
        self.last = (vals, idx, out)
        return out

    def outputs(self):
        """Host copies of what the last round handed its caller: labels and inertia of the E-step, the new centres,
        top-k values and indices, and the vote (at N > 1 the per-row arrays are this rank's shard)."""
        vals, idx, (names, counts, distinct, rows, _) = self.last
        out = dict(labels=self.labels, inertia=self.inertia, centers=self.centers, topk_vals=vals, topk_idx=idx,
                   vote_names=names, vote_counts=counts, vote_distinct=distinct, cluster_rows=rows)
        return {k: t.cpu().numpy() for k, t in out.items()}

    def capture(self, n_graphs=2):
        """Record rounds into CUDA graphs (the round is launch-bound at N > 1), one per timed step up to `n_graphs`, all
        of the same round.  Every graph carries its own pair of EXTERNAL timing events around the scoring/top-k launches
        (event-record nodes), so the dominant kernel is timed inside the replayed, back-to-back region itself - one
        sample per timed step."""
        n_graphs = max(1, n_graphs)
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self.run(); self.run()                       # steady state: the planes of C0 are in the E-step workspace
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graphs, events, phase_events = [], [], []
            pool = torch.cuda.graph_pool_handle()
            for _ in range(n_graphs):
                try:
                    evs = (torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True))
                except TypeError:
                    evs = None
                try:
                    pevs = [torch.cuda.Event(enable_timing=True, external=True) for _ in range(len(self.PHASES) + 1)]
                except TypeError:
                    pevs = None
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side, pool=pool):
                    self.run(ev_name=evs, ev_phase=pevs)
                graphs.append(g)
                events.append(evs)
                phase_events.append(pevs)
            self.graphs, self.graph_events, self.graph_phase_events, self.gstep = graphs, events, phase_events, 0
        except Exception as e:                                  # eager launches are always available
            sys.stderr.write(f'[bench] CUDA graph capture failed, timing eager launches: {e}\n')
            self.graphs = None
            torch.cuda.synchronize()
        return self.graphs is not None

    def step(self):
        if self.graphs is not None:
            self.graphs[self.gstep % len(self.graphs)].replay()
            self.gstep += 1
            self.estep.ready_for = self.C0.data_ptr()
        else:
            self.run()

    def graph_kernel_ms(self, last_n):
        """Scoring/top-k durations (ms) recorded by the event nodes of the last `last_n` replays, or None."""
        if self.graphs is None or not self.graph_events or self.graph_events[0] is None:
            return None
        n = len(self.graphs)
        try:
            idx = {(self.gstep - 1 - j) % n for j in range(min(last_n, n, self.gstep))}
            return [self.graph_events[i][0].elapsed_time(self.graph_events[i][1]) for i in sorted(idx)]
        except Exception as e:
            sys.stderr.write(f'[bench] event nodes inside the graphs could not be read ({e}); timing eager launches instead\n')
            return None

    def graph_phase_us(self, last_n):
        """Per-phase durations (us, mean over the last `last_n` replays) from the event nodes inside the graphs, or None."""
        if self.graphs is None or not getattr(self, 'graph_phase_events', None) or self.graph_phase_events[0] is None:
            return None
        n = len(self.graphs)
        try:
            idx = sorted({(self.gstep - 1 - j) % n for j in range(min(last_n, n, self.gstep))})
            out = {}
            for p, name in enumerate(self.PHASES):
                out[name] = round(float(np.mean([self.graph_phase_events[i][p].elapsed_time(self.graph_phase_events[i][p + 1]) for i in idx])) * 1e3, 1)
            return out
        except Exception as e:
            sys.stderr.write(f'[bench] phase event nodes could not be read ({e})\n')
            return None

    def drop_graphs(self):
        self.graphs = None


def measure(rnd, steps, warmup, world, group, use_graph, sampler=None, keep_outputs=False):
    """Warm up, (capture,) time `steps` rounds with CUDA events between barriers, then time the scoring/top-k launches
    of a few eager rounds.  Returns (ms_per_step, naming_ms, graphed) as the max over ranks.  `keep_outputs`: host
    copies of the last timed round's results go to `rnd.timed_outputs`, taken before any later round overwrites them."""
    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier(group=group)
        torch.cuda.synchronize()

    for _ in range(warmup):
        rnd.run()
    barrier()
    graphed = rnd.capture(min(steps, 64)) if use_graph else False
    if world > 1:                                   # every rank must take the same path (collectives inside)
        import torch.distributed as dist
        flag = torch.tensor([1 if graphed else 0], device='cuda')
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if not bool(flag.item()):
            rnd.drop_graphs()
            graphed = False
    if graphed:
        for _ in range(2):
            rnd.step()
    barrier()
    if sampler is not None:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    name_evs = []
    ev0.record()
    for _ in range(steps):
        if graphed:
            rnd.step()
        else:                                       # eager: the same events, recorded around the launches of every timed step
            evs = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            rnd.run(ev_name=evs)
            name_evs.append(evs)
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    if keep_outputs:
        rnd.timed_outputs = rnd.outputs()
    # the dominant kernel, timed live INSIDE the timed region: event-record nodes of the replayed graphs (or the eager
    # events above); only if a graph could not carry events, a few eager rounds right after the region
    per_step = rnd.graph_kernel_ms(steps) if graphed else [a.elapsed_time(b) for a, b in name_evs]
    where = 'event nodes inside the replayed graphs' if graphed else 'events around the eager launches of the timed steps'
    if per_step is None:
        name_evs = []
        for _ in range(max(3, min(steps, 20))):
            evs = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            rnd.run(ev_name=evs)
            name_evs.append(evs)
        barrier()
        per_step = [a.elapsed_time(b) for a, b in name_evs]
        where = 'eager rounds right after the timed region'
    name_ms = float(np.mean(per_step))
    rnd.phase_us = rnd.graph_phase_us(steps) if graphed else None
    t = torch.tensor([ms_total, name_ms], dtype=torch.float64, device='cuda')
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    rnd.kernel_timing = f'{where}, mean of {len(per_step)} steps'
    return float(t[0]) / steps, float(t[1]), graphed


def parity_block(rnd, data, world, group):
    """One round from the initial centroids on the N ranks; hashes of the gathered labels / top-k indices / voted names;
    on rank 0 the same round recomputed on ONE GPU over all rows (`equals_n1`).  At N = 1 the hashes are the reference
    values a reader compares the N > 1 lines with."""
    from scd_b200 import kmeans, naming
    cfg = rnd.cfg
    names, counts, _, _, ovf = rnd.run()
    vals, idx, _ = rnd.last
    torch.cuda.synchronize()
    if world > 1:
        rec = rnd.records                                        # gathered records of this very round
        if isinstance(rec, tuple):                               # sorted runs [global row id, names] + per-rank offsets
            labels_all, idx_all = rnd.px.unpack_sorted(*rec)
        else:
            labels_all, idx_all = rec[:, 0].long(), rec[:, 1:].long()
    else:
        labels_all, idx_all = rnd.labels, idx
    out = dict(labels_sha=sha(labels_all), topk_idx_sha=sha(idx_all), voted_sha=sha(names), vote_counts_sha=sha(counts),
               vote_overflow=int(ovf.item()), rows=int(labels_all.shape[0]))
    if world > 1 and rnd.rank == 0:
        dev = torch.device('cuda')
        X = data['X'].to(dev)
        lab1 = torch.empty(cfg.n, dtype=torch.int64, device=dev)
        kmeans._estep(X, rnd.C0, lab1, None)
        del X
        vocab = naming.Vocabulary(data['W'].to(dev))
        _, idx1 = naming.score_topk(naming._feats_bf16(data['Xc']), vocab, k=TOPK, softmax=False)
        names1, counts1, _, _, _ = naming.vote_device(idx1, lab1, cfg.k, TOPK, NUM_COMMON)
        torch.cuda.synchronize()
        out.update(n1=dict(labels_sha=sha(lab1), topk_idx_sha=sha(idx1), voted_sha=sha(names1), vote_counts_sha=sha(counts1)),
                   labels_mismatch=int((lab1 != labels_all).sum().item()), topk_idx_mismatch=int((idx1 != idx_all).sum().item()),
                   voted_mismatch=int((names1 != names).sum().item()))
        out['equals_n1'] = bool(out['labels_mismatch'] == 0 and out['topk_idx_mismatch'] == 0 and out['voted_mismatch'] == 0 and
                                torch.equal(counts1, counts))
    return out


def extra_block(name, rank, world, group, peaks, steps, naming_shard, vocab_ways=None, exchange='peer', fused_em=False):
    """Timing + parity of one of the other BASELINE.json configs on the same N GPUs (device-generated inputs)."""
    from scd_b200 import synth
    cfg = synth.CONFIGS[name]
    t0 = time.time()
    data = device_data(cfg, torch.device('cuda'), synth.D)
    rnd = Round(cfg, rank, world, group, naming_shard, vocab_ways, data=data, exchange=exchange, fused_em=fused_em)
    if world == 1:
        data_keep = None
    else:
        data_keep = data if rank == 0 else None
    del data
    ms, name_ms, graphed = measure(rnd, steps, 3, world, group, use_graph=True)
    rnd.drop_graphs()
    par = parity_block(rnd, data_keep, world, group)
    achieved = rnd.name_flops / (name_ms * 1e-3) / 1e12
    blk = dict(workload=f'{cfg.name}: {cfg.n}x{synth.D} image features, K={cfg.k}, V={cfg.v} names, top-{TOPK}, vote top-{NUM_COMMON}',
               sharding=('rows' if rnd.naming_shard == 'rows' else f'{world // rnd.ways} row groups x {rnd.ways} vocabulary shards'),
               ms_per_step=round(ms, 4), naming_ms=round(name_ms, 4), rest_ms=round(ms - name_ms, 4), steps=steps,
               phases_us_rank0=getattr(rnd, 'phase_us', None),
               kernel_tflops=round(achieved, 1), kernel_frac=round(achieved / peaks['tflops'], 4),
               kernel_frac_of_sustained=round(achieved / peaks['tflops_sustained'], 4),
               launch_mode='cuda-graph replay' if graphed else 'eager', data='synthetic, generated on the device',
               parity=par, wall_s=round(time.time() - t0, 1))
    del rnd, data_keep
    torch.cuda.empty_cache()
    return blk


def e2e_round(cfg, host, vocab, pinned, out_host):
    """One round through the public API from HOST buffers: H2D of the step's inputs, the round, D2H of the results.
    The PCIe link is the bound (780 MB up), so the round is ordered around it: the CLIP-like features go first (scored
    chunk by chunk under their own upload), their top-k lists leave on a side stream while the k-means features go up in
    panels (each panel assigned while the next is on the wire); M-step, vote and the small results follow the last byte."""
    from scd_b200 import kmeans, naming, synth
    synth_d = synth.D
    main = torch.cuda.current_stream()
    C = pinned['C0'].to('cuda', non_blocking=True)
    vals, idx = naming.score_topk(pinned['Xc'], vocab, k=TOPK, softmax=False)       # host features: chunked upload under the kernel
    side = torch.cuda.Stream()
    side.wait_stream(main)
    with torch.cuda.stream(side):
        out_host['vals'].copy_(vals, non_blocking=True)
        out_host['idx'].copy_(idx, non_blocking=True)
    ms = kmeans._MStep(cfg.n, synth_d, cfg.k, C.device)
    fused = False           # one-pass E+M (scd_estep_mstep) per panel was tried here too: 14.51 vs 14.46 ms - the last panel's slower launch eats what the shorter tail gains
    X, labels, inertia = kmeans.assign_from_host(pinned['X'], C, mstep=ms if fused else None)   # panels up, E(+M) per panel
    centers, counts, _, ms = kmeans.update_centers(X, labels, cfg.k, mstep=ms if fused else None)
    names, counts_v, distinct, rows, ovf = naming.vote_device(idx, labels if fused else None, cfg.k, TOPK, NUM_COMMON,
                                                              presorted=None if fused else ms)
    for key, t in (('labels', labels), ('centers', centers), ('names', names), ('counts', counts_v), ('inertia', inertia)):
        out_host[key].copy_(t, non_blocking=True)
    main.wait_stream(side)
    torch.cuda.synchronize()
    vals.record_stream(side); idx.record_stream(side)
    h2d = pinned['X'].numel() * 4 + C.numel() * 4 + pinned['Xc'].numel() * 4
    d2h = sum(t.numel() * t.element_size() for t in out_host.values())
    return h2d, d2h


def h2d_gbs(pinned_t):
    """Measured pinned host -> device copy bandwidth (GB/s) of this box: the floor of `e2e` is its bytes over this."""
    dst = torch.empty_like(pinned_t, device='cuda')
    dst.copy_(pinned_t, non_blocking=True)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    dst.copy_(pinned_t, non_blocking=True)
    ev1.record()
    torch.cuda.synchronize()
    return pinned_t.numel() * pinned_t.element_size() / (ev0.elapsed_time(ev1) * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='C2')
    ap.add_argument('--naming-shard', default='rows', choices=['rows', 'vocab'],
                    help='N > 1: how the scoring/top-k is partitioned (rows: no exchange; vocab: all-gather + k-way merge)')
    ap.add_argument('--vocab-ways', type=int, default=0, help='with --naming-shard vocab: vocabulary shards per row group (default: N)')
    ap.add_argument('--exchange', default='peer', choices=['peer', 'nccl'],
                    help='N > 1: the M-step sum and the vote-record replication run over NVLink peer memory inside the kernels '
                         '(scd_b200/peer.py), or as NCCL all-reduce / all-gather launches between them')
    ap.add_argument('--fused-em', action='store_true', help='k-means iteration as ONE pass over X (scd_estep_mstep: rows re-read from L2 and reduced with red.v4 after the argmin) - measured slower than the two-pass default, DESIGN 3.3')
    ap.add_argument('--no-graph', action='store_true', help='time eager launches instead of CUDA-graph replays')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-torch-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-clocks', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the c5 / c4_vocab_shard / sustained blocks')
    ap.add_argument('--extra-steps', type=int, default=5)
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the results of the last timed round as DIR/<name>.npy (one GPU, B200 arm; at most 64 MB)')
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup

    from scd_b200 import synth
    cfg = synth.CONFIGS[args.config]
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.dump_outputs and (args.impl != 'b200' or world > 1):
        ap.error('--dump-outputs writes the round of the B200 arm in one process: use it with --impl b200 and no launcher')
    feat_mb = cfg.n * synth.D * 6 / 1e6
    voc_mb = cfg.v * synth.D * 2 / 1e6
    if world == 1:
        par = 'single GPU'
    elif args.naming_shard == 'rows':
        if args.exchange == 'peer':
            par = (f'rows/{world} for k-means (sums+counts+inertia summed over NVLink peer loads inside the divide kernel) and for '
                   f'naming (vocabulary replicated, no exchange); [label, top-k names] int32 records stored into every rank over '
                   f'peer memory by the pack kernel, exact vote replicated')
        else:
            par = (f'rows/{world} for k-means (packed NCCL all-reduce of sums+counts+inertia) and for naming (vocabulary replicated, '
                   f'no exchange); [label, top-k names] int32 records all-gathered once, exact vote replicated')
    else:
        ways = args.vocab_ways or world
        par = (f'rows/{world} (k-means, all-reduce) x naming on a {world // ways} x {ways} rows x vocabulary grid (all-gather of '
               f'[rows, k] lists inside a row group + k-way merge); vote records all-gathered once, exact vote replicated')
    config = dict(workload=f'{cfg.name}: {cfg.n}x{synth.D} image features, K={cfg.k}, V={cfg.v} names, top-5, vote top-20',
                  n=cfg.n, d=synth.D, k=cfg.k, v=cfg.v, topk=5,
                  l2=(f'inputs ({feat_mb:.0f} MB features + {voc_mb:.0f} MB vocabulary) exceed the 126 MB L2' if feat_mb + voc_mb > 126 else
                      f'inputs ({feat_mb:.0f} MB features + {voc_mb:.0f} MB vocabulary) FIT the 126 MB L2: not a valid timing config, parity only'),
                  parallelism=par)

    # -------------------------------------------------------------------------------- reference arm
    if args.impl == 'reference':
        if rank != 0:
            return 0
        threads = os.cpu_count() or 1
        vals = []
        for s in range(max(args.steps, 1) + max(args.warmup, 0)):
            ms, detail, n_s = cpu_round_ms(cfg, CPU_SAMPLE_ROWS, threads, repeats=1)
            if s >= args.warmup:
                vals.append(ms)
        v = float(np.median(vals))
        sample = f'{n_s} of {cfg.n} rows (all {cfg.k} centroids, all {cfg.v} names), time scaled linearly in rows'
        print(json.dumps(dict(impl='reference', metric=METRIC, value=round(v, 1), unit='ms', n_gpus=args.gpus, steps=args.steps,
                              warmup=args.warmup, ms_per_step=round(v, 1), higher_is_better=False, scaling='strong',
                              vs_baseline=None, dtype='f32', data='synthetic', config=config,
                              cpu_baseline=dict(value=round(v, 1), unit='ms', cores=threads, kind=cpu_kind(), kind_detail=CPU_KIND_DETAIL[cpu_kind()], sample=sample, split_ms=detail,
                                                reference_checkout_present=reference_dir() is not None),
                              e2e=dict(value=round(v, 1), unit='ms', h2d_bytes_per_step=0, d2h_bytes_per_step=0))))
        return 0

    # -------------------------------------------------------------------------------- B200 arm
    assert torch.cuda.is_available(), 'bench.py needs a GPU (the B200 path has no CPU fallback)'
    # stdout carries exactly ONE JSON line: NCCL prints its version banner on fd 1 when NCCL_DEBUG is set (seen on the
    # 2-GPU box), so everything libraries write to fd 1 is sent to stderr and the line goes to the saved descriptor
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    group = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
        group = dist.group.WORLD
    peaks = load_peaks()
    host = synth.make(cfg)
    rnd = Round(cfg, rank, world, group, args.naming_shard, args.vocab_ways or None, host_data=host, exchange=args.exchange, fused_em=args.fused_em)

    sampler = ClockSampler(physical_gpu_index(local_rank), enabled=not args.no_clocks)
    ms_per_step, name_ms, graphed = measure(rnd, args.steps, args.warmup, world, group, not args.no_graph, sampler,
                                            keep_outputs=bool(args.dump_outputs))
    clocks = sampler.result()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rnd.timed_outputs, cfg.n)
    launches_per_round = rnd.launches_per_round
    phase_us = getattr(rnd, 'phase_us', None)
    fused_flag = rnd.fused_em
    exchange_used = rnd.exchange
    rnd.drop_graphs()
    parity = parity_block(rnd, host, world, group)

    # roofline of the dominant kernel: fused scoring/top-k (tensor-core bound); algorithmic flops = 2 * rows * cols * D of this rank
    flops = rnd.name_flops
    achieved = flops / (name_ms * 1e-3) / 1e12
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'roofline_traffic.json')
    if os.path.exists(tpath) and world == 1 and cfg.name == 'C2':      # the ncu capture is of the single-GPU C2 launch
        with open(tpath) as f:
            traffic = json.load(f).get('name_topk_kernel_dram_bytes_per_launch')
    roofline = dict(bound='tensor', kernel='name_topk_kernel<5> (+ topk_merge)', achieved=round(achieved, 1), peak=peaks['tflops'],
                    unit='TFLOP/s', frac=round(achieved / peaks['tflops'], 4), traffic=traffic,
                    peak_source=f"{peaks['source']} bf16 burst (MEASURED_PEAKS.json); sustained figure: {peaks['tflops_sustained']}",
                    kernel_ms=round(name_ms, 4), flops_per_launch=flops, kernel_timing=rnd.kernel_timing)

    # sustained regime: the same graph replayed back to back for >= 2 s (power-capped clocks), against the sustained peak
    sustained = None
    if not args.no_extra and world == 1:
        rnd.capture(2)
        n_rep = max(50, int(2200.0 / max(ms_per_step, 0.05)))
        s2 = ClockSampler(physical_gpu_index(local_rank), enabled=not args.no_clocks)
        torch.cuda.synchronize()
        s2.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_rep):
            rnd.step()
        e1.record()
        torch.cuda.synchronize()
        ms_sus = e0.elapsed_time(e1) / n_rep
        ck = s2.result()
        k_ms = rnd.graph_kernel_ms(2)
        if k_ms:
            k_sus, how = float(np.mean(k_ms)), 'event nodes of the last two replays'
        else:
            k_sus, how = ms_sus - (ms_per_step - name_ms), 'sustained round minus the burst-measured rest of the round'
        sustained = dict(rounds=n_rep, seconds=round(ms_sus * n_rep / 1e3, 2), ms_per_step=round(ms_sus, 4), kernel_ms=round(k_sus, 4),
                         kernel_tflops=round(flops / (k_sus * 1e-3) / 1e12, 1),
                         kernel_frac_of_sustained_peak=round(flops / (k_sus * 1e-3) / 1e12 / peaks['tflops_sustained'], 4),
                         kernel_timing=how, clocks=ck)
        rnd.drop_graphs()

    e2e = None
    cpu_baseline = None
    torch_base = None
    if rank == 0 and world == 1 and not args.no_e2e:
        pinned = {k: host[k].pin_memory() for k in ('X', 'Xc', 'C0')}
        out_host = dict(vals=torch.empty(cfg.n, TOPK, dtype=torch.float32).pin_memory(), idx=torch.empty(cfg.n, TOPK, dtype=torch.int64).pin_memory(),
                        labels=torch.empty(cfg.n, dtype=torch.int64).pin_memory(), centers=torch.empty(cfg.k, synth.D).pin_memory(),
                        names=torch.empty(cfg.k, NUM_COMMON, dtype=torch.int64).pin_memory(),
                        counts=torch.empty(cfg.k, NUM_COMMON, dtype=torch.int32).pin_memory(), inertia=torch.empty(1, dtype=torch.float64).pin_memory())
        gbs = h2d_gbs(pinned['X'])
        for _ in range(2):
            h2d, d2h = e2e_round(cfg, host, rnd.vocab, pinned, out_host)
        torch.cuda.synchronize()
        n_e2e = max(3, min(args.steps, 10))
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            h2d, d2h = e2e_round(cfg, host, rnd.vocab, pinned, out_host)
        torch.cuda.synchronize()
        e2e = dict(value=round((time.perf_counter() - t0) * 1e3 / n_e2e, 3), unit='ms', h2d_bytes_per_step=int(h2d),
                   d2h_bytes_per_step=int(d2h), h2d_gbs_measured=round(gbs, 1), pcie_floor_ms=round(h2d / gbs / 1e6, 3),
                   api='naming.score_topk (host features, chunked upload under the kernel; top-k lists leave on a side stream) + kmeans.assign_from_host (panels assigned under the upload) + kmeans.update_centers + naming.vote_device, pinned host tensors in and out')
        del pinned
    elif world > 1:
        e2e = dict(value=None, unit='ms', h2d_bytes_per_step=0, d2h_bytes_per_step=0, note='measured at N=1 only')
    if rank == 0 and world == 1 and not args.no_torch_baseline:
        try:
            torch_base = torch_cuda_baseline(rnd)
        except Exception as e:                                     # a baseline, never a reason to lose the line
            torch_base = dict(value=None, error=str(e)[:200])
        torch.cuda.empty_cache()
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, detail, n_s = cpu_round_ms(cfg, CPU_SAMPLE_ROWS, threads, repeats=2)
        cpu_baseline = dict(value=round(v, 1), unit='ms', cores=threads, kind=cpu_kind(), kind_detail=CPU_KIND_DETAIL[cpu_kind()], split_ms=detail,
                            reference_checkout_present=reference_dir() is not None,
                            sample=f'{n_s} of {cfg.n} rows (all {cfg.k} centroids, all {cfg.v} names), time scaled linearly in rows')

    # the other BASELINE.json configs on the same N GPUs
    extra = {}
    del rnd, host
    torch.cuda.empty_cache()
    if not args.no_extra:
        try:
            extra['c5'] = extra_block('C5', rank, world, group, peaks, args.extra_steps, 'rows', exchange=args.exchange, fused_em=args.fused_em)
            extra['c4_vocab_shard'] = extra_block('C4', rank, world, group, peaks, args.extra_steps, 'vocab', exchange=args.exchange, fused_em=args.fused_em)
            extra['c4_rows'] = extra_block('C4', rank, world, group, peaks, args.extra_steps, 'rows', exchange=args.exchange, fused_em=args.fused_em)
            if world >= 4:
                extra['c4_grid_2d'] = extra_block('C4', rank, world, group, peaks, args.extra_steps, 'vocab', vocab_ways=2, exchange=args.exchange, fused_em=args.fused_em)
        except Exception as e:
            if world > 1:
                raise                                              # a rank that skips a collective would hang the others
            extra['error'] = str(e)[:300]

    if rank == 0:
        line = dict(metric=METRIC, value=round(ms_per_step, 4), unit='ms', n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=round(ms_per_step, 4), higher_is_better=False, scaling='strong', vs_baseline=None, dtype='bf16',
                    data='synthetic', config=config, clocks=clocks, e2e=e2e, gpu_launches=launches_per_round * args.steps,
                    launch_mode='cuda-graph replay' if graphed else 'eager',
                    roofline=roofline, cpu_baseline=cpu_baseline, torch_cuda_baseline=torch_base,
                    exchange=exchange_used, kmeans_pass='E-step + M-step sums fused in one pass over X' if fused_flag else 'E-step, label sort, segment sum: two passes over X',
                    split=dict(naming_ms=round(name_ms, 4), rest_ms=round(ms_per_step - name_ms, 4), phases_us_rank0=phase_us),
                    parity=parity, sustained=sustained, **extra)
        real_stdout.write(json.dumps(line) + '\n')
        real_stdout.flush()
    if world > 1:
        # Leave without tearing NCCL down: destroy_process_group() / interpreter exit can block for minutes while
        # a CUDA graph that captured NCCL kernels is still alive (seen on the 2-GPU box).  Every rank has passed
        # the final barrier and rank 0 has flushed its line, so a hard exit loses nothing.
        import torch.distributed as dist
        dist.barrier(group=group)
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


if __name__ == '__main__':
    sys.exit(main())
