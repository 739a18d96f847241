#!/usr/bin/env python
"""Bring-up diagnostics for the GPU box: each step runs in its own subprocess (a device trap in one step
must not take the others down) with a timeout, and everything is logged under gpurun_out/.
Usage: python tools/gpu_diag.py [step ...]      (no args = all steps)"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, 'gpurun_out')


def step_kmeans():
    import torch
    from oracle import kmeans_oracle
    from scd_b200 import kmeans
    torch.manual_seed(0)
    for (n, d, k) in [(600, 64, 12), (1, 8, 1), (130, 20, 65), (1000, 768, 100), (257, 4, 3), (5000, 768, 200), (3000, 128, 300), (2000, 64, 1000)]:
        X = torch.randn(n, d); X = X / X.norm(dim=1, keepdim=True)
        C = X[torch.randperm(n)[:k]].clone() if n >= k else torch.randn(k, d)
        ref = kmeans_oracle.pairwise_distance(X, C, None)
        got = kmeans.pairwise_distance(X.cuda(), C.cuda()).cpu()
        lab_o, mind_o, in_o = kmeans_oracle.estep(X, C)
        lab = kmeans.predict(X.cuda(), C.cuda()).cpu()
        mind = torch.empty(n, device='cuda'); acc = torch.zeros(1, dtype=torch.float64, device='cuda'); l2 = torch.empty(n, dtype=torch.int64, device='cuda')
        kmeans._estep(X.cuda(), C.cuda(), l2, acc, mind)
        print(f'pd n={n} d={d} k={k}: max|err|={float((ref-got).abs().max()):.3e} labels_equal={bool(torch.equal(lab, lab_o))}'
              f' mismatches={int((lab!=lab_o).sum())} mindist_err={float((mind.cpu()-mind_o).abs().max()):.3e} inertia_err={abs(acc.item()-float(in_o)):.3e}')
        cen_o = kmeans_oracle.mstep(X, lab_o, C.clone())
        ms = kmeans._MStep(n, d, k, 'cuda')
        ms.sums_counts(X.cuda(), lab_o.cuda())
        cn = torch.empty(k, d, device='cuda')
        ms.finalize(C.cuda(), cn)
        err = (cn.cpu() - cen_o)
        both_nan = torch.isnan(cn.cpu()) & torch.isnan(cen_o)
        err[both_nan] = 0
        sh_o = float(kmeans_oracle.center_shift(cen_o, C))
        print(f'   mstep max|err|={float(err.abs().max()):.3e} counts_ok={bool(torch.equal(ms.counts.cpu().long(), torch.bincount(lab_o, minlength=k)))}'
              f' shift={float(ms.shift.item()):.6f} oracle_shift={sh_o:.6f}')
    torch.cuda.synchronize()


def _naming_case(n, v, d, k, softmax=False, verbose=False):
    import torch
    from scd_b200 import naming
    g = torch.Generator().manual_seed(n * 7 + v)
    X = torch.randn(n, d, generator=g); X = (X / X.norm(dim=1, keepdim=True)).bfloat16()
    W = torch.randn(v, d, generator=g); W = (W / W.norm(dim=1, keepdim=True)).bfloat16()
    Xd, Wd = X.cuda(), W.cuda()
    logits = 100. * (Xd.float() @ Wd.float().t())
    if softmax:
        logits = torch.softmax(logits, dim=1)
    kk = min(k, v)
    rv, ri = logits.topk(kk, 1, True, True)
    vocab = naming.Vocabulary(Wd.float().t().contiguous())
    vals, idx, _, _ = naming.name_topk_raw(Xd, vocab, k, softmax)
    torch.cuda.synchronize()
    vals, idx = vals[:, :kk], idx[:, :kk]
    verr = float((vals - rv).abs().max())
    agree = float((idx == ri).float().mean())
    print(f'naming n={n} v={v} d={d} k={k} softmax={softmax}: max|val err|={verr:.3e} idx agree={agree:.5f}')
    if verbose and (agree < 0.999 or verr > 1e-2):
        bad_rows = ((idx != ri).any(dim=1)).nonzero().view(-1)
        print('   bad rows:', bad_rows[:40].tolist(), 'count', int(bad_rows.numel()))
        for r in bad_rows[:4].tolist():
            print('   row', r, 'got', idx[r].tolist(), [round(x, 3) for x in vals[r].tolist()], 'want', ri[r].tolist(), [round(x, 3) for x in rv[r].tolist()])
    return verr, agree


def step_naming_tiny():
    _naming_case(256, 256, 64, 5, verbose=True)
    _naming_case(256, 256, 64, 1, verbose=True)
    _naming_case(128, 512, 128, 5, verbose=True)
    _naming_case(256, 256, 768, 5, verbose=True)


def step_naming_shapes():
    for (n, v, d, k) in [(700, 300, 64, 5), (2048, 300, 64, 5), (2500, 1000, 64, 8), (1, 1, 64, 1), (300, 5000, 768, 5),
                         (1000, 3000, 768, 5), (513, 257, 72, 2), (100, 255, 768, 3), (5000, 21000, 768, 5)]:
        _naming_case(n, v, d, k, verbose=True)
    _naming_case(1000, 3000, 768, 5, softmax=True, verbose=True)
    _naming_case(300, 5000, 64, 5, softmax=True, verbose=True)


def step_vote():
    import numpy as np
    import torch
    from oracle import naming_oracle
    from scd_b200 import naming
    g = torch.Generator().manual_seed(3)
    n, k, v = 5000, 17, 400
    idx = torch.randint(0, v, (n, 5), generator=g)
    idx[:, 0] = torch.randint(0, 30, (n,), generator=g)
    preds = torch.randint(0, k, (n,), generator=g).numpy()
    for known in (None, [1, 2, 3, 7]):
        co = naming_oracle.vote(idx, preds, list(range(k)), 5, known_name_idx=known)
        cg = naming.vote(idx, preds, list(range(k)), 5, 20, known_name_idx=known)
        bad = sum([(int(a), int(b)) for a, b in cg[c].most_common(20)] != [(int(a), int(b)) for a, b in co[c].most_common(20)] for c in range(k))
        print(f'vote known={known}: clusters differing = {bad} / {k}')


def step_naming_time():
    import torch
    from scd_b200 import naming
    n, v, d = 127000, 21000, 768
    X = torch.randn(n, d, device='cuda'); X = (X / X.norm(dim=1, keepdim=True)).bfloat16()
    W = torch.randn(v, d, device='cuda'); W = (W / W.norm(dim=1, keepdim=True)).bfloat16()
    vocab = naming.Vocabulary.from_rows(W)
    for _ in range(2):
        naming.name_topk_raw(X, vocab, 5, False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        vals, idx, _, _ = naming.name_topk_raw(X, vocab, 5, False)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    print(f'name_topk C2: {ms:.3f} ms -> {2*n*v*d/ms/1e9:.1f} TFLOP/s')
    # check a row sample against torch
    rows = torch.randperm(n, device='cuda')[:2048]
    ref = (100. * (X[rows].float() @ W.float().t())).topk(5, 1, True, True)
    print('   sample idx agree', float((idx[rows] == ref[1]).float().mean()), 'max val err', float((vals[rows] - ref[0]).abs().max()))
    from scd_b200 import kmeans
    Xf = torch.randn(n, d, device='cuda'); Xf = Xf / Xf.norm(dim=1, keepdim=True)
    C = Xf[:100].clone()
    labels = torch.empty(n, dtype=torch.int64, device='cuda'); acc = torch.zeros(1, dtype=torch.float64, device='cuda')
    ms_ = kmeans._MStep(n, d, 100, 'cuda'); cn = torch.empty_like(C)
    for name, fn in (('estep', lambda: kmeans._estep(Xf, C, labels, acc)), ('mstep', lambda: (ms_.sums_counts(Xf, labels), ms_.finalize(C, cn)))):
        fn(); torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            fn()
        e1.record(); torch.cuda.synchronize()
        print(f'{name} C2: {e0.elapsed_time(e1)/5:.3f} ms')


def step_name_prof():
    """Cycle counters of the naming kernel's issuer / epilogue (scd_debug_set_name_profile)."""
    import torch
    from scd_b200 import naming, _lib
    n, v, d = 127000, 21000, 768
    X = torch.randn(n, d, device='cuda'); X = (X / X.norm(dim=1, keepdim=True)).bfloat16()
    W = torch.randn(v, d, device='cuda'); W = (W / W.norm(dim=1, keepdim=True)).bfloat16()
    vocab = naming.Vocabulary.from_rows(W)
    for _ in range(2):
        naming.name_topk_raw(X, vocab, 5, False)
    prof = torch.zeros(74 * 32 + 5 * 384, dtype=torch.int64, device='cuda')
    _lib.load().scd_debug_set_name_profile(prof.data_ptr())
    naming.name_topk_raw(X, vocab, 5, False)
    torch.cuda.synchronize()
    _lib.load().scd_debug_set_name_profile(None)
    full = prof.cpu()
    p = full[:74 * 32].view(74, 32).double()
    names = {0: 'issuer total', 1: 'issuer wait tmem_empty', 2: 'issuer wait a_full', 3: 'issuer wait b_full (blocking)',
             4: 'issuer wait token', 5: 'tiles', 6: 'B producer 0 total', 7: 'B producer 0 wait empty', 12: 'B producer 1 total',
             13: 'B producer 1 wait empty', 14: 'B producer 2 total', 15: 'B producer 2 wait empty',
             23: 'peer B producer 0 wait empty', 29: 'peer B producer 1 wait empty', 31: 'peer B producer 2 wait empty',
             8: 'epi total', 9: 'epi wait tmem_full', 10: 'epi item-final scan'}
    for k, nm in names.items():
        col = p[:, k]
        print(f'{nm:32s} mean={col.mean():12.0f} min={col.min():12.0f} max={col.max():12.0f}')
    _print_issuer_shares_and_clock(p)
    print('issuer busy-issue cycles per tile:', float(((p[:, 0] - p[:, 1] - p[:, 2] - p[:, 3] - p[:, 4]) / p[:, 5]).mean()))
    print('per-pair issuer total (first 10):', p[:10, 0].tolist())
    tr = full[74 * 32:74 * 32 + 4 * 384].view(4, 128, 3)      # the last 384 entries are the per-item timeline
    t0 = int(tr[0, 0, 0])
    print('trace pair 0 (cycles since first event): issuer0 / issuer1 runs: ready, token, issued')
    for i in range(30, 48):
        a, b = tr[0, i].tolist(), tr[1, i].tolist()
        print(f'  run {i}: I0 ready {a[0]-t0:8d} tok {a[1]-t0:8d} issued {a[2]-t0:8d} (issue {a[2]-a[1]:5d}) | I1 ready {b[0]-t0:8d} tok {b[1]-t0:8d} issued {b[2]-t0:8d} (issue {b[2]-b[1]:5d})')
    print('epilogue warp 4: tile full-seen, released, done')
    for i in range(4, 12):
        a = tr[2, i].tolist()
        print(f'  tile {i}: full {a[0]-t0:8d} released {a[1]-t0:8d} (+{a[1]-a[0]}) done {a[2]-t0:8d} (+{a[2]-a[0]})')
    print('producer 0 issue times:', [int(tr[3, i, 0]) - t0 for i in range(24, 44)])


def _gpu_query():
    """Card name, power limit and maximum SM clock (a query only; it changes no setting)."""
    import subprocess
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f'(nvidia-smi unavailable: {e})'
    print('gpu:', out)


def _print_issuer_shares_and_clock(p, launch_ms=None):
    """Issuer waits as shares of the issuer's cycles, and the effective SM clock of the launch: the issuer's clock64
    span over its %globaltimer span (column 17, ns).  A build that does not record the span gets the cycles over the
    timed launch (`launch_ms`, which includes the merge and launch gaps: a lower bound on the clock)."""
    tot = p[:, 0].sum()
    te, bf, tok = p[:, 1].sum() / tot, p[:, 3].sum() / tot, p[:, 4].sum() / tot
    print(f'issuer shares: tmem_empty {100 * te:.1f} %  b_full {100 * bf:.1f} %  tmem_empty + b_full {100 * (te + bf):.1f} %  '
          f'token {100 * tok:.1f} %')
    ns = p[:, 17]
    if float(ns.min()) > 0:
        mhz = p[:, 0] / ns * 1e3
        print(f'effective SM clock: mean {float(mhz.mean()):.0f} MHz  min {float(mhz.min()):.0f}  max {float(mhz.max()):.0f} '
              f'(issuer span {float(ns.mean()) / 1e3:.1f} us)')
    elif launch_ms:
        print(f'effective SM clock >= {float(p[:, 0].mean()) / (launch_ms * 1e3):.0f} MHz (issuer cycles / timed launch; span not recorded)')
    _gpu_query()


def step_estep_prof():
    """Cycle counters of the E-step kernel's warp roles (scd_debug_set_name_profile)."""
    import torch
    from scd_b200 import kmeans, _lib
    for (n, d, k) in [(127000, 768, 100), (127000, 768, 200), (127000, 768, 1000)]:
        X = torch.randn(n, d, device='cuda'); X = X / X.norm(dim=1, keepdim=True)
        C = X[:k].clone()
        labels = torch.empty(n, dtype=torch.int64, device='cuda'); acc = torch.zeros(1, dtype=torch.float64, device='cuda')
        for _ in range(2):
            kmeans._estep(X, C, labels, acc)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            kmeans._estep(X, C, labels, acc)
        e1.record(); torch.cuda.synchronize()
        print(f'estep n={n} k={k}: {e0.elapsed_time(e1)/5*1e3:.1f} us (incl. centroid split)')
        prof = torch.zeros(148, 16, dtype=torch.int64, device='cuda')
        _lib.load().scd_debug_set_name_profile(prof.data_ptr())
        kmeans._estep(X, C, labels, acc)
        torch.cuda.synchronize()
        _lib.load().scd_debug_set_name_profile(None)
        p = prof.cpu().double()
        names = {0: 'X producer total', 1: 'X producer wait x_empty', 2: 'C producer wait b_empty', 3: 'issuer total', 4: 'issuer wait t_empty',
                 5: 'issuer wait a_full', 6: 'issuer wait b_full', 7: 'converter total', 8: 'converter wait x_full', 9: 'converter wait a_empty',
                 10: 'epilogue wait t_full', 11: 'tiles', 12: 'issuer 0 wait token'}
        for kk, nm in names.items():
            col = p[:, kk]
            print(f'   {nm:28s} mean={col.mean():12.0f} min={col.min():12.0f} max={col.max():12.0f}')


def _time(fn, reps=10, warm=2):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def step_naming_scale():
    """The scoring/top-k launch at the per-rank shapes of the 1/2/4/8-GPU runs (one GPU is enough to see how the
    kernel behaves on a small row shard or a vocabulary shard)."""
    import numpy as np
    import torch
    from scd_b200 import naming, _lib
    d = 768
    print('SCD_NAME_WAIT_HINT_NS =', os.environ.get('SCD_NAME_WAIT_HINT_NS', '(unset)'))
    Xall = torch.randn(160000, d, device='cuda'); Xall = (Xall / Xall.norm(dim=1, keepdim=True)).bfloat16()
    Wall = torch.randn(100000, d, device='cuda'); Wall = (Wall / Wall.norm(dim=1, keepdim=True)).bfloat16()
    shapes = [(127000, 21000), (63500, 21000), (31750, 21000), (15875, 21000),           # C2 rows / N
              (127000, 10500), (127000, 5250), (127000, 2625),                              # C2 vocabulary / N
              (127000, 82000), (15875, 82000), (127000, 10250), (31750, 41000),             # C4: rows/8, vocab/8, 4x2 grid
              (160000, 100000)]                                                             # C5 rows / 8
    for n, v in shapes:
        X, vocab = Xall[:n].contiguous(), naming.Vocabulary.from_rows(Wall[:v].contiguous())
        plan = naming.TopKPlan(n, v, 5, 'cuda')
        ms = _time(lambda: plan.run(X, vocab, False), reps=5 if n * v > 5e9 else 20)
        pl = np.zeros(6, dtype=np.int32)
        _lib.load().scd_name_topk_plan(n, v, 5, pl.ctypes.data)
        print(f'rows {n:7d} x vocab {v:6d}: {ms*1e3:9.1f} us  {2*n*v*d/ms/1e9:7.1f} TFLOP/s   plan rb={pl[0]} tiles={pl[1]} pairs={pl[2]} slots={pl[3]} tiles_per_pair={pl[4]} items={pl[5]}')


def step_small_kernels():
    """The k-means pass and the vote at the row counts of a 1-GPU and an 8-GPU rank (everything but the big GEMM)."""
    import torch
    from scd_b200 import kmeans, naming
    d, k = 768, 100
    for n in (127000, 15875):
        X = torch.randn(n, d, device='cuda'); X = X / X.norm(dim=1, keepdim=True)
        C = X[:k].clone(); cn = torch.empty_like(C)
        labels = torch.empty(n, dtype=torch.int64, device='cuda'); acc = torch.zeros(1, dtype=torch.float64, device='cuda')
        ms_, es = kmeans._MStep(n, d, k, 'cuda'), kmeans._EStep(k, d, 'cuda')
        print(f'--- rows {n}')
        print(f'estep (+split)        {_time(lambda: kmeans._estep(X, C, labels, acc))*1e3:8.1f} us')
        def estep_ready():
            es.ready_for = C.data_ptr(); es.run(X, C, labels, acc)
        es.run(X, C, labels, acc)
        print(f'estep (planes ready)  {_time(estep_ready)*1e3:8.1f} us')
        print(f'mstep sums            {_time(lambda: ms_.sums_counts(X, labels))*1e3:8.1f} us')
        print(f'finalize (+planes)    {_time(lambda: ms_.finalize(C, cn, estep=es, shift=False))*1e3:8.1f} us')
        print(f'finalize (+shift)     {_time(lambda: ms_.finalize(C, cn))*1e3:8.1f} us')
    n = 127000
    idx = torch.randint(0, 21000, (n, 5), device='cuda'); idx[:, 0] = torch.randint(0, 300, (n,), device='cuda')
    labels = torch.randint(0, k, (n,), device='cuda')
    vp = naming.VotePlan(n, k, 20, 'cuda')
    ms_ = kmeans._MStep(n, d, k, 'cuda')
    X = torch.randn(n, d, device='cuda')
    ms_.sums_counts(X, labels)
    print(f'vote (sort + vote)    {_time(lambda: naming.vote_device(idx, labels, k, 5, 20, plan=vp))*1e3:8.1f} us')
    print(f'vote presorted        {_time(lambda: naming.vote_device(idx, None, k, 5, 20, plan=vp, presorted=ms_))*1e3:8.1f} us')
    rec = naming.pack_vote_records(labels, idx, 5)
    print(f'pack records          {_time(lambda: naming.pack_vote_records(labels, idx, 5, out=rec))*1e3:8.1f} us')
    print(f'vote records          {_time(lambda: naming.vote_records(rec, k, 20, plan=vp))*1e3:8.1f} us')
    n5, k5 = 1280000, 1000
    idx = torch.randint(0, 100000, (n5, 5), device='cuda'); labels = torch.randint(0, k5, (n5,), device='cuda')
    vp = naming.VotePlan(n5, k5, 20, 'cuda')
    print(f'C5 vote (sort + vote) {_time(lambda: naming.vote_device(idx, labels, k5, 5, 20, plan=vp), reps=5)*1e3:8.1f} us')


def step_name_items():
    """Per-work-item timeline of the naming kernel (pair 0) at a full-size and two small-shard shapes: where does the
    fixed cost per work item go?"""
    import numpy as np
    import torch
    from scd_b200 import naming, _lib
    d = 768
    Xall = torch.randn(127000, d, device='cuda'); Xall = (Xall / Xall.norm(dim=1, keepdim=True)).bfloat16()
    Wall = torch.randn(21000, d, device='cuda'); Wall = (Wall / Wall.norm(dim=1, keepdim=True)).bfloat16()
    for n, v in ((127000, 21000), (15875, 21000), (127000, 2625)):
        X, vocab = Xall[:n].contiguous(), naming.Vocabulary.from_rows(Wall[:v].contiguous())
        plan = naming.TopKPlan(n, v, 5, 'cuda')
        for _ in range(2):
            plan.run(X, vocab, False)
        ms = _time(lambda: plan.run(X, vocab, False), reps=5)
        prof = torch.zeros(74 * 32 + 5 * 384, dtype=torch.int64, device='cuda')
        _lib.load().scd_debug_set_name_profile(prof.data_ptr())
        plan.run(X, vocab, False)
        torch.cuda.synchronize()
        _lib.load().scd_debug_set_name_profile(None)
        full = prof.cpu()
        p = full[:74 * 32].view(74, 32).double()
        pl = np.zeros(6, dtype=np.int32)
        _lib.load().scd_name_topk_plan(n, v, 5, pl.ctypes.data)
        print(f'=== rows {n} x vocab {v}: {ms*1e3:.1f} us; plan rb={pl[0]} tiles={pl[1]} pairs={pl[2]} slots={pl[3]} tiles_per_pair={pl[4]} items={pl[5]}')
        for k, nm in {0: 'issuer total', 1: 'issuer wait tmem_empty', 2: 'issuer wait a_full', 3: 'issuer wait b_full', 4: 'issuer wait token',
                      5: 'tiles', 8: 'epi total', 9: 'epi wait tmem_full', 10: 'epi item-final scan+write'}.items():
            col = p[:, k]
            print(f'   {nm:28s} mean={col.mean():11.0f} min={col.min():11.0f} max={col.max():11.0f}')
        _print_issuer_shares_and_clock(p[p[:, 0] > 0], ms)
        it = full[74 * 32 + 4 * 384:].view(64, 6)
        t0 = int(it[0, 0]) if int(it[0, 0]) else int(it[0, 1])
        print('   pair 0 items: first MMA | first tile seen | tiles done | scan done | results written | A loads issued   (cycles since the first MMA)')
        for i in range(64):
            if int(it[i, 1]) == 0:
                break
            a = [int(x) - t0 if int(x) else -1 for x in it[i].tolist()]
            print(f'     item {i:2d}: {a[0]:9d} {a[1]:9d} {a[2]:9d} {a[3]:9d} {a[4]:9d} {a[5]:9d}   (tiles {a[2]-a[1]:8d}, scan {a[3]-a[2]:6d}, write {a[4]-a[3]:6d})')


STEPS = ['kmeans', 'naming_tiny', 'naming_shapes', 'vote', 'naming_time']

if __name__ == '__main__':
    if len(sys.argv) > 2 and sys.argv[1] == '--run':
        globals()['step_' + sys.argv[2]]()
        sys.exit(0)
    os.makedirs(OUT, exist_ok=True)
    steps = sys.argv[1:] or STEPS
    for s in steps:
        t0 = time.time()
        try:
            p = subprocess.run([sys.executable, os.path.abspath(__file__), '--run', s], capture_output=True, text=True, timeout=240)
            rc, out = p.returncode, p.stdout + '\n--- stderr ---\n' + p.stderr[-6000:]
        except subprocess.TimeoutExpired as e:
            rc, out = -999, 'TIMEOUT\n' + str(e.stdout)[-3000:] + str(e.stderr)[-3000:]
        with open(os.path.join(OUT, f'diag_{s}.txt'), 'w') as f:
            f.write(out)
        print(f'===== {s}: rc={rc} ({time.time()-t0:.1f}s)')
        print(out[-3500:])
