"""Small shapes of every kernel this round touched, for `compute-sanitizer --tool memcheck python tools/sanitize_small.py`."""
import sys
import torch
sys.path.insert(0, '.')
from scd_b200 import kmeans, naming

g = torch.Generator().manual_seed(0)
# scoring / top-k: several work items per pair, pieces of row blocks, k = 1 / 5 / 8, softmax, narrow and full widths
for (n, v, d, k, sm) in [(700, 900, 768, 5, False), (20000, 700, 128, 1, False), (5000, 3000, 256, 8, True), (300, 50000, 64, 5, False)]:
    X = torch.nn.functional.normalize(torch.randn(n, d, generator=g), dim=1).bfloat16().cuda()
    W = torch.nn.functional.normalize(torch.randn(v, d, generator=g), dim=1).bfloat16().cuda()
    vocab = naming.Vocabulary.from_rows(W)
    vals, idx, _, _ = naming.name_topk_raw(X, vocab, k, sm)
    torch.cuda.synchronize()
    print('name_topk', (n, v, d, k, sm), int(idx.min()), int(idx.max()))
# k-means: E-step (both kernel variants), M-step, divide; vote (shared-memory and spill tables)
for (n, d, k) in [(3000, 768, 100), (2000, 256, 300), (1000, 96, 33)]:
    X = torch.nn.functional.normalize(torch.randn(n, d, generator=g), dim=1).cuda()
    C = X[:k].clone()
    es, ms = kmeans._EStep(k, d, X.device), kmeans._MStep(n, d, k, X.device)
    lab = torch.empty(n, dtype=torch.int64, device='cuda'); acc = torch.zeros(1, dtype=torch.float64, device='cuda')
    es.run(X, C, lab, acc)
    ms.sums_counts(X, lab)
    cn = torch.empty_like(C); ms.finalize(C, cn, estep=es if ms.tc else None, shift=False)
    idx = torch.randint(0, 500, (n, 5), device='cuda')
    out = naming.vote_device(idx, lab, k, 5, 20)
    out2 = naming.vote_device(idx, None, k, 5, 20, presorted=ms)
    torch.cuda.synchronize()
    assert torch.equal(out[0], out2[0])
    print('kmeans + vote', (n, d, k), float(acc))
big = torch.randint(0, 40000, (60000, 5), device='cuda')
out = naming.vote_device(big, torch.randint(0, 3, (60000,), device='cuda'), 3, 5, 20)       # clusters of 20 k rows: spill tables
torch.cuda.synchronize()
print('vote with spill tables ok', int(out[4]))
