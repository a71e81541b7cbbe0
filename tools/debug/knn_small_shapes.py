"""Small-cloud self-kNN: (QT, GP) sweep per problem shape (whole call, L2 flushed)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "hit-adv_b200"), os.path.join(ROOT, "tools")):
    sys.path.insert(0, p)
import torch
from hitgeom import functional as F
from bench import make_clouds
from bench_ops import timeit

flush = (torch.empty(256 << 20, dtype=torch.uint8, device="cuda"), torch.zeros(64 << 20, dtype=torch.float32, device="cuda"))
SHAPES = ((32, 1024, 20), (32, 1024, 6), (388, 1024, 6), (388, 1024, 20), (64, 2048, 6), (32, 2048, 20), (16, 4096, 6))
if len(sys.argv) > 1 and sys.argv[1] == 'big':
    SHAPES = ((32, 8192, 6), (64, 8192, 6), (16, 16384, 6), (128, 16384, 6), (32, 8192, 20), (16, 16384, 20))
for B, N, k1 in SHAPES:
    x = torch.from_numpy(make_clouds(B, N, 3)[1]).cuda()
    F.force_knn_shape(0, 0)
    ref = F.knn_self(x, k1)
    line = f"B={B} N={N} k1={k1}: auto {timeit(lambda: F.knn_self(x, k1), flush=flush) * 1e3:7.1f} us |"
    for qt in ((1, 2, 4) if k1 <= 6 else (1, 2)):
        for gp in (1, 2, 4):
            F.force_knn_shape(qt, gp)
            try:
                out = F.knn_self(x, k1)
                ok = torch.equal(out[1], ref[1])
                line += f" q{qt}g{gp} {timeit(lambda: F.knn_self(x, k1), flush=flush) * 1e3:6.1f}{'' if ok else '!'}"
            except Exception as e:
                line += f" q{qt}g{gp} n/a"
    F.force_knn_shape(0, 0)
    print(line, flush=True)
