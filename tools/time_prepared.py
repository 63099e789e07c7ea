"""Development aid: device time of the prepared-operand k-NN call at a C4-like shape, for whichever
library HM_MATCHER_SO points to (timing experiments of the tensor-core pipeline)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from slam_experiments_b200 import _native as nat, synth
nq, nt = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (2000, 8192000)
v = os.environ.get("HM_TRACE_VARIANT", "f4")
t_host = synth.uniform(nt, 2)
# HM_TP_DIST=M: matchable queries (60 % noisy copies of train rows), the distribution bench.py's C4 line uses
q_host = synth.matchable_queries(t_host, nq, 3) if os.environ.get("HM_TP_DIST") == "M" else synth.uniform(nq, 1)
q = torch.from_numpy(q_host).cuda()
t = torch.from_numpy(t_host).cuda()
tp, qp = nat.prepare(t, variant=v), nat.prepare(q, variant=v)
# sanity check of the library under test: tensor core == POPC on a slice
cq, ct = q[:1000], t[:50000]
same = torch.equal(nat.knn2_keys(cq, ct, variant=v), nat.knn2_keys(cq, ct, variant="popc"))
for _ in range(3):
    nat.knn2_keys_prepared(qp, nq, tp, nt, variant=v)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
n = int(os.environ.get("HM_TP_ITERS", "20"))
e0.record()
for _ in range(n):
    nat.knn2_keys_prepared(qp, nq, tp, nt, variant=v)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / n
tiles_per_sm = (nq + 255) // 256 * ((nt + 127) // 128) / nat.sm_count()
print(f"{os.path.basename(nat.SO_PATH)} {v} {nq}x{nt}: {ms:.4f} ms, {nq * nt / ms / 1e6:.0f} Gpairs/s, "
      f"{ms * 1e-3 * 1.965e9 / tiles_per_sm:.0f} cycles per 128 columns at 1965 MHz, results {'OK' if same else 'WRONG'}")
