"""Two-rank TorchProblem worker (launched with torch.distributed.run, one rank per
GPU): the C3 workload partitioned over the ranks as the reference partitions it over
MPI ranks, with the objective and constraints summed by Context.allreduce_sum, against
the reference's two-rank history (tests/golden/C3_small_np2.json).  Rank 0 prints
one line `TORCH_MGPU {json}`."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from paropt_b200.api import Context, InteriorPoint  # noqa: E402
from tests.parity import compare_histories, load_golden  # noqa: E402
from tests.torch_problems import make  # noqa: E402

local_rank = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local_rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
ctx = Context(local_rank)
ctx.init_distributed()
gold = load_golden("C3_small_np2")
cfg = gold["config"]
prob = make(ctx, cfg)
ip = InteriorPoint(prob, dict(cfg["options"], history_level=2))
ip.optimize()
hist = ip.history()
n, worst, first = compare_histories(gold["history"], hist, cfg=cfg, label="C3_small_np2 torch")
verdict = {"world": ctx.size, "rows": len(gold["history"]), "got_rows": len(hist),
           "compared": n, "first_violation": first, "nvars_local": prob.nvars,
           "transfer_bytes": list(prob.transfer_bytes()), "status": ip.status(),
           "gold_status": gold["status"]}
ip.free()
prob.free()
if ctx.rank == 0:
    print("TORCH_MGPU " + json.dumps(verdict))
ctx.close()
dist.destroy_process_group()
