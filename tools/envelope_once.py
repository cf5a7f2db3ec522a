"""One envelope likelihood evaluation (tgp_loglike_env, want_alpha = 1) at configs[2] after one warm-up call: the
program behind the ncu launch list profiles/r2_launches_envelope_N40k.*"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import treegp_b200 as treegp  # noqa: E402
from treegp_b200 import backend  # noqa: E402
from treegp_b200.kernels import lower_kernel  # noqa: E402

n = int(os.environ.get("PN", "40000"))
X, _, kstr, _, _, noise, _ = bench.gp_problem(n, 16)
desc = lower_kernel(treegp.eval_kernel(kstr), 2)
Xd = backend.as_points(X)
plan = backend.plan_envelope(Xd, desc)
o = plan["order"]
y = backend.to_device(np.random.default_rng(0).normal(size=n))[o].contiguous()
e2 = backend.to_device(np.full(n, noise ** 2))
Xs = Xd[o].contiguous()
work = backend.alloc_matrix(n + 1, n)
for _ in range(2):
    out = backend.loglike(Xs, y, e2, desc, work=work, want_alpha=True, row_end=plan["row_end"])[0]
    torch.cuda.synchronize()
print("logL", float(out[0].item()))
