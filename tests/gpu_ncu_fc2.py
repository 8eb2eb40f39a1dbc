"""ncu target (not a pytest file): the AdaLog activation sweep and the weight sweep of a DeiT-B fc2-shaped layer
(128 images x 197 tokens, K=3072, N=768).
  ncu --set full --clock-control none --import-source on -k regex:'gen_log_cand|cand_gemm_err' -c 6 python tests/gpu_ncu_fc2.py"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
from adalog_b200 import sweep  # noqa: E402
from adalog_b200.quantizers import ShiftAdaLogQuantizer, UniformQuantizer  # noqa: E402
import adalog_oracle as O  # noqa: E402  (candidate seeding only; this is a profiling helper, not product code)

DEV = torch.device('cuda', 0)
Bn, T, D, Do = 128, 197, 3072, 768
torch.manual_seed(0)
x = torch.nn.functional.gelu(torch.randn(Bn, T, D, device=DEV))
W = torch.randn(Do, D, device=DEV) * 0.02
b = torch.zeros(Do, device=DEV)
y = torch.nn.functional.linear(x, W, b)
ctx = sweep.LinearCtx(x, y, Do)
wq = UniformQuantizer(4)
cs, cz = O.weight_candidates(W, 1, 8, 128)
wq.scale, wq.zero_point = cs[64].clone(), cz[64].clone().float()
lq = ShiftAdaLogQuantizer(4).to(DEV)
lq.scale = torch.nn.Parameter(torch.tensor([3.0], device=DEV))
lq.shift.data.fill_(O.SHIFT_GELU)
lq.inited = True
qc = torch.arange(10, 138, device=DEV).view(1, -1)
sc = torch.linspace(2.0, 4.0, 128, device=DEV).view(1, -1)
which = sys.argv[1] if len(sys.argv) > 1 else 'a'
if which == 'a':
    e = sweep.linear_err_log(ctx, W.view(1, Do, D), b, wq, lq, sc, qc)
elif which == 'u':      # uniform int8 activation sweep of the same shape
    x0 = torch.randn(Bn, T, D, device=DEV)
    uctx = sweep.LinearCtx(x0, torch.nn.functional.linear(x0, W, b), Do)
    acs, acz = O.activation_candidates(x0, 8, 128, False)
    e = sweep.linear_err_a(uctx, W.view(1, Do, D), b, wq, acs, acz, 8)
else:
    e = sweep.linear_err_w(ctx, W.view(1, Do, D), b, lq, cs, cz, 8)
torch.cuda.synchronize()
print('done', float(e.sum()))
