"""Sweep-level timing of the linear activation sweeps: fused generator + GEMM kernel vs generator -> workspace -> GEMM
(not a pytest file).  python tests/gpu_lin_bench.py [small|base]"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import adalog_oracle as O  # noqa: E402
from adalog_b200 import sweep  # noqa: E402
from adalog_b200.quantizers import ShiftAdaLogQuantizer, UniformQuantizer  # noqa: E402

DEV = 'cuda'


def uq(bits, s, z):
    q = UniformQuantizer(bits)
    q.scale, q.zero_point, q.inited = s, z, True
    return q


def timeit(fn, reps=5):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    which = sys.argv[1] if len(sys.argv) > 1 else 'small'
    D, bits = (384, 3) if which == 'small' else (768, 4)
    tokens = 128 * 197
    nl = 2 ** (bits - 1)
    for name, in_f, out_f, log in (('qkv', D, 3 * D, False), ('proj', D, D, False), ('fc1', D, 4 * D, False),
                                   ('fc2', 4 * D, D, True)):
        torch.manual_seed(1)
        x = torch.randn(tokens, in_f, device=DEV) * (torch.rand(in_f, device=DEV) * 2) + 0.3 * torch.randn(in_f, device=DEV)
        if log:
            x = torch.nn.functional.gelu(x)
        W = torch.nn.init.trunc_normal_(torch.empty(out_f, in_f, device=DEV), std=.02)
        b = torch.randn(out_f, device=DEV) * 0.02
        y = torch.nn.functional.linear(x, W, b)
        ctx = sweep.LinearCtx(x.view(128, 197, in_f), y.view(128, 197, out_f), out_f)
        W3 = W.view(1, out_f, in_f)
        wcs, wcz = O.weight_candidates(W, 1, nl, 128)
        wq = uq(bits, wcs[64].clone(), wcz[64].clone().float())
        if log:
            lq = ShiftAdaLogQuantizer(bits).to(DEV)
            lq.scale = torch.nn.Parameter(torch.tensor([float(x.max()) * 0.9 + O.SHIFT_GELU], device=DEV))
            lq.shift.data.fill_(O.SHIFT_GELU)
            lq.q.fill_(27)
            lq.update_table()
            lq.inited = True
            s0 = float(lq.scale.detach())
            sc = torch.linspace(s0 * 0.7, s0 * 1.1, 128, device=DEV).view(1, -1)
            qc = (torch.arange(128, device=DEV) % 24 + 18).view(1, -1)
            fn = lambda: sweep.linear_err_log(ctx, W3, b, wq, lq, sc, qc)
        else:
            acs, acz = O.activation_candidates(x.view(128, 197, in_f), nl, 128, False)
            fn = lambda: sweep.linear_err_a(ctx, W3, b, wq, acs, acz, nl)
        if os.environ.get('WSIDE'):
            # weight-side sweep of the same layer (tokens are the GEMM columns): cand_gemm_err_kernel MODE_RB
            aq = lq if log else uq(bits, acs[:, 64].clone(), acz[:, 64].clone().float())
            t_w = timeit(lambda: sweep.linear_err_w(ctx, W3, b, aq, wcs, wcz, nl))
            print(f'{which} {name:5s} K={in_f:5d} N(tokens)={tokens} units={out_f:5d} W-side {"bf16" if log else "i8"}: '
                  f'{t_w:7.3f} ms ({2.0 * 128 * tokens * in_f * out_f / t_w / 1e9:7.0f} Tops/s)', flush=True)
            continue
        policy = sweep._lin_fused_passes
        sweep._lin_fused_passes = lambda: 1 << 30      # fused wherever it fits
        t_f = timeit(fn)
        sweep._lin_fused_passes = lambda: None         # two-kernel path
        t_p = timeit(fn)
        sweep._lin_fused_passes = policy
        ops = 2.0 * 128 * tokens * in_f * out_f
        print(f'{which} {name:5s} K={in_f:5d} N={out_f:5d} {"log bf16" if log else "uniform i8"}: fused {t_f:7.3f} ms '
              f'({ops / t_f / 1e9:7.0f} Tops/s)   two-kernel {t_p:7.3f} ms ({ops / t_p / 1e9:7.0f} Tops/s)', flush=True)


if __name__ == '__main__':
    main()
