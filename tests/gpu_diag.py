"""GPU diagnostic (not a pytest file): structural probes of the tcgen05 tile and an early throughput probe.
Run on the B200 box:  python tests/gpu_diag.py [perf]"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
from adalog_b200 import ops, sweep  # noqa: E402

DEV = 'cuda'
PROBE_FROM = int(os.environ.get('PROBE_FROM', '0'))


def probe_tile():
    ok = True
    for ka, N in ((64, 64), (128, 208), (768, 256), (192, 600)):
        torch.manual_seed(1)
        A = torch.randint(-15, 16, (128, ka), device=DEV).to(torch.bfloat16)
        B = torch.randint(-15, 16, (N, ka), device=DEV).to(torch.bfloat16)
        try:
            D = ops.debug_gemm_tile(A, B)
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            print(f'tile ka={ka} N={N}: EXCEPTION {e}')
            return False
        ref = (A.double() @ B.double().t())
        wrong = (D.double() != ref)
        print(f'tile ka={ka} N={N}: wrong {wrong.sum().item()} / {wrong.numel()}  maxdiff {(D.double()-ref).abs().max().item()}')
        if wrong.any():
            ok = False
            # K mapping: A one-hot at k = m % ka, B[n,k] = k % 128  -> expect D[m,n] = (m % ka) % 128
            A1 = torch.zeros(128, ka, device=DEV)
            A1[torch.arange(128), torch.arange(128) % ka] = 1
            B1 = (torch.arange(ka, device=DEV) % 128).float().repeat(N, 1)
            D1 = ops.debug_gemm_tile(A1.to(torch.bfloat16), B1.to(torch.bfloat16))
            print('  K-map  got', D1[:16, 0].tolist(), ' expect', ((torch.arange(16) % ka) % 128).tolist())
            print('  K-map  rows 64..72 got', D1[64:72, 0].tolist())
            # N mapping
            A2 = torch.zeros(128, ka, device=DEV); A2[:, 0] = 1
            B2 = torch.zeros(N, ka, device=DEV); B2[:, 0] = (torch.arange(N, device=DEV) % 128).float()
            D2 = ops.debug_gemm_tile(A2.to(torch.bfloat16), B2.to(torch.bfloat16))
            print('  N-map  got', D2[0, :24].tolist())
            print('  N-map  tail got', D2[0, -8:].tolist(), ' expect', (torch.arange(N)[-8:] % 128).tolist())
            # M mapping
            A3 = torch.zeros(128, ka, device=DEV); A3[:, 0] = torch.arange(128, device=DEV).float()
            B3 = torch.zeros(N, ka, device=DEV); B3[:, 0] = 1
            D3 = ops.debug_gemm_tile(A3.to(torch.bfloat16), B3.to(torch.bfloat16))
            print('  M-map  got', D3[:8, 0].tolist(), D3[32:36, 0].tolist(), D3[120:, 0].tolist())
            break
    return ok


def timed(fn, iters=3):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def perf_probe():
    from adalog_b200.quantizers import UniformQuantizer
    import adalog_oracle as O
    for (Bn, T, D, Do, tag) in ((128, 197, 384, 1152, 'DeiT-S qkv'), (128, 197, 384, 384, 'DeiT-S proj'),
                                (128, 197, 1536, 384, 'DeiT-S fc2-shaped'), (128, 197, 768, 768, 'DeiT-B proj'),
                                (128, 197, 3072, 768, 'DeiT-B fc2-shaped'))[PROBE_FROM:]:
        torch.manual_seed(0)
        x = torch.randn(Bn, T, D, device=DEV)
        W = torch.randn(Do, D, device=DEV) * 0.02
        b = torch.zeros(Do, device=DEV)
        y = torch.nn.functional.linear(x, W, b)
        ctx = sweep.LinearCtx(x, y, Do)
        wq, aq = UniformQuantizer(4), UniformQuantizer(4)
        cs, cz = O.weight_candidates(W, 1, 8, 128)
        acs, acz = O.activation_candidates(x, 8, 128, False)
        wq.scale, wq.zero_point = cs[64].clone(), cz[64].clone().float()
        aq.scale, aq.zero_point = acs[:, 64].clone(), acz[:, 64].clone().float()
        flops = 2.0 * 128 * Bn * T * D * Do
        tw = timed(lambda: sweep.linear_err_w(ctx, W.view(1, Do, D), b, aq, cs, cz, 8))
        ta = timed(lambda: sweep.linear_err_a(ctx, W.view(1, Do, D), b, wq, acs, acz, 8))
        ts = timed(lambda: sweep.linear_err_a_self(ctx, acs, acz, 8, False))
        print(f'{tag}: W-sweep {tw:.2f} ms ({flops / tw / 1e9:.0f} TFLOP/s)  A-sweep {ta:.2f} ms '
              f'({flops / ta / 1e9:.0f} TFLOP/s)  a_self {ts:.2f} ms')
        if 'fc2' in tag:
            from adalog_b200.quantizers import ShiftAdaLogQuantizer
            lq = ShiftAdaLogQuantizer(4).to(DEV)
            lq.scale = torch.nn.Parameter(torch.tensor([3.0], device=DEV))
            lq.shift.data.fill_(O.SHIFT_GELU)
            lq.inited = True
            xg = torch.nn.functional.gelu(x)
            gctx = sweep.LinearCtx(xg, y, Do)
            qc = torch.arange(10, 138, device=DEV).view(1, -1)
            sc = torch.linspace(2.0, 4.0, 128, device=DEV).view(1, -1)
            tl = timed(lambda: sweep.linear_err_log(gctx, W.view(1, Do, D), b, wq, lq, sc, qc))
            tlw = timed(lambda: sweep.linear_err_w(gctx, W.view(1, Do, D), b, lq, cs, cz, 8))
            print(f'{tag}: log A-sweep {tl:.2f} ms ({flops / tl / 1e9:.0f} TFLOP/s)  W-sweep(log act) {tlw:.2f} ms')
            for nm, fn in (('log A-sweep', lambda: sweep.linear_err_log(gctx, W.view(1, Do, D), b, wq, lq, sc, qc)),
                           ('W-sweep(log act)', lambda: sweep.linear_err_w(gctx, W.view(1, Do, D), b, lq, cs, cz, 8)),
                           ('A-sweep', lambda: sweep.linear_err_a(ctx, W.view(1, Do, D), b, wq, acs, acz, 8))):
                ops.profile_reset(True)
                t = timed(fn, 2)
                fl, ms, n = ops.profile_gemm_summary()
                ops.profile_reset(False)
                print(f'   {nm}: {t:.2f} ms; GEMM kernel {ms / 3:.2f} ms in {n // 3} launches ({fl / ms / 1e9:.0f} TFLOP/s); '
                      f'rest {t - ms / 3:.2f} ms')


def perf_matmul():
    from adalog_b200.quantizers import UniformQuantizer
    import adalog_oracle as O
    Bn, H, T, dh = (128, 6, 197, 64) if not os.environ.get('SWIN_SHAPE') else (64 * 64, 4, 49, 32)   # DeiT-S / Swin-B stage 1
    torch.manual_seed(0)
    q = torch.randn(Bn, H, T, dh, device=DEV)
    k = torch.randn(Bn, H, dh, T, device=DEV)
    out = q @ k
    ctx = sweep.MatMulCtx(q, k, out)
    cs, cz = O.matmul_candidates(q, 4, 128, True)
    Aq, Bq = UniformQuantizer(3), UniformQuantizer(3)
    Aq.scale, Aq.zero_point = cs[64].clone(), cz[64].clone().float()
    Bq.scale, Bq.zero_point = cs[64].clone(), cz[64].clone().float()
    p = torch.softmax(out * 0.125, -1)
    v = torch.randn(Bn, H, T, dh, device=DEV)
    pctx = sweep.MatMulCtx(p, v, p @ v)
    qc = torch.arange(10, 138, device=DEV).view(-1, 1, 1, 1, 1)
    for tag, fn in (('QK A-sweep', lambda: sweep.matmul_err_A(ctx, Bq, cs, cz, 4, True)),
                    ('QK B-sweep', lambda: sweep.matmul_err_B(ctx, Aq, cs, cz, 4, True)),
                    ('PV log-base', lambda: sweep.matmul_err_A_log_base(pctx, Bq, qc, 4)),
                    ('PV B-sweep', lambda: sweep.matmul_err_B(pctx, _logq(), cs, cz, 4, True))):
        fn()
        torch.cuda.synchronize()
        ops.profile_reset(True)
        t = timed(fn, 2)
        flops, ms, n = ops.profile_gemm_summary()
        ff, fms, fn_ = ops.profile_fused_summary()
        ops.profile_reset(False)
        if fn_:
            print(f'{tag}: {t:.2f} ms per sweep; FUSED kernel {fms / 3:.2f} ms in {fn_ // 3} launches '
                  f'({ff / fms / 1e9:.0f} TFLOP/s); rest {t - fms / 3:.2f} ms')
        else:
            print(f'{tag}: {t:.2f} ms per sweep; GEMM kernel {ms / 3:.2f} ms in {n // 3} launches '
                  f'({flops / ms / 1e9:.0f} TFLOP/s); generator+rest {t - ms / 3:.2f} ms')


def _logq():
    from adalog_b200.quantizers import AdaLogQuantizer
    a = AdaLogQuantizer(3).to(DEV)
    a.scale = torch.nn.Parameter(torch.ones(1, 1, 1, 1, device=DEV))
    a.inited = True
    return a


if __name__ == '__main__':
    print(torch.cuda.get_device_name(0))
    good = True if os.environ.get('SKIP_TILE') else probe_tile()
    print('TILE', 'OK' if good else 'BROKEN')
    if good and len(sys.argv) > 1 and sys.argv[1] == 'perf':
        perf_probe()
    if good and len(sys.argv) > 1 and sys.argv[1] == 'matmul':
        perf_matmul()
