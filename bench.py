#!/usr/bin/env python
"""FPCS calibration benchmark (BASELINE.json metric: FPCS calibration wall-time & candidates/s; fake-quant img/s).

One STEP = one complete FPCS calibration (QuantCalibrator.batching_quant_calib: capture forwards + all 3150 search
evaluations x 128 candidates) of DeiT-Small W3A3 on this rank's 128 synthetic 224x224 images (BASELINE.json
configs[1]); random-init weights, seed 5.  Weak scaling: every rank calibrates against its own 128-image shard and
the per-candidate FP64 error sums are all-reduced (NCCL), so N ranks calibrate one model on N*128 images.

  python bench.py [--gpus N --steps K --warmup W]          our arm (CUDA kernels through libadalog_b200.so)
  python bench.py --impl reference [...]                    reference arm: the oracle port of the reference's own
                                                            CPU path on the host cores (bounded sample per step)
  python bench.py --config {1..5} [...]                     BASELINE.json configs[i-1]: 1 DeiT-T W4A4 / 32 images,
                                                            2 DeiT-S W3A3 / 128 per GPU (default, weak scaling),
                                                            3 ViT-B W4A4 / 512 images in total (strong scaling),
                                                            4 DeiT-B W4A4 / 1024 in total (headline), 5 Swin-B W6A6 / 1024
  With --gpus 8 and the default config the line also carries a `headline` record: one calibration of config 4.
  python bench.py --dump-outputs DIR [...]                  also write the calibrated model of the last timed step
                                                            as DIR/<state_dict key>.npy (see dump_outputs)

Prints ONE JSON line (rank 0).  `value` = candidate scorings per second with the images resident in HBM;
`e2e` = the same through the public API starting from pinned host images (H2D inside the timed region) and ending
with the calibrated quantizer parameters read back to the host.  Both legs run --steps timed steps.
"""
import argparse
import copy
import importlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL_ALIASES = {'deit_tiny': 'deit_tiny_patch16_224', 'deit_small': 'deit_small_patch16_224',
                 'deit_base': 'deit_base_patch16_224', 'vit_base': 'vit_base_patch16_224',
                 'vit_small': 'vit_small_patch16_224', 'swin_base': 'swin_base_patch4_window7_224',
                 'swin_tiny': 'swin_tiny_patch4_window7_224', 'vit_test': 'vit_test_patch8_32'}
DIMS = {'deit_tiny': (192, 3, 12), 'deit_small': (384, 6, 12), 'deit_base': (768, 12, 12), 'vit_base': (768, 12, 12),
        'vit_small': (384, 6, 12)}
TOKENS = 197
# BASELINE.json configs: (model, bits, images in total or per GPU, scaling)
CONFIGS = {1: ('deit_tiny', 4, 32, 'weak'), 2: ('deit_small', 3, 128, 'weak'), 3: ('vit_base', 4, 512, 'strong'),
           4: ('deit_base', 4, 1024, 'strong'), 5: ('swin_base', 6, 1024, 'strong')}


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed `ncu --set full`
    summary (profiles/), or None: a bench run cannot measure DRAM traffic itself (never a number taken under a profiler)"""
    for name in ('r2_ncu_full_lin_fused_i8.json', 'r2_ncu_full_lin_fused_log.json', 'r1_ncu_full_cand_gemm_err_v2.json'):
        path = os.path.join(ROOT, 'profiles', name)
        if os.path.exists(path):
            try:
                d = json.load(open(path))
                t = d.get('dram_bytes_per_launch')
                if t:
                    return float(t), f"profiles/{name}: {d.get('what', '')}"[:300]
            except Exception:  # noqa: BLE001
                pass
    return None, 'no ncu summary with dram_bytes_per_launch under profiles/'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', type=int, default=None, choices=sorted(CONFIGS))
    ap.add_argument('--model', default=None)
    ap.add_argument('--bits', type=int, default=None)
    ap.add_argument('--images-per-gpu', type=int, default=None)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-parity', action='store_true', help='skip the free-running parity / gpu_reference checker leg')
    ap.add_argument('--no-headline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the calibrated model of the last timed step as DIR/<state_dict key>.npy')
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if a.dump_outputs and a.impl == 'reference':
        ap.error('--dump-outputs needs --impl ours: the reference arm times a sample of sweeps, not a calibration')
    world = int(os.environ.get('WORLD_SIZE', '1'))
    model, bits, images, scaling = CONFIGS[a.config or 2]
    a.scaling = scaling if a.images_per_gpu is None else 'weak'
    a.model = a.model or model
    a.bits = a.bits or bits
    if a.images_per_gpu is None:
        a.images_per_gpu = images if scaling == 'weak' else max(1, images // world)
    a.images_total = a.images_per_gpu * world
    return a


def load_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(tflops=p.get('bf16_tflops_sustained', p.get('bf16_tflops')), hbm=p.get('hbm_gbs'), src='measured')
    return dict(tflops=1400.0, hbm=6650.0, src='fallback')   # B200_PROFILING.md fallback (sustained)


def count_evals(model):
    """search evaluations of one calibration, from the wrapped model's module classes (SURVEY.md section 3.4):
    plain asymmetric linear 48, channel-wise linear 6 + 48, post-GELU linear 6 + 3 x 13, Q.K^T 36, post-softmax P.V 21,
    patch-embedding conv 6"""
    per = {'AsymmetricallyBatchingQuantLinear': 48, 'AsymmetricallyChannelWiseBatchingQuantLinear': 54,
           'PostGeluLogBasedBatchingQuantLinear': 45, 'AsymmetricallyBatchingQuantMatMul': 36,
           'PostSoftmaxAsymmetricallyBatchingQuantMatMul': 21, 'AsymmetricallyBatchingQuantConv2d': 6}
    return sum(per.get(type(m).__name__, 0) for m in model.modules())


def model_eval_counts(model_key):
    """(evaluations, candidates, average MACs per token per candidate) for a ViT/DeiT: SURVEY.md section 3.4"""
    D, H, depth = DIMS[model_key]
    evals = depth * 258 + 6 + 48
    macs = (36 * 3 + 36 * 1 + 36 * 4 + 39 * 4) * D * D + (36 + 21) * TOKENS * D     # per token, per block
    return evals, evals * 128, macs / 258.0


# ------------------------------------------------------------------------------------------------ CPU arm
def eval_counts_per_block():
    """search evaluations of one ViT/DeiT block by sweep type (SURVEY.md section 3.4; 258 in total)"""
    return {
        'qkv.a_self_cw': 6, 'qkv.w_self': 6, 'qkv.a_self': 6, 'qkv.w': 18, 'qkv.a': 18,
        'proj.w_self': 6, 'proj.a_self': 6, 'proj.w': 18, 'proj.a': 18,
        'fc1.a_self_cw': 6, 'fc1.w_self': 6, 'fc1.a_self': 6, 'fc1.w': 18, 'fc1.a': 18,
        'fc2.w_self': 6, 'fc2.log': 21, 'fc2.w': 18,
        'matmul1.A': 18, 'matmul1.B': 18, 'matmul2.log_base': 3, 'matmul2.B': 18,
    }


def cpu_stratified_sample(model_key, bits, n_img, threads):
    """Bounded, STRATIFIED sample of the reference's CPU path (oracle port): ONE evaluation (128 candidates) of every
    sweep type of a transformer block -- weight / activation / self-error searches of qkv, proj, fc1, fc2 (post-GELU
    AdaLog), Q.K^T operand searches, the post-softmax base search and the V search -- on n_img synthetic images at the
    model's real layer sizes.  The seconds of each type are weighted by how often a calibration runs it
    (eval_counts_per_block x depth) and scaled linearly from n_img to the bench's images (every sweep is a sum over
    samples).  Returns (estimated seconds of a full calibration per image, image-independent seconds, per-type seconds)."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import adalog_oracle as O
    torch.set_num_threads(threads)
    D, H, depth = DIMS[model_key]
    nl = 2 ** (bits - 1)
    g = torch.Generator().manual_seed(5)

    def lnlike(n, c):
        return torch.randn(n_img, TOKENS, c, generator=g) * (torch.rand(c, generator=g) * 2) + 0.3 * torch.randn(c, generator=g)

    t = {}

    def clock(name, fn):
        t0 = time.perf_counter()
        with torch.no_grad():
            fn()
        t[name] = time.perf_counter() - t0

    for name, in_f, out_f, n_V in (('qkv', D, 3 * D, 3), ('proj', D, D, 1), ('fc1', D, 4 * D, 1), ('fc2', 4 * D, D, 1)):
        log = name == 'fc2'
        x = torch.nn.functional.gelu(lnlike(n_img, in_f)) if log else lnlike(n_img, in_f)
        W = torch.nn.init.trunc_normal_(torch.empty(out_f, in_f), std=.02, generator=g)
        b = torch.zeros(out_f)
        y = torch.nn.functional.linear(x, W, b)
        s = O.LinearSearch(W, b, x, y, bits, bits, n_V=n_V, calib_batch_size=32, a_kind='adalog' if log else 'uniform')
        s.init_calib()
        wcs, wcz = O.weight_candidates(W, n_V, nl, 128)
        s.wq.scale, s.wq.zero_point = wcs[64].clone(), wcz[64].clone().float()
        if log:
            ud, sc = O.postgelu_candidates(x, O.SHIFT_GELU, 128)
            s.aq.scale = sc[:, -2].clone()
            s.aq.update_table()
            qc = torch.arange(10, 138).view(1, -1)
            clock('fc2.log', lambda: s.sims_log(sc, qc))
        else:
            acs, acz = O.activation_candidates(x, nl, 128, False)
            s.aq.scale, s.aq.zero_point = acs[:, 64].clone(), acz[:, 64].clone().float()
            clock(name + '.a', lambda: s.sims_a(acs, acz))
            clock(name + '.a_self', lambda: s.sims_a_self(acs, acz))
            if name in ('qkv', 'fc1'):
                ccs, ccz = O.activation_candidates(x, nl, 128, True)
                s.a_channel_wise = True
                clock(name + '.a_self_cw', lambda: s.sims_a_self(ccs, ccz))
                s.a_channel_wise = False
        clock(name + '.w', lambda: s.sims_w(wcs, wcz))
        clock(name + '.w_self', lambda: s.sims_w_self(wcs, wcz))
    dh = D // H
    q = torch.randn(n_img, H, TOKENS, dh, generator=g)
    k = torch.randn(n_img, H, dh, TOKENS, generator=g)
    m = O.MatMulSearch(q, k, q @ k, bits, bits, H, calib_batch_size=32)
    m.init_calib()
    cs, cz = O.matmul_candidates(q, nl, 128, True)
    kcs, kcz = O.matmul_candidates(k, nl, 128, True)
    m.Aq.scale, m.Aq.zero_point = cs[-2].clone(), cz[-2].clone().float()
    m.Bq.scale, m.Bq.zero_point = kcs[-2].clone(), kcz[-2].clone().float()
    clock('matmul1.A', lambda: m.sims_A(cs, cz))
    clock('matmul1.B', lambda: m.sims_B(kcs, kcz))
    pr = torch.softmax(torch.randn(n_img, H, TOKENS, TOKENS, generator=g) * 2, dim=-1)
    v = torch.randn(n_img, H, TOKENS, dh, generator=g)
    m2 = O.MatMulSearch(pr, v, pr @ v, bits, bits, H, calib_batch_size=32, post_softmax=True)
    m2.init_calib()
    vcs, vcz = O.matmul_candidates(v, nl, 128, True)
    m2.Bq.scale, m2.Bq.zero_point = vcs[-2].clone(), vcz[-2].clone().float()
    clock('matmul2.log_base', lambda: m2.sims_A_log_base(torch.arange(10, 138).view(-1, 1, 1, 1, 1)))
    clock('matmul2.B', lambda: m2.sims_B(vcs, vcz))
    counts = eval_counts_per_block()
    # the weight self-error sweeps touch no calibration sample: their seconds do not scale with the image count
    per_image_block = sum(counts[k_] * t[k_] for k_ in counts if not k_.endswith('.w_self')) / n_img
    fixed_block = sum(counts[k_] * t[k_] for k_ in counts if k_.endswith('.w_self'))
    return per_image_block * depth, fixed_block * depth, t


def cpu_arm_value(model_key, bits, n_img, images_per_gpu, threads):
    """(candidates/s in the bench's unit, seconds the sample took, candidates it scored, per-type seconds)"""
    t0 = time.perf_counter()
    per_image, fixed, per_type = cpu_stratified_sample(model_key, bits, n_img, threads)
    secs = time.perf_counter() - t0
    evals, cands, _ = model_eval_counts(model_key)
    est_calibration_s = per_image * images_per_gpu + fixed   # blocks only: patch embedding (6) and head (48) are < 1%
    return cands / est_calibration_s, secs, 128 * len(per_type), per_type


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n_img = 4
    for _ in range(min(args.warmup, 1)):
        cpu_arm_value(args.model, args.bits, 2, args.images_per_gpu, threads)
    vals, secs_all = [], []
    for _ in range(args.steps):
        v, secs, cands, _ = cpu_arm_value(args.model, args.bits, n_img, args.images_per_gpu, threads)
        vals.append(v)
        secs_all.append(secs)
    value = statistics.mean(vals)
    sample = (f'oracle port of the reference CPU path, {threads} threads: per step ONE evaluation (128 candidates) of each '
              f'of the 21 sweep types of a {args.model} W{args.bits}A{args.bits} block on {n_img} images at the real layer '
              f'sizes; per-type seconds weighted by their count in a calibration (258 per block x depth) and scaled '
              f'linearly to {args.images_per_gpu} images (every sweep is a sum over samples)')
    out = dict(metric='fpcs_candidates_per_s', value=value, unit='candidates/s', n_gpus=args.gpus, steps=args.steps,
               warmup=args.warmup, ms_per_step=1e3 * statistics.mean(secs_all), higher_is_better=True, scaling=args.scaling,
               vs_baseline=None, dtype='f32', data='synthetic', impl='reference',
               config=workload_config(args),
               cpu_baseline=dict(value=value, unit='candidates/s', cores=threads, kind='port', sample=sample),
               e2e=dict(value=value, unit='candidates/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(out))


def workload_config(args):
    return dict(workload=f'{args.model} W{args.bits}A{args.bits} FPCS calibration (eq_n=128, steps=6, search_round=3), '
                         f'{args.images_per_gpu} synthetic 224x224 images per GPU, random-init weights, seed 5',
                baseline_config=args.config or 2, images_per_gpu=args.images_per_gpu,
                images_total=args.images_per_gpu * args.gpus,
                l2='inputs larger than L2 + 256 MiB L2 flush between steps',
                parallelism=f'dp{args.gpus} (samples sharded, FP64 error sums all-reduced)')


# ------------------------------------------------------------------------------------------------ our arm
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        try:
            self.p = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms',
                                       '200', '-i', str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.p = None

    def stop(self):
        if self.p is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.strip().split(', ') for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, reasons, mx = [], set(), None
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, col in (('hw_slowdown', 5), ('hw_thermal_slowdown', 6), ('sw_thermal_slowdown', 7),
                                  ('sw_power_cap', 8)):
                    if r[col].strip().lower() == 'active':
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                continue
        busy = [v for v in sm if v > 0]
        return dict(sm_mhz=statistics.median(busy) if busy else None, sm_max_mhz=mx, reasons=sorted(reasons),
                    samples=len(sm))


def build_wrapped(model_name, cfg, device):
    from adalog_b200.utils import models as zoo
    from adalog_b200.utils.wrap_net import wrap_modules_in_net
    torch.manual_seed(5)
    model = zoo.create_model(model_name).eval()
    model = wrap_modules_in_net(model, cfg, reparam=True)
    return model.to(device).eval()


def calibrate(model, images, bs):
    from adalog_b200.utils.calibrator import QuantCalibrator
    loader = [(images[i:i + bs], None) for i in range(0, images.shape[0], bs)]
    cal = QuantCalibrator(model, loader)
    cal.progress = False
    cal.batching_quant_calib()


def quant_params_to_host(model):
    out, nbytes = {}, 0
    for k, v in model.state_dict().items():
        if 'quantizer' in k:
            out[k] = v.cpu()
            nbytes += v.numel() * v.element_size()
    return out, nbytes


DUMP_SAMPLE = 1 << 16
DUMP_LIMIT = 64 << 20


def dump_outputs(model, out_dir):
    """Writes the calibrated model's state_dict -- what a caller of the timed calibration receives, and what
    test_quant.py saves as the checkpoint -- as out_dir/<key>.npy: float32 tensors as float32, every other dtype as
    float64 (exact for the int64 base indices and the bool flags).  A tensor of more than DUMP_SAMPLE elements is
    written flattened, as its elements at DUMP_SAMPLE fixed seeded positions (sorted), so two builds of the project
    compare position for position; DeiT-S comes to about 14 MB instead of 88 MB."""
    arrays = {}
    for k, v in model.state_dict().items():
        v = v.detach()
        if v.numel() > DUMP_SAMPLE:
            pos = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            v = v.reshape(-1)[pos.to(v.device)]
        arrays[k] = v.to(torch.float32 if v.dtype == torch.float32 else torch.float64).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f'--dump-outputs: {total} bytes exceed the {DUMP_LIMIT} byte limit')
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def run_ours(args):
    import torch.distributed as dist
    from adalog_b200 import _lib, ops
    from adalog_b200.utils.wrap_net import wrap_reparamed_modules_in_net

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    _lib.load()   # fail loudly if the extension is missing

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_stepper(model_key, bits, images_per_gpu):
        """(one_step(from_host) -> (ms, wall_ms, d2h_bytes, model), host images, device images, evaluations)"""
        cfg = importlib.import_module(f'adalog_b200.configs.{bits}bit').Config()
        cfg.calib_size, cfg.calib_batch_size = images_per_gpu, 32
        base = build_wrapped(MODEL_ALIASES[model_key], cfg, dev)
        g = torch.Generator().manual_seed(5 + 1000 * rank)
        img = 32 if model_key == 'vit_test' else 224
        host_images = torch.randn(images_per_gpu, 3, img, img, generator=g).pin_memory()
        dev_images = host_images.to(dev)

        def one_step(from_host):
            model = copy.deepcopy(base)
            flush.fill_(1)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            images = host_images.to(dev, non_blocking=True) if from_host else dev_images
            calibrate(model, images, 32)
            d2h = 0
            if from_host:
                _, d2h = quant_params_to_host(model)
            e1.record()
            barrier()
            ms = e0.elapsed_time(e1)
            wall = (time.perf_counter() - t0) * 1e3
            if world > 1:
                t = torch.tensor([ms], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = t.item()
            return ms, wall, d2h, model
        return one_step, host_images, dev_images, count_evals(base)

    one_step, host_images, dev_images, evals = make_stepper(args.model, args.bits, args.images_per_gpu)

    for _ in range(args.warmup):
        one_step(False)

    sampler = ClockSampler(local) if rank == 0 else None
    _lib.LAUNCHES['count'] = 0
    ops.profile_reset(True)
    times = []
    model = None
    for _ in range(args.steps):
        ms, wall, _, model = one_step(False)
        times.append(ms)
    gemm_split = ops.profile_gemm_summary(split=True)          # cand_gemm_err_kernel (W-side, conv, chunked A-side)
    lin_split = ops.profile_lin_summary()                      # lin_fused_kernel (A-side sweeps of the linear layers)
    fz_flops, fz_ms, fz_launches = ops.profile_fused_summary()
    ops.profile_reset(False)
    gemm_ms = sum(v[1] for v in gemm_split.values()) + sum(v[1] for v in lin_split.values())
    gemm_launches = sum(v[2] for v in gemm_split.values()) + sum(v[2] for v in lin_split.values())
    launches = _lib.LAUNCHES['count']
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:      # every rank calibrates to the same parameters (errors are all-reduced)
        dump_outputs(model, args.dump_outputs)

    e2e_ms, d2h = None, 0
    if not args.no_e2e:
        e_times, d2h = [], 0
        for _ in range(args.steps):
            ms, wall, d2h, _ = one_step(True)
            e_times.append(ms)
        e2e_ms = statistics.mean(e_times)

    # fake-quant forward throughput of the calibrated model (second half of BASELINE's metric): the default forward
    # (bit-identical to the reference's composition) and the opt-in exact-integer tensor-core forward, with their
    # top-1 agreement on the batch
    from adalog_b200.utils.wrap_net import set_tensor_core_forward
    model = wrap_reparamed_modules_in_net(model)

    def fq_rate(bs):
        with torch.no_grad():
            # two untimed forwards: the second runs out of the caching allocator's free lists (the checker legs between
            # the measurements -- oracle torch ops, CUDA-graph capture -- leave them fragmented, and a forward that has
            # to cudaMalloc its operand buffers measured 3-6x slower than the same forward in a fresh process)
            for _ in range(2):
                logits = [model(dev_images[:bs])]
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            logits = [model(dev_images[i:i + bs]) for i in range(0, args.images_per_gpu, bs)]
            e1.record()
            torch.cuda.synchronize()
        return args.images_per_gpu / (e0.elapsed_time(e1) / 1e3), torch.cat(logits)

    fq_img_s, logits_ref = fq_rate(32)
    # checker: the same calibrated model with every quantizer forward evaluated by the oracle's torch ops on this GPU
    # (the reference's own forward composition): the default forward must reproduce it bit for bit
    fwd_parity = None
    if rank == 0 and not args.no_parity:
        for pth in (os.path.join(ROOT, 'oracle'), os.path.join(ROOT, 'tests')):
            if pth not in sys.path:
                sys.path.insert(0, pth)
        import _oracle_backend as fake
        from gpu_parity import _Patch
        mp = _Patch()
        try:
            from adalog_b200 import ops as _ops
            for name in ('uniform_fakequant', 'log_fakequant', 'twin_fakequant'):
                mp.setattr(_ops, name, getattr(fake, name))
            with torch.no_grad():
                ref_fwd = torch.cat([model(dev_images[i:i + 32]) for i in range(0, args.images_per_gpu, 32)])
        finally:
            mp.undo()
        fwd_parity = dict(default_forward_bit_identical_to_reference_forward=bool(torch.equal(ref_fwd, logits_ref)),
                          top1_agreement=float((ref_fwd.argmax(-1) == logits_ref.argmax(-1)).float().mean()),
                          max_abs_logit_diff=float((ref_fwd - logits_ref).abs().max()), images=int(ref_fwd.shape[0]),
                          what='calibrated model, default forward (sm_100a fake-quant kernels + FP32 products) vs the '
                               'same model with the quantizer forwards evaluated by the oracle\'s torch ops on this GPU')
    # the same default forward replayed from a CUDA graph (batch 32 is launch-latency bound)
    graphed_img_s, graphed_equal = None, None
    try:
        from adalog_b200.utils.graph import GraphedForward
        gf = GraphedForward(model, dev_images[:32])
        outs = []
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for i in range(0, args.images_per_gpu, 32):
            outs.append(gf(dev_images[i:i + 32]).clone())
        g1.record()
        torch.cuda.synchronize()
        graphed_img_s = args.images_per_gpu / (g0.elapsed_time(g1) / 1e3)
        graphed_equal = bool(torch.equal(torch.cat(outs), logits_ref))
        del gf
    except Exception as e:                              # reported, never fatal for the calibration metric
        graphed_equal = f'capture failed: {type(e).__name__}: {e}'[:200]
    torch.cuda.empty_cache()
    fq_big, _ = fq_rate(args.images_per_gpu)
    set_tensor_core_forward(model, True)
    fq_tc, logits_tc = fq_rate(32)
    fq_tc_big, _ = fq_rate(args.images_per_gpu)
    set_tensor_core_forward(model, False)
    fq_extra = dict(parity=fwd_parity, batch32_img_per_s=fq_img_s, batch32_cuda_graph_img_per_s=graphed_img_s,
                    batch32_cuda_graph_bit_identical=graphed_equal, full_batch_img_per_s=fq_big, tensor_core_batch32_img_per_s=fq_tc,
                    tensor_core_full_batch_img_per_s=fq_tc_big,
                    tensor_core_top1_agreement=float((logits_tc.argmax(-1) == logits_ref.argmax(-1)).float().mean()),
                    tensor_core_max_rel_logit_diff=float((logits_tc - logits_ref).abs().max() / logits_ref.abs().max()),
                    note='fakequant_img_per_s is the default forward (bit-identical to the reference composition). The '
                         'opt-in tensor-core forward equals it per layer to ~1e-6 of the output range (tests/'
                         'test_gpu_gemm.py, tests/gpu_tc_debug.py); end-to-end logits of a random-init low-bit network '
                         'amplify such rounding-level differences through 12 blocks of 3-bit rounding, so the '
                         'agreement figures here measure that sensitivity, not an error of either path')

    # ---- headline sub-record (BASELINE config 4: DeiT-B W4A4, 1024 images on 8 GPUs) when run on 8 GPUs
    headline = None
    if world == 8 and (args.config or 2) == 2 and not args.no_headline:
        hm, hb, himg = CONFIGS[4][0], CONFIGS[4][1], CONFIGS[4][2] // world
        h_step, _, _, h_evals = make_stepper(hm, hb, himg)
        h_sampler = ClockSampler(local) if rank == 0 else None
        h_ms, h_wall, _, h_model = h_step(False)
        h_clocks = h_sampler.stop() if h_sampler else None
        del h_model
        headline = dict(workload=f'{hm} W{hb}A{hb} FPCS calibration, {himg * world} synthetic images on {world} GPUs '
                                 f'({himg} per GPU), one calibration, no warm-up of its own',
                        baseline_config=4, calibration_wall_s=h_ms / 1e3, evaluations=h_evals,
                        candidates_per_s=world * 128 * h_evals / (h_ms / 1e3),
                        candidates_per_s_note='bench unit: one candidate scored on one rank\'s shard; '
                                              f'{128 * h_evals / (h_ms / 1e3):.0f} candidates/s counted on all {himg * world} images',
                        host_wall_s=h_wall / 1e3, clocks=h_clocks)

    # ---- checker leg (rank 0, one GPU): free-running parity against the reference-on-GPU, and its timing
    parity = gpu_reference = None
    if rank == 0 and world == 1 and not args.no_parity and (args.config or 2) in (1, 2) and args.model in ('deit_tiny', 'deit_small'):
        for pth in (os.path.join(ROOT, 'oracle'), os.path.join(ROOT, 'tests')):
            if pth not in sys.path:
                sys.path.insert(0, pth)
        from gpu_parity import run_parity
        slice_model = 'deit_tiny_patch16_224' if args.model == 'deit_tiny' else 'deit_small_depth1_patch16_224'
        rec = run_parity(slice_model, args.bits, args.images_per_gpu, with_ref64=False, log=lambda *_: None)
        parity = {k: rec[k] for k in (
            'model', 'bits', 'images', 'evaluations', 'forced_max_rel_diff', 'forced_max_rel_diff_patch_embed',
            'evaluations_over_1e5', 'evaluations_over_1e5_unexcused', 'forced_checkpoint_bit_identical',
            'forced_logits_bit_identical', 'topk_sets_differing', 'topk_sets_differing_outside_reference_noise',
            'worst_gap_over_reference_noise', 'exact_ties_in_reference', 'exact_ties_preserved',
            'free_running_quantizer_tensors_identical', 'quantizer_tensors_total', 'free_running_top1_agreement',
            'probe_images')}
        parity['what'] = ('tests/gpu_parity.py: oracle (pinned to the unmodified reference) on this GPU vs the CUDA sweeps, '
                          'teacher-forced (scores, ties, checkpoint) and free running (tensors identical, top-1); '
                          'patch embedding + block 0 + head of the bench model' if 'depth1' in slice_model else
                          'tests/gpu_parity.py on the whole model')
        parity['accuracy_vs_fp64_by_sweep'] = {k: dict(product=v['product_vs_fp64'], reference_fp32=v['ref32_vs_fp64'])
                                                for k, v in rec['by_sweep'].items()}
        gpu_reference = dict(kind='oracle port of the reference on the same B200 (torch-CUDA, FP32 like the reference; '
                                  'each evaluation additionally re-scored in FP64 for the noise measurement)',
                             model=slice_model, evaluations=rec['evaluations'], seconds=rec['reference_on_gpu_seconds'],
                             candidates_per_s=128 * rec['evaluations'] / rec['reference_on_gpu_seconds'],
                             product_seconds_same_slice=rec['product_seconds'],
                             product_candidates_per_s=128 * rec['evaluations'] / rec['product_seconds'])

    if rank == 0:
        cands = 128 * evals
        ms_step = statistics.mean(times)
        value = world * cands / (ms_step / 1e3)
        peaks = load_peaks()
        # int8 MMAs (tcgen05 kind::i8) run at twice the bf16 rate and MEASURED_PEAKS.json holds a bf16 peak only, so an
        # int8 operation counts as half a bf16 FLOP: `achieved` is bf16-equivalent TFLOP/s = tensor-pipe occupancy x peak
        bf_ops = gemm_split['bf16'][0] + lin_split['bf16'][0]
        i8_ops = gemm_split['i8'][0] + lin_split['i8'][0]
        achieved = (bf_ops + 0.5 * i8_ops) / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0

        def per_type(d):
            return {k: dict(launches=v[2], kernel_ms_per_step=v[1] / max(1, args.steps),
                            tera_ops_per_s=(v[0] / (v[1] / 1e3) / 1e12 if v[1] > 0 else 0.0)) for k, v in d.items()}
        traffic, traffic_note = ncu_traffic()
        out = dict(metric='fpcs_candidates_per_s', value=value, unit='candidates/s', n_gpus=world, steps=args.steps,
                   warmup=args.warmup, ms_per_step=ms_step, higher_is_better=True, scaling=args.scaling, vs_baseline=None,
                   dtype='int8 + bf16 operands holding exact integers (s32 / f32 accumulate), f64 error sums', data='synthetic',
                   config=workload_config(args), evaluations_per_step=evals, candidates_per_step=cands,
                   calibration_wall_s=ms_step / 1e3, fakequant_img_per_s=fq_img_s, fakequant_forward=fq_extra,
                   gpu_launches=launches, clocks=clocks,
                   roofline=dict(kernel='candidate GEMMs with fused error epilogue: cand_gemm_err_kernel (weight-side / '
                                        'conv sweeps) + lin_fused_kernel (activation-side sweeps, candidates generated '
                                        'in shared memory); both tcgen05 + TMEM + TMA',
                                 bound='tensor', achieved=achieved, peak=peaks['tflops'], unit='TFLOP/s',
                                 frac=achieved / peaks['tflops'] if peaks['tflops'] else None, traffic=traffic,
                                 traffic_note=traffic_note,
                                 peak_source=f"{peaks['src']} bf16_tflops_sustained",
                                 note='achieved = algorithmic 2*128*units*N*K ops of every launch / CUDA-event time of '
                                      'the launches inside the timed steps, in bf16-equivalent TFLOP/s (an int8 op '
                                      'counts 1/2: kind::i8 runs at 2x the bf16 rate; the measured peak is bf16)',
                                 cand_gemm_err_kernel=per_type(gemm_split), lin_fused_kernel=per_type(lin_split),
                                 launches=gemm_launches, kernel_ms_per_step=gemm_ms / max(1, args.steps),
                                 share_of_step=gemm_ms / max(1e-9, sum(times)),
                                 other_kernels=[dict(
                                     kernel='fused_cand_gemm_err_kernel (attention sweeps: candidates generated in '
                                            'shared memory + tcgen05 GEMM + error epilogue)',
                                     bound='CUDA-core issue slots: K = 64 per unit, so generating the 128 x K tile and '
                                           'reducing the 128 x N error cost more instructions than the MMA has clocks '
                                           '(DESIGN.md section 4; TMEM read-out measured at 320-440 B/clk/SM is not the bound)',
                                     launches=fz_launches, kernel_ms_per_step=fz_ms / max(1, args.steps),
                                     achieved=fz_flops / (fz_ms / 1e3) / 1e12 if fz_ms > 0 else 0.0, unit='TFLOP/s',
                                     share_of_step=fz_ms / max(1e-9, sum(times)))]))
        if e2e_ms is not None:
            out['e2e'] = dict(value=world * cands / (e2e_ms / 1e3), unit='candidates/s',
                              h2d_bytes_per_step=host_images.numel() * 4, d2h_bytes_per_step=d2h,
                              ms_per_step=e2e_ms)
        if headline is not None:
            out['headline'] = headline
        if parity is not None:
            out['parity'] = parity
            out['gpu_reference'] = gpu_reference
        if not args.no_cpu_baseline and world == 1 and args.model in DIMS:
            threads = os.cpu_count() or 1
            v, secs, c, per_type_s = cpu_arm_value(args.model, args.bits, 8, args.images_per_gpu, threads)
            out['cpu_baseline'] = dict(
                value=v, unit='candidates/s', cores=threads, kind='port',
                sample=f'oracle port of the reference CPU path, stratified: ONE evaluation (128 candidates) of each of '
                       f'the 21 sweep types of a {args.model} block on 8 images at the real layer sizes ({secs:.1f} s '
                       f'in total), each type weighted by its count in a calibration and scaled linearly to '
                       f'{args.images_per_gpu} images',
                seconds_per_sweep_type_on_8_images={k: round(t_, 4) for k, t_ in per_type_s.items()})
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
