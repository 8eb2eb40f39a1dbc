"""GPU helper (not a pytest file): per-module timing of one calibration.  python tests/gpu_profile_calib.py deit_small 3 128"""
import importlib
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from adalog_b200.utils.calibrator import QuantCalibrator  # noqa: E402

model_key, bits, n_img = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
cfg = importlib.import_module(f'adalog_b200.configs.{bits}bit').Config()
cfg.calib_size, cfg.calib_batch_size = n_img, 32
dev = torch.device('cuda', 0)
for rep in range(2):
    model = bench.build_wrapped(bench.MODEL_ALIASES[model_key], cfg, dev)
    images = torch.randn(n_img, 3, 224, 224, generator=torch.Generator().manual_seed(5)).to(dev)
    loader = [(images[i:i + 32], None) for i in range(0, n_img, 32)]
    cal = QuantCalibrator(model, loader)
    cal.progress = False
    cal.timing = True
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    cal.batching_quant_calib()
    torch.cuda.synchronize()
    print(f'rep {rep}: total {time.perf_counter() - t0:.2f} s')
agg = {}
for name, (c, s) in cal.timings.items():
    kind = name.split('.')[-1]
    a = agg.setdefault(kind, [0, 0.0, 0.0])
    a[0] += 1; a[1] += c; a[2] += s
print('kind        n  capture_s  search_s')
for k, (n, c, s) in agg.items():
    print(f'{k:10s} {n:3d}  {c:8.2f}  {s:8.2f}')
