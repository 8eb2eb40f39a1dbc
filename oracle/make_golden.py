"""Generate tests/golden/*.pt from the UNMODIFIED reference (run in the build container only).

TEST INFRASTRUCTURE ONLY.  Usage:  python oracle/make_golden.py   (needs /root/reference)

For every hot-path class of the reference (SURVEY.md section 8a) a small seeded case is driven exactly like
utils/calibrator.py:49-62 drives it; torch.topk is wrapped so that every search evaluation's
similarity tensor, k, dim and returned index list is recorded, together with the inputs and the final
state_dict.  tests/test_oracle_golden.py replays the same inputs through oracle/adalog_oracle.py and
demands bit equality (CPU vs CPU), which pins the oracle to the reference.
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_shim  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), 'tests', 'golden')


class TopkTap:
    """records every torch.topk (and, with argmax=True, every Tensor.argmax: the twin-uniform search of linear.py:691
    selects with argmax) as (similarities, k, dim, indices)"""

    def __init__(self, argmax=False):
        self.evals = []
        self._orig = torch.topk
        self._orig_argmax = torch.Tensor.argmax
        self._argmax = argmax

    def __enter__(self):
        def tapped(inp, k, dim=-1, **kw):
            res = self._orig(inp, k=k, dim=dim, **kw)
            self.evals.append(dict(sims=inp.detach().clone(), k=k, dim=dim, idx=res[1].clone()))
            return res
        torch.topk = tapped
        if self._argmax:
            orig = self._orig_argmax

            def tapped_argmax(t, *a, **kw):
                res = orig(t, *a, **kw)
                self.evals.append(dict(sims=t.detach().clone(), k=1, dim=kw.get('dim', a[0] if a else None),
                                       idx=res.clone(), argmax=True))
                return res
            torch.Tensor.argmax = tapped_argmax
        return self

    def __exit__(self, *a):
        torch.topk = self._orig
        torch.Tensor.argmax = self._orig_argmax


def lnlike(*shape):
    """LayerNorm-output-like activations: per-channel spread + offset."""
    c = shape[-1]
    return torch.randn(*shape) * (torch.rand(c) * 2) + 0.3 * torch.randn(c)


def save(name, obj):
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + '.pt')
    torch.save(obj, path)
    print(f'{name}: {len(obj.get("evals", []))} evals, {os.path.getsize(path) / 1024:.0f} KiB')


def sd(module):
    return {k: v.detach().clone() for k, v in module.state_dict().items()}


def run_linear(name, cls_name, in_f, out_f, x, w_bit, a_bit, n_V=1, bs=4, total_memory=None, bias=True, seed=0,
               fpcs=True, **extra):
    import quant_layers
    ref_shim.install(total_memory if total_memory is not None else 16 * 2 ** 30)
    cls = getattr(quant_layers, cls_name)
    m = cls(in_f, out_f, bias=bias, w_bit=w_bit, a_bit=a_bit, calib_batch_size=bs, eq_n=128, fpcs=fpcs, steps=6,
            search_round=3, n_V=n_V, **extra)
    torch.manual_seed(seed + 100)
    torch.nn.init.trunc_normal_(m.weight, std=.02)
    m.weight.data *= (1 + torch.rand(out_f, 1) * 3)  # rows of unequal range
    if bias:
        m.bias.data = torch.randn(out_f) * 0.02
    rec = dict(kind=cls_name, cfg=dict(in_f=in_f, out_f=out_f, w_bit=w_bit, a_bit=a_bit, n_V=n_V, bs=bs, bias=bias,
                                      memory=ref_shim._Props.total_memory // 2, fpcs=fpcs, **extra),
               weight=m.weight.detach().clone(), bias=m.bias.detach().clone() if bias else None, x=x.clone())
    ln = None
    if cls_name == 'AsymmetricallyChannelWiseBatchingQuantLinear':
        ln = torch.nn.LayerNorm(in_f)
        ln.weight.data = 1 + 0.1 * torch.randn(in_f)
        ln.bias.data = 0.1 * torch.randn(in_f)
        m.prev_layer = ln
        rec['ln_weight'], rec['ln_bias'] = ln.weight.detach().clone(), ln.bias.detach().clone()
    with torch.no_grad(), TopkTap(argmax='Twin' in cls_name) as tap:
        m.raw_input = x
        m.raw_out = m(x)
        rec['raw_out'] = m.raw_out.clone()
        m.hyperparameter_searching()
        if ln is not None:
            m.reparam()
    rec['evals'] = tap.evals
    rec['state'] = sd(m)
    if ln is not None:
        rec['ln_weight_after'], rec['ln_bias_after'] = ln.weight.detach().clone(), ln.bias.detach().clone()
    # fake-quant forward of the calibrated module on the calibration input
    with torch.no_grad():
        m.mode = 'quant_forward'
        xin = m.raw_input if hasattr(m, 'raw_input') and m.raw_input is not None else x
        x_eval = x if ln is None else None
        if x_eval is not None:
            rec['quant_out'] = m(x_eval).clone()
        if hasattr(m, 'reparam_bias'):
            m.reparam_bias()
            rec['state_bias_reparamed'] = sd(m)
            rec['quant_out_bias_reparamed'] = m(x).clone()
    save(name, rec)


def run_matmul(name, post_softmax, A, B, A_bit, B_bit, H, bs=4, total_memory=None, hcw=True, quantizer='adalog'):
    import quant_layers
    ref_shim.install(total_memory if total_memory is not None else 16 * 2 ** 30)
    kw = dict(A_bit=A_bit, B_bit=B_bit, calib_batch_size=bs, search_round=3, eq_n=128, head_channel_wise=hcw,
              num_heads=H, fpcs=True, steps=6)
    if post_softmax:
        m = quant_layers.PostSoftmaxAsymmetricallyBatchingQuantMatMul(quantizer=quantizer, **kw)
    else:
        m = quant_layers.AsymmetricallyBatchingQuantMatMul(**kw)
    rec = dict(kind=type(m).__name__, cfg=dict(A_bit=A_bit, B_bit=B_bit, H=H, bs=bs, hcw=hcw, quantizer=quantizer,
                                              memory=ref_shim._Props.total_memory // 2), A=A.clone(), B=B.clone())
    with torch.no_grad(), TopkTap() as tap:
        m.raw_input = [A, B]
        m.raw_out = m(A, B)
        rec['raw_out'] = m.raw_out.clone()
        m.hyperparameter_searching()
    rec['evals'] = tap.evals
    rec['state'] = sd(m)
    with torch.no_grad():
        m.mode = 'quant_forward'
        rec['quant_out'] = m(A, B).clone()
    save(name, rec)


def run_conv(name, x, ic, oc, k, w_bit, bs=4):
    import quant_layers
    ref_shim.install(16 * 2 ** 30)
    m = quant_layers.AsymmetricallyBatchingQuantConv2d(ic, oc, k, stride=k, w_bit=w_bit, a_bit=8, calib_batch_size=bs,
                                                       search_round=3, eq_n=128, fpcs=True, steps=6)
    torch.manual_seed(7)
    m.weight.data = torch.randn_like(m.weight) * 0.05 * (1 + torch.rand(oc, 1, 1, 1) * 2)
    m.bias.data = torch.randn(oc) * 0.02
    rec = dict(kind=type(m).__name__, cfg=dict(ic=ic, oc=oc, k=k, w_bit=w_bit, bs=bs,
                                              memory=ref_shim._Props.total_memory // 2),
               weight=m.weight.detach().clone(), bias=m.bias.detach().clone(), x=x.clone())
    with torch.no_grad(), TopkTap() as tap:
        m.raw_input = x
        m.raw_out = m(x)
        rec['raw_out'] = m.raw_out.clone()
        m.hyperparameter_searching()
    rec['evals'] = tap.evals
    rec['state'] = sd(m)
    with torch.no_grad():
        m.mode = 'quant_forward'
        rec['quant_out'] = m(x).clone()
    save(name, rec)


def run_quantizers():
    """Known-answer vectors for every quantizer forward (SURVEY.md 8a rows Q1-Q5)."""
    ref_shim.install()
    import quantizers as Q
    torch.manual_seed(11)
    out = dict(kind='quantizers', cases=[])
    x = torch.randn(6, 5, 24) * 1.7
    xp = torch.softmax(3 * torch.randn(4, 2, 9, 9), dim=-1)
    xp[0, 0, 0, :3] = 0.0
    xg = torch.nn.functional.gelu(torch.randn(6, 5, 24) * 1.5)
    for bits in (3, 4, 6, 8):
        # uniform, per-tensor / per-channel / per-row / per-head broadcast, integer and non-integer zp
        for shape_tag, xs, sshape in (('tensor', x, (1,)), ('channel', x, (24,)), ('rows', x.view(2, 15, 24), (2, 15, 1)),
                                      ('head', xp, (1, 2, 1, 1))):
            q = Q.UniformQuantizer(n_bits=bits, symmetric=False, channel_wise=True)
            q.scale = torch.nn.Parameter(torch.rand(*sshape) * 0.2 + 0.05)
            zp = torch.randint(0, 2 ** bits, sshape).float()
            if shape_tag == 'tensor':
                zp = zp + 0.3  # exercises round_ste on a non-integer zero point
            q.zero_point = torch.nn.Parameter(zp)
            q.inited = True
            with torch.no_grad():
                out['cases'].append(dict(q='uniform', bits=bits, tag=shape_tag, x=xs.clone(), scale=q.scale.detach().clone(),
                                         zero_point=q.zero_point.detach().clone(), y=q(xs).clone()))
        qs = Q.UniformQuantizer(n_bits=bits, symmetric=True)
        qs.scale = torch.nn.Parameter(torch.tensor([0.11]))
        qs.inited = True
        with torch.no_grad():
            out['cases'].append(dict(q='uniform_sym', bits=bits, x=x.clone(), scale=qs.scale.detach().clone(), y=qs(x).clone()))
        for qv in (10, 23, 37, 50, 137):
            q = Q.AdaLogQuantizer(n_bits=bits)
            q.scale = torch.nn.Parameter(torch.ones(1, 1, 1, 1))
            q.q.data.copy_(torch.tensor([qv]))
            q.update_table()
            q.inited = True
            with torch.no_grad():
                out['cases'].append(dict(q='adalog', bits=bits, qv=qv, x=xp.clone(), scale=q.scale.detach().clone(),
                                         table1=q.table1.clone(), table2=q.table2.clone(), y=q(xp).clone()))
            for reparamed in (False, True):
                q = Q.ShiftAdaLogQuantizer(n_bits=bits)
                q.scale = torch.nn.Parameter(torch.tensor([2.3]))
                q.shift.data.copy_(torch.tensor(0.16997124254703522))
                q.q.data.copy_(torch.tensor([qv]))
                q.update_table()
                q.bias_reparamed.data.copy_(torch.tensor(reparamed))
                q.inited = True
                with torch.no_grad():
                    out['cases'].append(dict(q='shift_adalog', bits=bits, qv=qv, reparamed=reparamed, x=xg.clone(),
                                             scale=q.scale.detach().clone(), shift=q.shift.detach().clone(),
                                             table1=q.table1.clone(), table2=q.table2.clone(), y=q(xg).clone()))
        for nm, cls in (('log2', Q.Log2Quantizer), ('logsqrt2', Q.LogSqrt2Quantizer)):
            q = cls(n_bits=bits)
            q.scale = torch.nn.Parameter(torch.ones(1, 1, 1, 1))
            q.inited = True
            with torch.no_grad():
                out['cases'].append(dict(q=nm, bits=bits, x=xp.clone(), scale=q.scale.detach().clone(), y=q(xp).clone()))
        for nm, cls in (('shift_log2', Q.ShiftLog2Quantizer), ('shift_logsqrt2', Q.ShiftLogSqrt2Quantizer)):
            q = cls(n_bits=bits)
            q.scale = torch.nn.Parameter(torch.tensor([2.3]))
            q.shift.data.copy_(torch.tensor(0.16997124254703522))
            q.inited = True
            with torch.no_grad():
                out['cases'].append(dict(q=nm, bits=bits, x=xg.clone(), scale=q.scale.detach().clone(),
                                         shift=q.shift.detach().clone(), y=q(xg).clone()))
        q = Q.TwinUniformQuantizer(n_bits=bits)
        q.scale = torch.nn.Parameter(torch.tensor([[0.21], [0.16997124254703522 / 2 ** (bits - 1)]]))
        q.inited = True
        with torch.no_grad():
            out['cases'].append(dict(q='twin', bits=bits, x=xg.clone(), scale=q.scale.detach().clone(), y=q(xg).clone()))
    os.makedirs(OUT, exist_ok=True)
    torch.save(out, os.path.join(OUT, 'quantizers.pt'))
    print('quantizers:', len(out['cases']), 'cases', os.path.getsize(os.path.join(OUT, 'quantizers.pt')) // 1024, 'KiB')


def main():
    run_quantizers()
    torch.manual_seed(5)
    run_linear('linear_asym_w4a4', 'AsymmetricallyBatchingQuantLinear', 32, 24, lnlike(8, 10, 32), 4, 4)
    run_linear('linear_asym_w3a3_nv3', 'AsymmetricallyBatchingQuantLinear', 32, 36, lnlike(8, 10, 32), 3, 3, n_V=3)
    run_linear('linear_asym_w6a6_chunked', 'AsymmetricallyBatchingQuantLinear', 32, 24, lnlike(6, 10, 32), 6, 6,
               total_memory=2 * 4 * 64 * (8 * 4 * 10 * 32 + 16 * 4 * 10 * 24) + 64)  # -> parallel_eq_n = 64, ragged batch
    run_linear('linear_head_2d_w4a4', 'AsymmetricallyBatchingQuantLinear', 32, 20, lnlike(8, 32), 4, 4)
    run_linear('linear_swin4d_w4a4', 'AsymmetricallyBatchingQuantLinear', 16, 24, lnlike(8, 3, 3, 16), 4, 4)
    run_linear('linear_nobias_w4a4', 'AsymmetricallyBatchingQuantLinear', 16, 24, lnlike(8, 6, 16), 4, 4, bias=False)
    run_linear('linear_cw_reparam_w4a4_nv3', 'AsymmetricallyChannelWiseBatchingQuantLinear', 32, 36, lnlike(8, 10, 32),
               4, 4, n_V=3)
    run_linear('linear_cw_reparam_w3a3', 'AsymmetricallyChannelWiseBatchingQuantLinear', 32, 24, lnlike(8, 10, 32), 3, 3)
    xg = torch.nn.functional.gelu(lnlike(8, 10, 48))
    run_linear('linear_postgelu_w4a4', 'PostGeluLogBasedBatchingQuantLinear', 48, 24, xg, 4, 4, quantizer='adalog')
    run_linear('linear_postgelu_w3a3', 'PostGeluLogBasedBatchingQuantLinear', 48, 24, xg, 3, 3, quantizer='adalog')
    run_linear('linear_postgelu_w6a6', 'PostGeluLogBasedBatchingQuantLinear', 48, 24, xg, 6, 6, quantizer='adalog')
    q = torch.randn(8, 2, 10, 16) * (1 + torch.arange(2).view(1, 2, 1, 1))
    k = torch.randn(8, 2, 16, 10) * 1.3
    run_matmul('matmul_qk_a4', False, q, k, 4, 4, 2)
    run_matmul('matmul_qk_a3', False, q, k, 3, 3, 2)
    run_matmul('matmul_qk_a6_pooled', False, q, k, 6, 6, 2, hcw=False)
    p = torch.softmax(torch.randn(8, 2, 10, 10) * 2, dim=-1)
    v = torch.randn(8, 2, 10, 16) * (1 + torch.arange(2).view(1, 2, 1, 1))
    run_matmul('matmul_pv_s4a4', True, p, v, 4, 4, 2)
    run_matmul('matmul_pv_s3a3', True, p, v, 3, 3, 2)
    run_matmul('matmul_pv_s6a6', True, p, v, 6, 6, 2)
    run_conv('conv_patch_w4', torch.randn(8, 3, 16, 16), 3, 12, 4, 4)
    run_conv('conv_patch_w6', torch.randn(8, 3, 16, 16), 3, 12, 4, 6)




def main_round2():
    """non-default branches selectable by config string (SURVEY.md 8a rows L16, L19, M6): post-GELU search without
    FPCS, the fixed-base post-GELU / post-softmax quantizers, the PTQ4ViT twin-uniform baseline"""
    ref_shim.install()
    torch.manual_seed(6)
    xg = torch.nn.functional.gelu(lnlike(8, 10, 48))
    run_linear('linear_postgelu_nofpcs_w4a4', 'PostGeluLogBasedBatchingQuantLinear', 48, 24, xg, 4, 4, fpcs=False,
               quantizer='adalog')
    run_linear('linear_postgelu_log2_w4a4', 'PostGeluLogBasedBatchingQuantLinear', 48, 24, xg, 4, 4, quantizer='log2')
    run_linear('linear_postgelu_logsqrt2_w3a3', 'PostGeluLogBasedBatchingQuantLinear', 48, 24, xg, 3, 3,
               quantizer='logsqrt2')
    run_linear('linear_twin_w4a4', 'PostGeluTwinUniformBatchingQuantLinear', 48, 24, xg, 4, 4)
    run_linear('linear_twin_nofpcs_w3a3', 'PostGeluTwinUniformBatchingQuantLinear', 48, 24, xg, 3, 3, fpcs=False)
    p = torch.softmax(torch.randn(8, 2, 10, 10) * 2, dim=-1)
    v = torch.randn(8, 2, 10, 16) * (1 + torch.arange(2).view(1, 2, 1, 1))
    run_matmul('matmul_pv_log2_s4a4', True, p, v, 4, 4, 2, quantizer='log2')
    run_matmul('matmul_pv_logsqrt2_s4a4', True, p, v, 4, 4, 2, quantizer='logsqrt2')
    run_matmul('matmul_pv_logsqrt2_s6a6', True, p, v, 6, 6, 2, quantizer='logsqrt2')


# ------------------------------------------------------------------------------------------------ model level
def install_fake_timm():
    """Register a minimal `timm` so the reference's utils/wrap_net.py imports: its Attention / WindowAttention
    classes are the stand-ins of adalog_b200/utils/models.py (timm itself is not installable here)."""
    import types
    repo = os.path.dirname(HERE)
    if repo not in sys.path:
        sys.path.insert(0, repo)
    from adalog_b200.utils import models as zoo
    timm = types.ModuleType('timm')
    timm.create_model = zoo.create_model
    tm = types.ModuleType('timm.models')
    vt = types.ModuleType('timm.models.vision_transformer')
    vt.Attention, vt.Block = zoo.Attention, zoo.Block
    st = types.ModuleType('timm.models.swin_transformer')
    st.WindowAttention, st.SwinTransformerBlock, st.PatchMerging = zoo.WindowAttention, zoo.SwinTransformerBlock, zoo.PatchMerging
    timm.models, tm.vision_transformer, tm.swin_transformer = tm, vt, st
    sys.modules.update({'timm': timm, 'timm.models': tm, 'timm.models.vision_transformer': vt,
                        'timm.models.swin_transformer': st})
    return zoo


def sims_digest(t):
    import hashlib
    return hashlib.sha1(t.detach().contiguous().numpy().tobytes()).hexdigest()


def run_model(name, model_name, bits, n_img=8, bs=4, img=32):
    zoo = install_fake_timm()
    ref_shim.install(16 * 2 ** 30)
    import importlib
    wrap_net = importlib.import_module('utils.wrap_net')
    calibrator = importlib.import_module('utils.calibrator')
    cfg_mod = importlib.import_module(f'configs.{bits}bit')
    cfg = cfg_mod.Config()
    cfg.calib_size, cfg.calib_batch_size = n_img, bs
    torch.manual_seed(5)
    model = zoo.create_model(model_name).eval()
    init_state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    images = torch.randn(n_img, 3, img, img)
    loader = [(images[i:i + bs], torch.zeros(bs, dtype=torch.long)) for i in range(0, n_img, bs)]
    with torch.no_grad():
        fp_logits = model(images).clone()
    model = wrap_net.wrap_modules_in_net(model, cfg, reparam=True)
    order = [n for n, m in model.named_modules() if hasattr(m, 'calibrated')]
    with TopkTap() as tap:
        calibrator.QuantCalibrator(model, loader).batching_quant_calib()
    model = wrap_net.wrap_reparamed_modules_in_net(model)
    state_calib = sd(model)
    with torch.no_grad():
        logits = model(images).clone()
    for _, m in model.named_modules():          # test_quant.py:130-133 finish_training
        if hasattr(m, 'mode') and hasattr(m, 'reparam_bias'):
            m.reparam_bias()
    with torch.no_grad():
        logits_final = model(images).clone()
    evals = [dict(digest=sims_digest(e['sims']), shape=tuple(e['sims'].shape), k=e['k'], dim=e['dim'], idx=e['idx'])
             for e in tap.evals]
    save(name, pack_model_golden(dict(
        kind='model', model=model_name, bits=bits, n_img=n_img, bs=bs, init_state=init_state, images=images, order=order,
        fp_logits=fp_logits, evals=evals, state_calib=state_calib, logits=logits, state_final=sd(model),
        logits_final=logits_final, memory=ref_shim._Props.total_memory // 2)))


def pack_model_golden(g):
    """Keeps a model golden under 1 MB without dropping any value: every evaluation's top-k indices (candidate numbers,
    0..127) become uint8 views of one shared storage, and a state tensor equal to the one before it in init_state ->
    state_calib -> state_final is stored once.  torch.save writes shared storages once; the tests read the indices
    through .to(torch.int64)."""
    flat = torch.cat([e['idx'].reshape(-1) for e in g['evals']])
    assert int(flat.min()) >= 0 and int(flat.max()) < 256
    flat = flat.to(torch.uint8)
    o = 0
    for e in g['evals']:
        n = e['idx'].numel()
        e['idx'] = flat[o:o + n].view(e['idx'].shape)
        o += n
    prev = g['init_state']
    for key in ('state_calib', 'state_final'):
        st = g[key]
        for k, v in st.items():
            if k in prev and prev[k].dtype == v.dtype and prev[k].shape == v.shape and torch.equal(prev[k], v):
                st[k] = prev[k]
        prev = st
    return g


def main_models():
    run_model('model_vit_test_w4a4', 'vit_test_patch8_32', 4)
    run_model('model_swin_test_w4a4', 'swin_test_patch2_window4_32', 4)


if __name__ == '__main__':
    what = sys.argv[1] if len(sys.argv) > 1 else 'all'
    if what in ('layers', 'all'):
        main()
    if what in ('round2', 'all'):
        main_round2()
    if what in ('models', 'all'):
        main_models()
