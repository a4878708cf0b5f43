"""CPU-side tests (-m "not gpu"): the C-ABI library loads and exports every symbol the header
declares (no compute calls), and the host logic of the engine (argument system, LR schedule,
ramp-up, CutMix mask generator, flat parameter arena, plugin registration) behaves like the
reference."""
import ctypes
import gzip
import json
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, 'tests', 'golden')


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as ge
    ge.build()
    from pixelssl_b200 import _lib
    header = open(os.path.join(ROOT, 'include', 'pixelssl_b200.h')).read()
    declared = set(re.findall(r'\b(pxl_[a-z0-9_]+)\s*\(', header))
    declared -= {'pxl_conv_geom'}
    assert declared, 'no declarations parsed'
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), 'missing export: ' + name
    # the ctypes table covers exactly the header
    assert set(_lib.SIGNATURES) == declared
    assert _lib.load().pxl_abi_version() == 3
    # ... with the same number of parameters per entry point (a pointer passed in the wrong slot is silent in ctypes)
    text = re.sub(r'/\*.*?\*/', ' ', header, flags=re.S)
    for name in sorted(declared):
        m = re.search(r'\b' + name + r'\s*\(([^;{]*?)\)\s*;', text, flags=re.S)
        assert m, 'declaration of %s not found' % name
        params = m.group(1).strip()
        n = 0 if params in ('', 'void') else params.count(',') + 1
        assert n == len(_lib.SIGNATURES[name][1]), '%s: header declares %d parameters, _lib.SIGNATURES %d' % (
            name, n, len(_lib.SIGNATURES[name][1]))


def test_ops_fail_loudly_without_cuda():
    from pixelssl_b200 import ops
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    with pytest.raises(TypeError):
        ops.mse_consistency_raw(torch.zeros(8), torch.zeros(8))


def test_rampup_and_poly_lr_match_golden():
    from pixelssl_b200.nn import func, lrer
    g = np.load(os.path.join(G, 'ops.npz'))
    mine = [func.sigmoid_rampup(c, 30) for c in range(0, 40, 3)] + [func.sigmoid_rampup(5, 0)]
    np.testing.assert_allclose(mine, g['rampup'], rtol=1e-12)
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([{'params': [p], 'lr': 0.00025}], lr=0.00025, momentum=0.9)
    sch = lrer.PolynomialLR(opt, epochs=2, iters_per_epoch=5, power=0.9)
    lrs = [opt.param_groups[0]['lr']]
    for _ in range(8):
        opt.step()
        sch.step()
        lrs.append(opt.param_groups[0]['lr'])
    np.testing.assert_allclose(lrs, g['poly_lr'], rtol=1e-12)


def test_box_mask_generator_bit_exact():
    from pixelssl_b200.ssl_algorithm.ssl_cutmix import BoxMaskGenerator
    g = np.load(os.path.join(G, 'ops.npz'))
    np.random.seed(1234)
    masks = BoxMaskGenerator((0.5, 0.5)).produce(4, (65, 97))
    assert masks.dtype == np.float32 and np.array_equal(masks, g['cutmix_masks'])
    np.random.seed(99)
    full = BoxMaskGenerator((0.25, 0.5)).produce(3, (513, 513))
    assert np.array_equal(full.reshape(3, 513, 513)[:, ::8, ::8], g['cutmix_masks_b'])
    assert np.array_equal(full.reshape(3, -1).sum(1), g['cutmix_masks_b_sum'])
    # empty / degenerate: zero masks requested
    assert BoxMaskGenerator((0.5, 0.5)).produce(0, (9, 9)).shape == (0, 1, 9, 9)


def test_build_args_and_autoset_fields():
    import pixelssl_b200
    a = pixelssl_b200.build_args({'ssl_algorithm': 'ssl_mt', 'cons_for_labeled': False, 'cons_scale': 1.0,
                                  'cons_rampup_epochs': 3, 'ema_decay': 0.99, 'lr': 0.00025, 'momentum': 0.9,
                                  'weight_decay': 0.0005, 'epochs': 20, 'batch_size': 16, 'unlabeled_batch_size': 8,
                                  'models': {'model': 'deeplabv2'}}, iters_per_epoch=7)
    assert (a.labeled_batch_size, a.iters_per_epoch, a.is_epoch_lrer, a.num_classes, a.ignore_index) == (8, 7, False, 21, 255)
    assert a.cons_for_labeled is False and a.models == {'model': 'deeplabv2'}
    with pytest.raises(SystemExit):     # log_err convention: print + exit
        pixelssl_b200.create_parser('ssl_unknown')


def test_param_arena_layout_and_segments():
    from pixelssl_b200.nn.arena import ParamArena
    from pixelssl_b200.nn.modules import Conv2d, BatchNorm2d
    net = torch.nn.Sequential(Conv2d(3, 8, 3, bias=False), BatchNorm2d(8), Conv2d(8, 5, 1, bias=True))
    ref = {n: p.detach().clone() for n, p in net.named_parameters()}
    arena = ParamArena(net)
    for n, p in net.named_parameters():
        assert torch.equal(p, ref[n])                      # values preserved
        assert p.data_ptr() >= arena.data.data_ptr() and p.grad is not None
        if p.dim() == 4:
            assert p.is_contiguous(memory_format=torch.channels_last)
    # a 3x3 weight written through the parameter lands [Cout][kh][kw][Cin] in the flat buffer
    w = net[0].weight
    w.data[1, 2, 0, 1] = 42.0
    assert arena.data[arena.offsets[0] + ((1 * 3 + 0) * 3 + 1) * 3 + 2] == 42.0
    # gradient accumulation from autograd lands in the flat gradient buffer
    arena.zero_grad()
    (w * 2).sum().backward()
    assert float(arena.grad[:w.numel()].sum()) == 2.0 * w.numel()
    groups = [list(net[0].parameters()) + list(net[1].parameters()), list(net[2].parameters())]
    segs = [arena.segments(g) for g in groups]
    assert segs[0] == [(0, arena.offsets[3])] and segs[1][0][0] == arena.offsets[3]
    assert sum(b - a for s in segs for a, b in s) == arena.numel


def _reference_host():
    """What the unmodified reference returned for the host-side comparisons below (oracle/make_golden.py host)."""
    with open(os.path.join(G, 'reference_host.json')) as f:
        return json.load(f)


def _as_json(value):
    """``value`` as it reads back from the JSON golden (tuples become lists)."""
    return json.loads(json.dumps(value))


def _parser_table(parser, option_strings=True):
    return {a.dest: (a.default, getattr(a.type, '__name__', a.type), a.choices) + ((tuple(a.option_strings),) if option_strings else ())
            for a in parser._actions if a.dest != 'help'}


def _checkpoint_keys(src):
    """Top-level keys of the ``state`` dict an algorithm's ``_save_checkpoint`` writes, read from its source."""
    body = src[src.index('def _save_checkpoint'):]
    body = body[body.index('state = {'):]
    body = body[:body.index('}') + 1]
    return sorted(set(re.findall(r"'([a-z_]+)'\s*:", body)))


def _lr_trajectory(mod, name):
    """Per-group learning rates of ``mod``'s scheduler ``name`` on a toy two-group optimizer, parser defaults."""
    import argparse
    parser = argparse.ArgumentParser()
    mod.add_parser_arguments(parser)
    args = parser.parse_args([])
    args.epochs, args.iters_per_epoch = 6, 4
    w = [torch.nn.Parameter(torch.zeros(2)), torch.nn.Parameter(torch.zeros(2))]
    opt = torch.optim.SGD([{'params': [w[0]], 'lr': 0.1}, {'params': [w[1]], 'lr': 1.0}], lr=0.1, momentum=0.9)
    sched = getattr(mod, name)(args)(opt)
    traj = []
    steps = args.epochs * args.iters_per_epoch - 1 if name == 'polynomiallr' else args.epochs
    for _ in range(steps):
        traj.append([g['lr'] for g in opt.param_groups])
        opt.step()
        sched.step()
    return traj


def _optimizer_summary(mod, name):
    """Class and per-group hyper-parameters of the optimizer ``mod``'s export ``name`` builds with parser defaults."""
    import argparse
    parser = argparse.ArgumentParser()
    mod.add_parser_arguments(parser)
    args = parser.parse_args(['--lr', '0.00025'])
    w = [torch.nn.Parameter(torch.zeros(2)), torch.nn.Parameter(torch.zeros(3))]
    groups = [{'params': [w[0]], 'lr': args.lr}, {'params': [w[1]], 'lr': 10 * args.lr}]
    opt = getattr(mod, name)(args)(groups)
    return {'class': type(opt).__module__ + '.' + type(opt).__qualname__,
            'groups': [{k: v for k, v in g.items() if k != 'params'} for g in opt.param_groups]}


SHAPE_HOOKS = ('sslcct_ad_in_channels', 'sslcct_ad_out_channels', 'sslcct_ad_upsample_scale', 'sslgct_fd_in_channels',
               'ssladv_fcd_in_channels', 'ssls4l_rc_in_channels')


def test_register_into_unmodified_pixelssl():
    """register_into_pixelssl on a package laid out like the unmodified pixelssl (the attributes its runner and
    TaskProxy look up by name): algorithm modules and the sampler class are replaced, and the rank-aware sampler
    yields the reference sampler's index stream at world size 1 (golden).  The unmodified package itself is not
    imported, so that its real module layout and ``runner.create_parser`` accept the engine's modules is not checked
    here; the stand-in restates the name lookups of pixelssl/runner.py:22 and task_template/proxy.py:433-434."""
    import argparse
    import types
    import pixelssl_b200
    ref = _reference_host()['register']
    pixelssl = types.SimpleNamespace(ssl_algorithm=types.ModuleType('pixelssl.ssl_algorithm'),
                                     nn=types.SimpleNamespace(data=types.ModuleType('pixelssl.nn.data')))
    pixelssl.ssl_algorithm.SSL_ALGORITHMS = list(ref['ssl_algorithms'])
    pixelssl.nn.data.TwoStreamBatchSampler = None
    pixelssl_b200.register_into_pixelssl(pixelssl)
    for name in pixelssl_b200.SSL_ALGORITHMS:
        mod = pixelssl.ssl_algorithm.__dict__[name]
        assert mod.__name__.startswith('pixelssl_b200.')
        assert callable(getattr(mod, name)) and callable(mod.add_parser_arguments)
        assert name in pixelssl.ssl_algorithm.SSL_ALGORITHMS
    # the proxy's sampler lookup (pixelssl.nn.data.TwoStreamBatchSampler) now resolves to the rank-aware one,
    # which at world size 1 yields exactly what the reference's own class yields
    assert pixelssl.nn.data.TwoStreamBatchSampler.__module__ == 'pixelssl_b200.nn.data'
    np.random.seed(5)
    got = [list(map(int, b)) for b in pixelssl.nn.data.TwoStreamBatchSampler(list(range(9)), list(range(50, 83)), 2, 3)]
    assert got == ref['sampler_seed5'] and len(got) == 11
    # the reference's parser builder looks the algorithm module up by name (pixelssl/runner.py:22)
    parser = argparse.ArgumentParser()
    pixelssl.ssl_algorithm.__dict__['ssl_mt'].add_parser_arguments(parser)
    ns = parser.parse_args(['--cons-scale', '1.0', '--ema-decay', '0.99'])
    assert ns.cons_scale == 1.0 and ns.ema_decay == 0.99


def test_two_stream_sampler_matches_reference_streams():
    """World size 1: the index stream equals the reference sampler's (golden, 3 epochs, seeded np.random).
    World size 2: the two ranks partition every reference GLOBAL batch, labeled-first per rank."""
    from pixelssl_b200.nn.data import TwoStreamBatchSampler
    g = np.load(os.path.join(G, 'val.npz'))
    for c, (nl, nu, lb, ub) in enumerate(g['sampler_cfgs']):
        lab, unl = list(range(nl)), list(range(1000, 1000 + nu))
        np.random.seed(100 + c)
        smp = TwoStreamBatchSampler(lab, unl, int(lb), int(ub), rank=0, world_size=1)
        for e in range(3):
            want = g['sampler_%d_epoch%d' % (c, e)]
            got = np.array([list(map(int, b)) for b in smp], dtype=np.int64).reshape(want.shape)
            assert len(smp) == len(want)
            assert np.array_equal(got, want), (c, e)
        if lb % 2 or ub % 2:
            continue
        hl, hu = int(lb) // 2, int(ub) // 2
        per_rank = []
        for r in range(2):
            np.random.seed(100 + c)
            s2 = TwoStreamBatchSampler(lab, unl, hl, hu, rank=r, world_size=2)
            per_rank.append([[list(map(int, b)) for b in s2] for _ in range(3)])
        for e in range(3):
            want = g['sampler_%d_epoch%d' % (c, e)]
            for k, gb in enumerate(want):
                L, U = list(gb[:lb]), list(gb[lb:])
                for r in range(2):
                    assert per_rank[r][e][k] == L[r * hl:(r + 1) * hl] + U[r * hu:(r + 1) * hu]


def test_two_stream_sampler_private_seed_and_errors():
    from pixelssl_b200.nn.data import TwoStreamBatchSampler
    a = TwoStreamBatchSampler(list(range(20)), list(range(100, 160)), 2, 3, rank=1, world_size=2, seed=9)
    b = TwoStreamBatchSampler(list(range(20)), list(range(100, 160)), 2, 3, rank=1, world_size=2, seed=9)
    assert [list(x) for x in a] == [list(x) for x in b]
    assert all(len(x) == 5 and all(i < 100 for i in x[:2]) and all(i >= 100 for i in x[2:]) for x in a)
    with pytest.raises(ValueError):
        TwoStreamBatchSampler([0, 1], [2, 3], 1, 1, rank=2, world_size=2)
    with pytest.raises(AssertionError):
        TwoStreamBatchSampler([0, 1], [2, 3, 4, 5], 2, 1, rank=0, world_size=2)


def test_summarize_confusion_matrix_matches_golden():
    from pixelssl_b200.task.sseg.func import summarize_confusion_matrix
    g = np.load(os.path.join(G, 'val.npz'))
    for k in range(2):
        v = summarize_confusion_matrix(g['metrics_cmat_sum%d' % k])
        got = np.array([v['acc'], v['acc-class'], v['mIoU'], v['fwIoU']])
        np.testing.assert_allclose(got, g['metrics_values%d' % k], rtol=1e-12)


def test_device_prefetch_falls_back_to_plain_iteration_without_cuda():
    from pixelssl_b200.ssl_algorithm import ssl_base
    if torch.cuda.is_available():
        pytest.skip('GPU present: the CUDA path is covered by the gpu tests')
    batches = [((torch.full((2, 3), float(i)),), (torch.full((2, 1), float(-i)),)) for i in range(4)]
    got = list(ssl_base.device_prefetch(batches))
    assert len(got) == 4
    for (gi, gg), (bi, bg) in zip(got, batches):
        assert gi[0] is bi[0] and gg[0] is bg[0]
    assert list(ssl_base.device_prefetch([])) == []


def test_deferred_step_log_prints_same_text_one_interval_late(monkeypatch):
    """_SSLBase._log_step: line k is emitted at call k+1 (or at flush) with the values it had at call k."""
    from pixelssl_b200.ssl_algorithm import ssl_base
    from pixelssl_b200.utils import logger
    emitted = []
    monkeypatch.setattr(logger, 'log_info', lambda msg: emitted.append(msg))
    alg = ssl_base._SSLBase(args=None)
    for k in range(3):
        alg.meters.update('task_loss', float(k) + 0.5)
        alg._log_step(lambda m, a=(k,): 'step {0}: {meters[task_loss]:.3f}'.format(*a, meters=m))
        assert len(emitted) == k                      # nothing for this step yet
    alg._flush_log()
    assert emitted == ['step 0: 0.500 (0.500)', 'step 1: 1.500 (1.000)', 'step 2: 2.500 (1.500)']
    alg._flush_log()
    assert len(emitted) == 3


TASK_MODELS = [('deeplabv2', 'resnet101'), ('pspnet', 'resnet50'), ('pspnet', 'resnet101')]


def _task_model_layout(model_mod, name, backbone):
    """state_dict keys / shapes / dtypes and the LR groups (as parameter names) of ``model_mod``'s task model."""
    from pixelssl_b200 import runner
    args = runner.build_args({'ssl_algorithm': 'ssl_null', 'lr': 0.00025, 'momentum': 0.9, 'weight_decay': 0.0005,
                              'epochs': 2, 'batch_size': 2, 'unlabeled_batch_size': 0, 'ignore_unlabeled': True,
                              'backbone': backbone}, iters_per_epoch=5)
    m = getattr(model_mod, name)()(args)
    sd = m.state_dict()
    pname = {id(p): n for n, p in m.named_parameters()}
    return {'keys': list(sd.keys()), 'shapes': [list(v.shape) for v in sd.values()], 'dtypes': [str(v.dtype) for v in sd.values()],
            'group_lrs': [g['lr'] for g in m.param_groups], 'group_params': [[pname[id(p)] for p in g['params']] for g in m.param_groups]}


@pytest.mark.parametrize('name,backbone', TASK_MODELS)
def test_task_model_state_dict_and_param_groups_match_reference(name, backbone):
    """Checkpoint compatibility (SURVEY 8f rank 3): same state_dict keys, shapes and dtypes as the reference task
    model (so its .ckpt files load), same LR groups in the same order (task/sseg/model.py:45-48,103-107)."""
    from pixelssl_b200.task.sseg import model as eng_model
    with gzip.open(os.path.join(G, 'reference_task_models.json.gz'), 'rt') as f:
        ref = json.load(f)['%s-%s' % (name, backbone)]
    eng = _task_model_layout(eng_model, name, backbone)
    assert eng['keys'] == ref['keys']
    for k, rs, es, rd, ed in zip(ref['keys'], ref['shapes'], eng['shapes'], ref['dtypes'], eng['dtypes']):
        assert rs == es and rd == ed, k
    assert eng['group_lrs'] == ref['group_lrs']
    assert eng['group_params'] == ref['group_params']


SSL_ALGS = ['ssl_null', 'ssl_mt', 'ssl_cutmix', 'ssl_adv', 'ssl_gct', 'ssl_cct']


@pytest.mark.parametrize('alg', SSL_ALGS)
def test_checkpoint_dict_keys_match_reference(alg):
    """Every algorithm saves the same top-level checkpoint keys as the reference's ``_save_checkpoint``
    (e.g. ssl_mt.py:296-307), so checkpoints are interchangeable between the two."""
    ref = _reference_host()['checkpoint_keys'][alg]
    with open(os.path.join(ROOT, 'pixelssl_b200', 'ssl_algorithm', '%s.py' % alg)) as f:
        eng = _checkpoint_keys(f.read())
    assert ref == eng and 'algorithm' in eng and 'epoch' in eng


@pytest.mark.parametrize('alg', SSL_ALGS)
def test_algorithm_parser_arguments_match_reference(alg):
    """add_parser_arguments of every algorithm module: same options, defaults, types and choices as the
    reference's (e.g. ssl_mt.py:27-38), so its scripts/configs parse identically."""
    import argparse
    from pixelssl_b200 import ssl_algorithm as eng
    pe = argparse.ArgumentParser()
    getattr(eng, alg).add_parser_arguments(pe)
    assert _reference_host()['parser_table'][alg] == _as_json(_parser_table(pe))


def test_full_argument_set_matches_reference_runner_and_sseg_proxy():
    """runner.create_parser + the proxy/task arguments: every option the reference's ``pixelssl.runner.create_parser``
    + ``task/sseg/proxy.add_parser_arguments`` defines exists here with the same default and type."""
    from pixelssl_b200 import runner as er
    # ssl_null: its options are the same in both implementations (tested above)
    pe = er.create_parser('ssl_null')
    er.add_proxy_arguments(pe)
    te = _parser_table(pe, option_strings=False)
    # engine-only option: the reference hard-codes the pretrained-backbone URL per backbone (task/sseg/model.py:69-80);
    # the engine exposes the same choice as a flag whose default 'auto' resolves to exactly those URLs
    assert te.pop('pretrained_backbone') == ('auto', 'str', None)
    assert _reference_host()['full_parser_table'] == _as_json(te)


LR_SCHEDULERS = ['steplr', 'multisteplr', 'exponentiallr', 'cosineannealinglr', 'polynomiallr']


@pytest.mark.parametrize('name', LR_SCHEDULERS)
def test_lr_scheduler_wrappers_follow_the_reference(name):
    """Every lrer export yields the reference's learning-rate trajectory (pixelssl/nn/lrer.py:51-179) on a toy
    two-group optimizer, including the per-scheduler defaults behind the parser's -1 placeholders."""
    from pixelssl_b200.nn import lrer as eng
    np.testing.assert_allclose(_lr_trajectory(eng, name), _reference_host()['lr_trajectory'][name], rtol=1e-12)


_BASE_CFG = {'lr': 0.00025, 'momentum': 0.9, 'weight_decay': 0.0005, 'epochs': 20, 'log_freq': 10 ** 6,
             'batch_size': 16, 'unlabeled_batch_size': 8}
_VALID = {
    'ssl_mt': {'cons_scale': 1.0, 'cons_rampup_epochs': 3},
    'ssl_cutmix': {'cons_scale': 20.0, 'cons_rampup_epochs': 0, 'cons_threshold': 0.97},
    'ssl_adv': {'adv_for_labeled': True, 'labeled_adv_scale': 0.01, 'unlabeled_adv_scale': 0.001, 'discriminator_scale': 1.0},
    'ssl_gct': {'fc_ssl_scale': 1.0, 'dc_ssl_scale': 100.0, 'dc_threshold': 0.6, 'dc_rampup_epochs': 5, 'mu': 0.5, 'nu': 1,
                'im_size': 65},
    'ssl_cct': {'cons_scale': 30.0, 'cons_rampup_epochs': 5, 'ad_lr_scale': 10.0},
}
_CASES = [(alg, None) for alg in _VALID] + [
    ('ssl_mt', {'cons_scale': -1.0}), ('ssl_mt', {'cons_rampup_epochs': -1}),
    ('ssl_cutmix', {'cons_threshold': -1.0}), ('ssl_cutmix', {'unlabeled_batch_size': 2, 'batch_size': 4}),
    ('ssl_cutmix', {'cons_scale': -1.0}),
    ('ssl_adv', {'labeled_adv_scale': -1.0}), ('ssl_adv', {'unlabeled_adv_scale': -1.0}),
    ('ssl_gct', {'dc_threshold': -1.0}), ('ssl_gct', {'mu': -1.0}), ('ssl_gct', {'nu': -1}),
    ('ssl_gct', {'fc_ssl_scale': -1.0}), ('ssl_gct', {'dc_rampup_epochs': -1}),
    ('ssl_cct', {'cons_scale': -1.0}), ('ssl_cct', {'cons_rampup_epochs': -1}), ('ssl_cct', {'ad_lr_scale': -1.0}),
]
_CLASSES = {'ssl_mt': 'SSLMT', 'ssl_cutmix': 'SSLCUTMIX', 'ssl_adv': 'SSLADV', 'ssl_gct': 'SSLGCT', 'ssl_cct': 'SSLCCT'}


def _case_id(alg, override):
    return alg + ' ' + json.dumps(override, sort_keys=True)


def _constructor_rejects(mod, alg, override):
    """True if ``mod``'s algorithm class refuses the configuration (``log_err``: banner + exit)."""
    from pixelssl_b200 import runner
    cfg = dict(_BASE_CFG, ssl_algorithm=alg, **_VALID[alg])
    cfg.update(override or {})
    try:
        getattr(mod, _CLASSES[alg])(runner.build_args(cfg, iters_per_epoch=5))
        return False
    except SystemExit:
        return True


@pytest.mark.parametrize('alg,override', _CASES)
def test_algorithm_constructors_validate_arguments_like_the_reference(alg, override, capsys):
    """``log_err`` (banner + exit) for the same unset / invalid SSL arguments as the reference's ``__init__`` checks
    (e.g. ssl_mt.py:76-92, ssl_cutmix.py:79-94), acceptance of the shipped-script values."""
    import importlib
    want = _reference_host()['constructor_rejects'][_case_id(alg, override)]
    got = _constructor_rejects(importlib.import_module('pixelssl_b200.ssl_algorithm.' + alg), alg, override)
    capsys.readouterr()
    assert got == want, 'reference rejects: %s, engine rejects: %s' % (want, got)
    if override is None:
        assert not got


def _task_func_args(arch):
    from pixelssl_b200 import runner
    return runner.build_args(dict(_BASE_CFG, ssl_algorithm='ssl_cct', models={'model': arch}, im_size=65, **_VALID['ssl_cct']),
                             iters_per_epoch=5)


@pytest.mark.parametrize('arch', ['deeplabv2', 'pspnet'])
def test_task_func_shape_hooks_match_reference(arch):
    """The scalar TaskFunc hooks the algorithms size their auxiliary networks with (task/sseg/func.py:134-253)."""
    from pixelssl_b200.task.sseg import func as eng_func
    ref = _reference_host()['task_func'][arch]
    eng = eng_func.task_func()(_task_func_args(arch))
    for hook in SHAPE_HOOKS:
        assert _as_json(getattr(eng, hook)()) == ref[hook], hook
    assert eng.METRIC_STR == ref['METRIC_STR']


OPTIMIZER_KEYS = {'sgd': ('lr', 'momentum', 'dampening', 'weight_decay', 'nesterov'),
                  'adam': ('lr', 'betas', 'eps', 'weight_decay')}


@pytest.mark.parametrize('name', ['sgd', 'adam'])
def test_optimizer_wrappers_build_the_reference_optimizer(name):
    """optimizer export functions (pixelssl/nn/optimizer.py:57-123): same torch optimizer class and the same
    hyper-parameters in every param group, including the defaults behind the parser's -1 placeholders."""
    from pixelssl_b200.nn import optimizer as eng
    ref = _reference_host()['optimizer'][name]
    got = _as_json(_optimizer_summary(eng, name))
    assert got['class'] == ref['class'] and len(got['groups']) == len(ref['groups'])
    # the hyper-parameters the reference sets (pixelssl/nn/optimizer.py); other keys are torch's own defaults and
    # change between torch versions
    for rg, eg in zip(ref['groups'], got['groups']):
        for k in OPTIMIZER_KEYS[name]:
            assert eg[k] == rg[k], (k, eg[k], rg[k])


def test_pretrained_backbone_url_resolution_and_key_filtered_load(tmp_path, monkeypatch):
    """--pretrained-backbone: 'auto' resolves to the URLs the reference hard-codes (task/sseg/model.py:69-80), 'none'
    keeps the initialisers; a zoo checkpoint found in the local cache is loaded key-filtered like resnet.py:145-156
    (torchvision layout: extra ``fc.*`` entries are dropped, backbone entries overwrite the initialisers)."""
    import argparse
    import torch
    from pixelssl_b200.task.sseg import model as M
    from pixelssl_b200.task.sseg.module import resnet as R
    ns = argparse.Namespace(backbone='resnet101', pretrained_backbone='auto')
    assert M.pretrained_backbone_url(ns) == 'https://download.pytorch.org/models/resnet101-5d3b4d8f.pth'
    ns.backbone = 'resnet101-coco'
    assert M.pretrained_backbone_url(ns).endswith('resnet101COCO-41f33a49.pth')
    ns.pretrained_backbone = 'none'
    assert M.pretrained_backbone_url(ns) is None
    ns.pretrained_backbone = '/some/file.pth'
    assert M.pretrained_backbone_url(ns) == '/some/file.pth'
    # synthetic torchvision-layout checkpoint for a ResNet-50 in the cache directory
    net = R.ResNet([3, 4, 6, 3], 16)
    g = torch.Generator().manual_seed(0)
    fake = {k: torch.randn(v.shape, generator=g) if v.is_floating_point() else v.clone() for k, v in net.state_dict().items()}
    fake['fc.weight'] = torch.randn(1000, 2048, generator=g)
    fake['fc.bias'] = torch.randn(1000, generator=g)
    torch.save(fake, tmp_path / 'resnet50-19c8e357.pth')
    monkeypatch.setenv('PXL_PRETRAINED_DIR', str(tmp_path))
    net2 = R.ResNet([3, 4, 6, 3], 16, pretrained_url=M.PRETRAINED_BACKBONE_URLS['resnet50'])
    for k, v in net2.state_dict().items():
        assert torch.equal(v, fake[k]), k
    assert net2.conv1.weight.is_contiguous(memory_format=torch.channels_last)
    # requested but unobtainable: an error, not a silent random init
    monkeypatch.setenv('PXL_PRETRAINED_DIR', str(tmp_path / 'nowhere'))
    monkeypatch.setattr(torch.hub, 'get_dir', lambda: str(tmp_path / 'nohub'))
    monkeypatch.setattr(torch.hub, 'load_state_dict_from_url', lambda *a, **k: (_ for _ in ()).throw(OSError('offline')))
    with pytest.raises(BaseException):
        R.ResNet([3, 4, 6, 3], 16, pretrained_url=M.PRETRAINED_BACKBONE_URLS['resnet50'])


def test_gpu_input_pipeline_host_tables_and_draws_match_the_oracle():
    """Host side of the GPU input pipeline (pixelssl_b200/task/sseg/gpu_input.py): Pillow's resampling tables and the
    reference's random-draw order, against oracle/input_oracle.py (itself pinned bit for bit to Pillow and to the
    reference's transform classes)."""
    import random
    from oracle import input_oracle as I
    from pixelssl_b200.task.sseg import gpu_input as G
    for n_in, n_out in [(53, 40), (37, 80), (64, 64), (90, 33), (500, 513), (375, 1026), (333, 257)]:
        bounds, taps = I._coefficients(n_in, n_out)
        b, w = G.bilinear_tables(n_in, n_out)
        assert b.shape == (n_out, 2) and w.shape[0] == n_out
        for i, ((x0, n), k) in enumerate(zip(bounds, taps)):
            assert (int(b[i, 0]), int(b[i, 1])) == (x0, n)
            assert np.array_equal(w[i, :n], k) and not w[i, n:].any()
        ramp = np.arange(n_in, dtype=np.int64)[None, :].repeat(2, 0)
        assert np.array_equal(G.nearest_table(n_in, n_out), I.resize_nearest(ramp, n_out, 2)[0])
    # the draws: composing the oracle's pixel functions with the product's geometry reproduces the oracle's pipeline
    rs = np.random.RandomState(5)
    for k, (h, w, base, crop) in enumerate([(37, 53, 40, 33), (64, 41, 40, 33), (50, 50, 24, 40), (33, 90, 60, 33)]):
        img = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
        lab = rs.randint(0, 21, (h, w)).astype(np.uint8)
        random.seed(900 + k)
        x_ref, y_ref = I.train_prehandle(img, lab, base, crop)
        random.seed(900 + k)
        ow, oh, x1, y1, flip = G.draw_train_geometry(h, w, base, crop)
        a, m = I.resize_bilinear_u8(img, ow, oh), I.resize_nearest(lab, ow, oh)
        a = np.pad(a, ((0, max(crop - oh, 0)), (0, max(crop - ow, 0)), (0, 0)))
        m = np.pad(m, ((0, max(crop - oh, 0)), (0, max(crop - ow, 0))))
        a, m = a[y1:y1 + crop, x1:x1 + crop], m[y1:y1 + crop, x1:x1 + crop]
        if flip:
            a, m = a[:, ::-1], m[:, ::-1]
        x, y = I.normalize_to_chw(a, m)
        assert np.array_equal(x, x_ref) and np.array_equal(y, y_ref)
