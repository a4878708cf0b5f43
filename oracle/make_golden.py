"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference) on CPU.

TEST INFRASTRUCTURE.  Run in the build container only (the reference does not exist on the GPU
box):   python oracle/make_golden.py
The committed fixtures are what pins ``oracle/sseg_oracle.py`` (tests/test_oracle_golden.py) and,
on the GPU box, the CUDA engine (tests/test_gpu_*.py).

Harness = SURVEY.md section 8(c): four monkeypatches so the reference's ``_train`` bodies run
without a GPU (``Tensor.cuda``/``Module.cuda`` -> identity, ``torch.cuda.device_count`` -> 1,
``model_zoo.load_url`` -> {}), args built through the reference's own parser, and a Python list
of (inp, gt) tuples standing in for the DataLoader.  Model weights are NOT taken from the
reference's RNG: ``oracle.sseg_oracle.init_deeplabv2(seed)`` state is loaded into the reference
modules, so tests can rebuild identical weights without shipping 176 MB.
"""
import os
import sys
import collections
import random

import numpy as np
import torch

REF = '/root/reference'
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, 'tests', 'golden')
sys.path.insert(0, ROOT)

from oracle import sseg_oracle as O  # noqa: E402


def patch_and_import():
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.nn.Module.cuda = lambda self, *a, **k: self
    torch.cuda.device_count = lambda: 1
    import torch.utils.model_zoo as mz
    mz.load_url = lambda *a, **k: {}
    sys.path.insert(0, REF)
    sys.path.insert(0, os.path.join(REF, 'task', 'sseg'))
    import logging
    import pixelssl
    logging.getLogger('PixelSSL').setLevel(logging.ERROR)
    import proxy as sseg_proxy
    return pixelssl, sseg_proxy


def make_args(pixelssl, sseg_proxy, algorithm, extra, batch, ubs, epochs=2, iters_per_epoch=5):
    from pixelssl import runner
    from pixelssl.utils import cmd
    cfg = collections.OrderedDict([
        ('exp_id', 'golden'), ('ssl_algorithm', algorithm),
        ('models', {'model': 'deeplabv2'}), ('optimizers', {'model': 'sgd'}),
        ('lrers', {'model': 'polynomiallr'}), ('criterions', {'model': 'sseg_criterion'}),
        ('lr', 0.00025), ('momentum', 0.9), ('weight_decay', 0.0005),
        ('output_stride', 16), ('backbone', 'resnet101'),
        ('epochs', epochs), ('batch_size', batch), ('unlabeled_batch_size', ubs),
        ('log_freq', 1000), ('visualize', False), ('im_size', 97),
    ])
    cfg.update(extra)
    parser = runner.create_parser(algorithm)
    sseg_proxy.add_parser_arguments(parser)
    args = cmd.parse_args(parser, cfg)
    # the fields TaskProxy autosets (task_template/proxy.py:63-71,195,239,252-268,414)
    args.gpus = 1
    args.task = 'sseg'
    args.labeled_batch_size = batch - ubs
    args.iters_per_epoch = iters_per_epoch
    args.is_epoch_lrer = False
    return args


def build_algorithm(pixelssl, args, algorithm):
    import model as sseg_model
    import criterion as sseg_criterion
    import func as sseg_func
    from pixelssl.nn import optimizer, lrer
    alg = pixelssl.ssl_algorithm.__dict__[algorithm].__dict__[algorithm](
        args, {'model': sseg_model.deeplabv2()}, {'model': optimizer.sgd(args)},
        {'model': lrer.polynomiallr(args)}, {'model': sseg_criterion.sseg_criterion()},
        sseg_func.task_func()(args))
    return alg


def load_state(dp_model, state):
    sd = {'module.model.' + k: v.clone() for k, v in state.items()}
    missing = dp_model.load_state_dict(sd, strict=True)
    return missing


def checksums(named):
    """[sum, sum of squares] in fp64 per tensor, in order."""
    return np.array([[float(t.double().sum()), float((t.double() ** 2).sum())] for _, t in named])


SAMPLE_PARAMS = ['backbone.conv1.weight', 'backbone.bn1.weight', 'backbone.bn1.bias',
                 'backbone.layer1.0.conv2.weight', 'backbone.layer1.0.downsample.0.weight',
                 'backbone.layer2.0.conv2.weight', 'backbone.layer3.11.bn2.weight',
                 'backbone.layer4.2.conv3.weight', 'classifier.conv2d_list.0.bias',
                 'classifier.conv2d_list.3.bias']


def sample_of(t, n=4096):
    f = t.detach().reshape(-1)
    stride = max(1, f.numel() // n)
    return f[::stride][:n].clone().numpy()


def golden_mt(pixelssl, sseg_proxy, size=97, lbs=2, ubs=2, steps=3):
    torch.manual_seed(0)
    args = make_args(pixelssl, sseg_proxy, 'ssl_mt',
                     {'cons_for_labeled': False, 'cons_scale': 1.0, 'cons_rampup_epochs': 1,
                      'ema_decay': 0.99}, lbs + ubs, ubs, epochs=2, iters_per_epoch=5)
    alg = build_algorithm(pixelssl, args, 'ssl_mt')
    s0 = O.randomize_bn_affine(O.init_deeplabv2(11, cls_bias_std=0.01), 12)
    t0 = O.randomize_bn_affine(O.init_deeplabv2(21, cls_bias_std=0.01), 22)
    load_state(alg.s_model, s0)
    load_state(alg.t_model, t0)
    names = [n for n, _, _ in O.deeplabv2_param_shapes()]
    rec = {'size': size, 'lbs': lbs, 'ubs': ubs, 'steps': steps,
           's_seed': np.array([11, 12]), 't_seed': np.array([21, 22]), 'data_seed': 100}
    batches = [O.synthetic_batch(100 + i, lbs + ubs, lbs, size, size) for i in range(steps)]
    loader = [((img.clone(),), (lab.clone(),)) for img, lab in batches]
    # run step by step so grads / logits of each step can be captured:
    # cur_step = len(loader_k) * epoch + idx; with a 1-element loader and epoch=k -> cur_step=k,
    # rampup total = 1 * cons_rampup_epochs = 1 step  => ramp(0)=exp(-5), ramp(k>=1)=1.
    for k in range(steps):
        alg._train([loader[k]], k)
        sm = alg.s_model.module.model
        tm = alg.t_model.module.model
        sp = dict(sm.named_parameters())
        tp = dict(tm.named_parameters())
        rec['s_task_loss_%d' % k] = float(alg.meters['s_task_loss'].val)
        rec['t_task_loss_%d' % k] = float(alg.meters['t_task_loss'].val)
        rec['cons_loss_%d' % k] = float(alg.meters['cons_loss'].val)
        rec['grad_checksum_%d' % k] = checksums([(n, sp[n].grad) for n in names])
        rec['s_param_checksum_%d' % k] = checksums([(n, sp[n]) for n in names])
        rec['t_param_checksum_%d' % k] = checksums([(n, tp[n]) for n in names])
        bufs = [(n, b) for n, b in sm.named_buffers() if 'num_batches' not in n]
        rec['s_buffer_checksum_%d' % k] = checksums(bufs)
        tbufs = [(n, b) for n, b in tm.named_buffers() if 'num_batches' not in n]
        rec['t_buffer_checksum_%d' % k] = checksums(tbufs)
        for n in SAMPLE_PARAMS:
            rec['grad_%d/%s' % (k, n)] = sample_of(sp[n].grad)
            rec['s_param_%d/%s' % (k, n)] = sample_of(sp[n])
        rec['lr_%d' % k] = np.array([g['lr'] for g in alg.s_optimizer.param_groups])
    rec['names'] = np.array(names)
    np.savez_compressed(os.path.join(OUT, 'mt_steps_%d.npz' % size), **rec)
    print('mt golden:', {k: rec[k] for k in rec if 'loss' in k})


def golden_forward(pixelssl, size=129, batch=2):
    """Reference DeepLabV2 forward (train-mode BN) + CE + softmax on oracle-initialised weights."""
    sys.path.insert(0, os.path.join(REF, 'task', 'sseg'))
    from module import deeplab_v2
    net = deeplab_v2.DeepLabV2('resnet101', 16, 21, True, False, None)
    st = O.randomize_bn_affine(O.init_deeplabv2(31, cls_bias_std=0.01), 32)
    net.load_state_dict({k: v.clone() for k, v in st.items()}, strict=True)
    net.train()
    img, lab = O.synthetic_batch(200, batch, batch, size, size)
    logits, latent = net(img)
    rec = {'size': size, 'batch': batch, 'seed': np.array([31, 32]), 'data_seed': 200,
           'logits': logits.detach().numpy(), 'latent_sample': sample_of(latent, 8192),
           'latent_checksum': checksums([('l', latent.detach())])}
    rec['running_checksum'] = checksums([(n, b) for n, b in net.named_buffers() if 'num_batches' not in n])
    np.savez_compressed(os.path.join(OUT, 'deeplabv2_forward_%d.npz' % size), **rec)
    print('forward golden: logits', tuple(logits.shape), float(logits.abs().max()))


def golden_ops(pixelssl, sseg_proxy):
    """Small op-level vectors from the reference's own classes / call sites."""
    import criterion as sseg_criterion
    from pixelssl.nn import func as pfunc
    from pixelssl.nn import lrer as plrer
    from pixelssl.nn.module import GaussianBlurLayer, GaussianNoiseLayer
    from pixelssl.ssl_algorithm import ssl_cutmix
    rec = {}
    # --- CommonSSEGCriterion (task/sseg/criterion.py:18-38)
    args = make_args(pixelssl, sseg_proxy, 'ssl_null', {'ignore_unlabeled': True}, 2, 0)
    crit = sseg_criterion.CommonSSEGCriterion(args)
    g = torch.Generator().manual_seed(7)
    logits = (torch.randn(3, 21, 37, 41, generator=g) * 3).requires_grad_(True)
    _, lab = O.synthetic_batch(8, 3, 3, 37, 41)
    loss = crit.forward((logits,), (lab,), (None,))
    loss.mean().backward()
    rec['ce_logits'] = logits.detach().numpy()
    rec['ce_labels'] = lab.numpy()
    rec['ce_loss'] = loss.detach().numpy()
    rec['ce_grad'] = logits.grad.numpy()
    # --- nn.MSELoss consistency (ssl_mt.py:115,179-187)
    a = torch.randn(2, 21, 33, 35, generator=g).requires_grad_(True)
    b = torch.randn(2, 21, 33, 35, generator=g)
    m = torch.nn.MSELoss()(a, b)
    (0.37 * m).backward()
    rec['mse_s'], rec['mse_t'] = a.detach().numpy(), b.numpy()
    rec['mse_loss'], rec['mse_grad_scale'], rec['mse_grad'] = float(m), 0.37, a.grad.numpy()
    # --- sigmoid_rampup, PolynomialLR
    rec['rampup'] = np.array([pfunc.sigmoid_rampup(c, 30) for c in range(0, 40, 3)] +
                             [pfunc.sigmoid_rampup(5, 0)])
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([{'params': [p], 'lr': 0.00025}], lr=0.00025, momentum=0.9)
    sch = plrer.PolynomialLR(opt, epochs=2, iters_per_epoch=5, power=0.9)
    lrs = [opt.param_groups[0]['lr']]
    for _ in range(8):
        opt.step()
        sch.step()
        lrs.append(opt.param_groups[0]['lr'])
    rec['poly_lr'] = np.array(lrs)
    # --- BoxMaskGenerator (ssl_cutmix.py:470-547) + mix (ssl_cutmix.py:195,428)
    np.random.seed(1234)
    gen = ssl_cutmix.BoxMaskGenerator(prop_range=(0.5, 0.5), boxes_num=1, random_aspect_ratio=True,
                                      area_prop=True, within_bounds=True, invert=True)
    masks = gen.produce(4, (65, 97))
    rec['cutmix_masks'] = masks
    np.random.seed(99)
    gen2 = ssl_cutmix.BoxMaskGenerator(prop_range=(0.25, 0.5), boxes_num=1, random_aspect_ratio=True,
                                       area_prop=True, within_bounds=True, invert=True)
    rec['cutmix_masks_b'] = gen2.produce(3, (513, 513)).reshape(3, 513, 513)[:, ::8, ::8].copy()
    np.random.seed(99)
    full = gen2.produce(3, (513, 513))
    rec['cutmix_masks_b_sum'] = full.reshape(3, -1).sum(1)
    u1 = torch.randn(4, 3, 65, 97, generator=g) * 1e3
    u2 = torch.randn(4, 3, 65, 97, generator=g)
    u1[0, 0, 0, :4] = torch.tensor([float('inf'), -0.0, 0.0, 1e-42])
    mk = torch.tensor(masks)
    rec['cutmix_a'], rec['cutmix_b'] = u1.numpy(), u2.numpy()
    rec['cutmix_mixed'] = (mk * u1 + (1 - mk) * u2).numpy()
    prob = torch.softmax(torch.randn(4, 21, 65, 97, generator=g) * 4, dim=1)
    rec['conf_prob'] = prob.numpy()
    rec['conf_value'] = float((prob.max(dim=1)[0] > 0.97).float().mean())
    # --- GaussianBlurLayer weights (gaussian_blur.py:52-64) and one blur
    for k in (5, 33, 65):
        layer = GaussianBlurLayer(1, k)
        rec['blur_w_%d' % k] = layer.op[1].weight.detach().numpy()[0, 0]
    x = torch.rand(2, 1, 40, 44, generator=g)
    rec['blur_x'] = x.numpy()
    rec['blur_y_5'] = GaussianBlurLayer(1, 5)(x).detach().numpy()
    rec['blur_y_33'] = GaussianBlurLayer(1, 33)(x).detach().numpy()
    # --- GaussianNoiseLayer (gaussian_noise.py:17-40) with a captured noise draw
    random.seed(5)
    torch.manual_seed(5)
    layer = GaussianNoiseLayer(0.3)
    xin = torch.randn(2, 3, 19, 23, generator=g)
    y = layer(xin.clone())
    rec['noise_x'], rec['noise_n'], rec['noise_y'] = xin.numpy(), layer.noise.numpy().copy(), y.numpy()
    # --- SyncBN multi-replica statistics (batchnorm.py:113-125)
    from pixelssl.nn.module import SynchronizedBatchNorm2d
    bn = SynchronizedBatchNorm2d(6)
    bn.weight.data = torch.randn(6, generator=g)
    bn.bias.data = torch.randn(6, generator=g)
    parts = [torch.randn(2, 6, 5, 7, generator=g) * 2 + 1, torch.randn(3, 6, 5, 7, generator=g)]
    sz = sum(p.numel() // 6 for p in parts)
    s = sum(p.transpose(0, 1).reshape(6, -1).sum(1) for p in parts)
    ss = sum((p ** 2).transpose(0, 1).reshape(6, -1).sum(1) for p in parts)
    mean, inv_std = bn._compute_mean_std(s, ss, sz)
    rec['sbn_parts0'], rec['sbn_parts1'] = parts[0].numpy(), parts[1].numpy()
    rec['sbn_w'], rec['sbn_b'] = bn.weight.detach().numpy(), bn.bias.detach().numpy()
    rec['sbn_mean'], rec['sbn_inv_std'] = mean.numpy(), inv_std.numpy()
    rec['sbn_running_mean'], rec['sbn_running_var'] = bn.running_mean.numpy(), bn.running_var.numpy()
    np.savez_compressed(os.path.join(OUT, 'ops.npz'), **rec)
    print('ops golden written:', len(rec), 'arrays')


def golden_null_cutmix(pixelssl, sseg_proxy, size=65):
    """One SSLNULL step and one SSLCUTMIX step through the reference's own _train bodies."""
    names = [n for n, _, _ in O.deeplabv2_param_shapes()]
    # --- supervised-only (ssl_null.py:78-144)
    args = make_args(pixelssl, sseg_proxy, 'ssl_null', {'ignore_unlabeled': True}, 2, 0)
    alg = build_algorithm(pixelssl, args, 'ssl_null')
    load_state(alg.model, O.randomize_bn_affine(O.init_deeplabv2(41, cls_bias_std=0.01), 42))
    img, lab = O.synthetic_batch(300, 2, 2, size, size)
    alg._train([((img.clone(),), (lab.clone(),))], 0)
    sp = dict(alg.model.module.model.named_parameters())
    rec = {'size': size, 'task_loss': float(alg.meters['task_loss'].val),
           'grad_checksum': checksums([(n, sp[n].grad) for n in names]),
           'param_checksum': checksums([(n, sp[n]) for n in names])}
    np.savez_compressed(os.path.join(OUT, 'null_step_%d.npz' % size), **rec)
    print('null golden:', rec['task_loss'])
    # --- CutMix (ssl_cutmix.py:132-255), lbs 2 + ubs 4 -> 2 mixed
    args = make_args(pixelssl, sseg_proxy, 'ssl_cutmix',
                     {'cons_scale': 20.0, 'cons_rampup_epochs': 0, 'cons_threshold': 0.05,
                      'ema_decay': 0.99, 'mask_prop_range': '(0.5, 0.5)', 'cons_type': 'mse'}, 6, 4)
    alg = build_algorithm(pixelssl, args, 'ssl_cutmix')
    load_state(alg.s_model, O.randomize_bn_affine(O.init_deeplabv2(51, cls_bias_std=0.01), 52))
    load_state(alg.t_model, O.randomize_bn_affine(O.init_deeplabv2(61, cls_bias_std=0.01), 62))
    img, lab = O.synthetic_batch(400, 6, 2, size, size)
    np.random.seed(4321)
    alg._train([((img.clone(),), (lab.clone(),))], 0)
    sp = dict(alg.s_model.module.model.named_parameters())
    tp = dict(alg.t_model.module.model.named_parameters())
    rec = {'size': size, 'task_loss': float(alg.meters['task_loss'].val),
           'cons_loss': float(alg.meters['cons_loss'].val), 'mask_seed': 4321,
           'cons_threshold': 0.05,
           'grad_checksum': checksums([(n, sp[n].grad) for n in names]),
           's_param_checksum': checksums([(n, sp[n]) for n in names]),
           't_param_checksum': checksums([(n, tp[n]) for n in names])}
    np.savez_compressed(os.path.join(OUT, 'cutmix_step_%d.npz' % size), **rec)
    print('cutmix golden:', rec['task_loss'], rec['cons_loss'])


def golden_adv(pixelssl, sseg_proxy, size=65):
    """One SSLADV._train step (ssl_adv.py:118-283): lbs 2 + ubs 2, adversarial terms on both."""
    from oracle import adv_oracle as A
    names = [n for n, _, _ in O.deeplabv2_param_shapes()]
    args = make_args(pixelssl, sseg_proxy, 'ssl_adv',
                     {'adv_for_labeled': True, 'labeled_adv_scale': 0.01, 'unlabeled_adv_scale': 0.001,
                      'discriminator_lr': 1e-4, 'discriminator_scale': 1.0, 'unlabeled_for_discriminator': True}, 4, 2)
    alg = build_algorithm(pixelssl, args, 'ssl_adv')
    load_state(alg.model, O.randomize_bn_affine(O.init_deeplabv2(81, cls_bias_std=0.01), 82))
    alg.d_model.load_state_dict({'module.' + k: v.clone() for k, v in A.init_fcd(83).items()}, strict=True)
    img, lab = O.synthetic_batch(600, 4, 2, size, size)
    alg._train([((img.clone(),), (lab.clone(),))], 0)
    sp = dict(alg.model.module.model.named_parameters())
    dp = dict(alg.d_model.module.named_parameters())
    dnames = [n for n, _ in A.fcd_shapes()]
    rec = {'size': size}
    for k in ('task_loss', 'labeled_adv_loss', 'unlabeled_adv_loss', 'fake_d_loss', 'real_d_loss'):
        rec[k] = float(alg.meters[k].val)
    rec['grad_checksum'] = checksums([(n, sp[n].grad) for n in names])
    rec['param_checksum'] = checksums([(n, sp[n]) for n in names])
    rec['d_grad_checksum'] = checksums([(n, dp[n].grad) for n in dnames])
    rec['d_param_checksum'] = checksums([(n, dp[n]) for n in dnames])
    rec['d_lr'] = alg.d_optimizer.param_groups[0]['lr']
    np.savez_compressed(os.path.join(OUT, 'adv_step_%d.npz' % size), **rec)
    print('adv golden:', {k: rec[k] for k in rec if 'loss' in k})


def golden_s4l(pixelssl, sseg_proxy, size=65):
    """One SSLS4L._train step (ssl_s4l.py:113-200): lbs 2 + ubs 2 doubled by the rotated copies."""
    from oracle import s4l_oracle as S
    names = [n for n, _, _ in O.deeplabv2_param_shapes()]
    args = make_args(pixelssl, sseg_proxy, 'ssl_s4l', {'rotated_sup_scale': 0.5, 'rotation_scale': 1.0}, 4, 2)
    alg = build_algorithm(pixelssl, args, 'ssl_s4l')
    st = O.randomize_bn_affine(O.init_deeplabv2(121, cls_bias_std=0.01), 122)
    sd = {'module.task_model.model.' + k: v.clone() for k, v in st.items()}
    sd.update({'module.rotation_classifier.' + k: v.clone() for k, v in S.init_rc(123).items()})
    missing = alg.model.load_state_dict(sd, strict=False)
    assert not [k for k in missing.missing_keys if 'num_batches' not in k and 'running' not in k], missing
    img, lab = O.synthetic_batch(1000, 4, 2, size, size)
    np.random.seed(77)
    alg._train([((img.clone(),), (lab.clone(),))], 0)
    sp = dict(alg.model.module.task_model.model.named_parameters())
    rp = dict(alg.model.module.rotation_classifier.named_parameters())
    rnames = [n for n, _ in S.rc_shapes()]
    rec = {'size': size, 'np_seed': 77}
    for k in ('unrotated_task_loss', 'rotated_task_loss', 'rotation_loss', 'rotation_acc'):
        rec[k] = float(alg.meters[k].val)
    rec['grad_checksum'] = checksums([(n, sp[n].grad) for n in names])
    rec['param_checksum'] = checksums([(n, sp[n]) for n in names])
    rec['rc_grad_checksum'] = checksums([(n, rp[n].grad) for n in rnames])
    rec['rc_param_checksum'] = checksums([(n, rp[n]) for n in rnames])
    rb = dict(alg.model.module.rotation_classifier.named_buffers())
    rec['rc_buffer_checksum'] = checksums([(n, b.float()) for n, b in rb.items()])
    rec['rc_buffer_names'] = np.array(list(rb.keys()))
    rec['lrs'] = np.array([g['lr'] for g in alg.optimizer.param_groups])
    # the rotated batch itself (bit-exact target of the rotate kernel)
    np.random.seed(77)
    angles = np.random.randint(low=1, high=4, size=4)
    rec['angles'] = angles
    rec['rot_img_sample'] = alg._rotate_tensor(img[1], int(angles[1])).numpy()
    np.savez_compressed(os.path.join(OUT, 's4l_step_%d.npz' % size), **rec)
    print('s4l golden:', {k: rec[k] for k in rec if 'loss' in k or 'acc' in k}, 'angles', angles)


def golden_gct(pixelssl, sseg_proxy, size=129):
    """One SSLGCT._train step (ssl_gct.py:176-298): two DeepLabV2 task models + FlawDetector, lbs 2 + ubs 2."""
    from oracle import gct_oracle as Gc
    names = [n for n, _, _ in O.deeplabv2_param_shapes()]
    args = make_args(pixelssl, sseg_proxy, 'ssl_gct',
                     {'ssl_mode': 'gct', 'fc_ssl_scale': 1.0, 'dc_ssl_scale': 100.0, 'dc_threshold': 0.45,
                      'dc_rampup_epochs': 0, 'fd_lr': 1e-4, 'fd_scale': 10.0, 'mu': 0.5, 'nu': 1, 'im_size': size}, 4, 2)
    alg = build_algorithm(pixelssl, args, 'ssl_gct')
    load_state(alg.l_model, O.randomize_bn_affine(O.init_deeplabv2(91, cls_bias_std=0.01), 92))
    load_state(alg.r_model, O.randomize_bn_affine(O.init_deeplabv2(93, cls_bias_std=0.01), 94))
    alg.fd_model.load_state_dict({'module.' + k: v.clone() for k, v in Gc.init_fd(95).items()}, strict=True)
    img, lab = O.synthetic_batch(700, 4, 2, size, size)
    alg._train([((img.clone(),), (lab.clone(),))], 0)
    rec = {'size': size}
    for k in ('l_task_loss', 'l_fc_loss', 'l_dc_loss', 'r_task_loss', 'r_fc_loss', 'r_dc_loss', 'l_fd_loss', 'r_fd_loss'):
        rec[k] = float(alg.meters[k].val)
    for mid, model in (('l', alg.l_model), ('r', alg.r_model)):
        sp = dict(model.module.model.named_parameters())
        rec[mid + '_grad_checksum'] = checksums([(n, sp[n].grad) for n in names])
        rec[mid + '_param_checksum'] = checksums([(n, sp[n]) for n in names])
    fp = dict(alg.fd_model.module.named_parameters())
    fnames = [n for n, _ in Gc.fd_param_shapes()]
    rec['fd_grad_checksum'] = checksums([(n, fp[n].grad) for n in fnames])
    rec['fd_param_checksum'] = checksums([(n, fp[n]) for n in fnames])
    rec['fd_buffer_checksum'] = checksums([(n, b) for n, b in alg.fd_model.module.named_buffers() if 'num_batches' not in n])
    rec['fd_lr'] = alg.fd_optimizer.param_groups[0]['lr']
    np.savez_compressed(os.path.join(OUT, 'gct_step_%d.npz' % size), **rec)
    print('gct golden:', {k: rec[k] for k in rec if 'loss' in k})


def golden_cct(pixelssl, sseg_proxy, size=65):
    """One SSLCCT._train step (ssl_cct.py:226-301) with one decoder of every kind, lbs 2 + ubs 2."""
    from oracle import cct_oracle as C
    names = [n for n, _, _ in O.deeplabv2_param_shapes()]
    args = make_args(pixelssl, sseg_proxy, 'ssl_cct',
                     {'cons_scale': 30.0, 'cons_rampup_epochs': 0, 'ad_lr_scale': 10.0, 'vat_dec_num': 1, 'drop_dec_num': 1,
                      'cut_dec_num': 1, 'context_dec_num': 1, 'object_dec_num': 1, 'fd_dec_num': 1, 'fn_dec_num': 1,
                      'vat_dec_xi': 1e-6, 'vat_dec_eps': 2.0, 'drop_dec_rate': 0.5, 'cut_dec_erase': 0.4,
                      'fn_dec_uniform': 0.3}, 4, 2)
    alg = build_algorithm(pixelssl, args, 'ssl_cct')
    st = O.randomize_bn_affine(O.init_deeplabv2(101, cls_bias_std=0.01), 102)
    dec = C.init_decoders(103, 7)
    sd = {'module.main_model.model.' + k: v.clone() for k, v in st.items()}
    sd.update({'module.' + k: v.clone() for k, v in dec.items()})
    missing = alg.model.load_state_dict(sd, strict=True)
    img, lab = O.synthetic_batch(800, 4, 2, size, size)
    random.seed(7); np.random.seed(8); torch.manual_seed(9)
    alg._train([((img.clone(),), (lab.clone(),))], 0)
    sp = dict(alg.model.module.main_model.model.named_parameters())
    dp = dict(alg.model.module.named_parameters())
    dnames = [n for i in range(7) for n, _ in C.decoder_param_shapes(i)]
    rec = {'size': size, 'task_loss': float(alg.meters['task_loss'].val), 'cons_loss': float(alg.meters['cons_loss'].val)}
    rec['grad_checksum'] = checksums([(n, sp[n].grad) for n in names])
    rec['param_checksum'] = checksums([(n, sp[n]) for n in names])
    rec['dec_grad_checksum'] = checksums([(n, dp[n].grad) for n in dnames])
    rec['dec_param_checksum'] = checksums([(n, dp[n]) for n in dnames])
    rec['lrs'] = np.array([g['lr'] for g in alg.optimizer.param_groups])
    np.savez_compressed(os.path.join(OUT, 'cct_step_%d.npz' % size), **rec)
    print('cct golden:', rec['task_loss'], rec['cons_loss'], rec['lrs'])


def golden_pspnet(pixelssl, size=97, batch=2):
    """Reference _PSPNet (ResNet-50, OS16) forward in train mode on oracle-initialised weights."""
    sys.path.insert(0, os.path.join(REF, 'task', 'sseg'))
    from module import _pspnet
    net = _pspnet._PSPNet('resnet50', 16, 21, True, False, None)
    st = O.randomize_bn_affine(O.init_pspnet(111), 112)
    net.load_state_dict({k: v.clone() for k, v in st.items()}, strict=True)
    net.train()
    img, _ = O.synthetic_batch(900, batch, batch, size, size)
    logits, px = net(img)
    rec = {'size': size, 'batch': batch, 'logits': logits.detach().numpy(), 'latent_checksum': checksums([('l', px.detach())]),
           'running_checksum': checksums([(n, b) for n, b in net.named_buffers() if 'num_batches' not in n])}
    np.savez_compressed(os.path.join(OUT, 'pspnet_forward_%d.npz' % size), **rec)
    print('pspnet golden: logits', tuple(logits.shape), float(logits.abs().max()))


def golden_val(pixelssl, sseg_proxy):
    """Validation metrics (task/sseg/func.py:36-80), the MT input-noise layer
    (pixelssl/nn/module/gaussian_noise.py) and the two-stream sampler (pixelssl/nn/data.py:126-177)."""
    import func as sseg_func
    from pixelssl.utils import logger as ref_logger
    from pixelssl.nn.module import GaussianNoiseLayer
    from pixelssl.nn import data as ref_data
    out = {}
    # ---- metrics over two batches -----------------------------------------------------------
    args = make_args(pixelssl, sseg_proxy, 'ssl_null', {}, 2, 0)
    tf = sseg_func.task_func()(args)
    meters = ref_logger.AvgMeterSet()
    g = torch.Generator().manual_seed(11)
    for k, (n, h, w) in enumerate([(3, 40, 37), (2, 33, 65)]):
        pred = torch.softmax(3.0 * torch.randn(n, args.num_classes, h, w, generator=g), dim=1)
        pred[0, :, 0, 0] = 0.25                       # an exact tie: argmax must pick the first index
        gt = torch.randint(0, args.num_classes, (n, 1, h, w), generator=g).float()
        gt[torch.rand(n, 1, h, w, generator=g) < 0.1] = 255.0
        gt[0, 0, 1, :3] = -1.0
        if k == 1:
            gt[gt == 7.0] = 3.0                       # a class absent from gt -> nanmean path
        tf.metrics((pred,), (gt,), None, meters, id_str='task')
        out['metrics_pred%d' % k], out['metrics_gt%d' % k] = pred.numpy(), gt.numpy()
        out['metrics_cmat_sum%d' % k] = np.array(meters['task_confusion_matrix'].sum)
        out['metrics_values%d' % k] = np.array([float(meters['task_metric_' + m].val)
                                                for m in ('acc', 'acc-class', 'mIoU', 'fwIoU')])
    # ---- gaussian noise layer ----------------------------------------------------------------
    torch.manual_seed(5)
    random.seed(5)
    layer = GaussianNoiseLayer(0.15)
    inp = torch.randn(3, 3, 29, 31) * torch.tensor([1.0, 5.0, 0.01]).view(3, 1, 1, 1) + 0.3
    res = layer.forward(inp.clone())
    out['gn_inp'], out['gn_noise'], out['gn_out'] = inp.numpy(), layer.noise.numpy().copy(), res.numpy()
    # ---- two-stream sampler: 3 epochs per configuration ---------------------------------------
    cfgs = np.array([[10, 37, 2, 3], [50, 13, 4, 2], [8, 8, 2, 2], [7, 29, 3, 5], [40, 90, 4, 6]])
    out['sampler_cfgs'] = cfgs
    for c, (nl, nu, lb, ub) in enumerate(cfgs):
        np.random.seed(100 + c)
        smp = ref_data.TwoStreamBatchSampler(list(range(nl)), list(range(1000, 1000 + nu)), int(lb), int(ub))
        for e in range(3):
            out['sampler_%d_epoch%d' % (c, e)] = np.array([list(map(int, b)) for b in smp], dtype=np.int64)
    np.savez_compressed(os.path.join(OUT, 'val.npz'), **out)
    print('val.npz written:', {k: v.shape for k, v in out.items() if not k.startswith('sampler_')})


def golden_input(pixelssl, sseg_proxy):
    """Training input pipeline (task/sseg/data.py:90-123,142-256) run through the reference's own transform classes on
    synthetic 8-bit images: the pin of oracle/input_oracle.py (and of a future GPU augmentation path)."""
    import types
    import data as sseg_data
    from PIL import Image
    out = {}
    rs = np.random.RandomState(77)
    cases = [(37, 53, 40, 33, True), (64, 41, 40, 33, True), (50, 50, 24, 40, True), (45, 70, 40, 33, False),
             (33, 90, 60, 33, False)]
    out['cases'] = np.array([[h, w, b, c, int(l)] for h, w, b, c, l in cases])
    for k, (h, w, base, crop, labeled) in enumerate(cases):
        img = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
        lab = rs.randint(0, 21, (h, w)).astype(np.uint8)
        lab[rs.rand(h, w) < 0.1] = 255
        fake = types.SimpleNamespace(args=types.SimpleNamespace(train_base_size=base, im_size=crop),
                                     IMAGE=sseg_data.PascalVocDataset.IMAGE, LABEL=sseg_data.PascalVocDataset.LABEL)
        random.seed(500 + k)
        x, y = sseg_data.PascalVocDataset._train_prehandle(
            fake, Image.fromarray(img), Image.fromarray(lab) if labeled else None)
        out['img%d' % k], out['lab%d' % k] = img, lab
        out['x%d' % k], out['y%d' % k] = x.numpy(), y.numpy()
    np.savez_compressed(os.path.join(OUT, 'input_pipeline.npz'), **out)
    print('input_pipeline.npz written:', {k: v.shape for k, v in out.items() if k.startswith(('x', 'y'))})


def golden_val_prehandle(pixelssl, sseg_proxy):
    """Validation input pipeline (task/sseg/data.py ``_val_prehandle``: optional FixedScaleResize + Normalize +
    ToTensor) on the inputs of tests/test_oracle_golden.py."""
    import types
    import data as sseg_data
    from PIL import Image
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import test_oracle_golden as T
    out = {}
    for k, (h, w, size, rescaling) in enumerate(T.VAL_PREHANDLE_CASES):
        img, lab = T.val_prehandle_inputs(h, w)
        fake = types.SimpleNamespace(args=types.SimpleNamespace(val_rescaling=rescaling, im_size=size),
                                     IMAGE=sseg_data.PascalVocDataset.IMAGE, LABEL=sseg_data.PascalVocDataset.LABEL)
        x, y = sseg_data.PascalVocDataset._val_prehandle(fake, Image.fromarray(img), Image.fromarray(lab))
        out['x%d' % k], out['y%d' % k] = x.numpy(), y.numpy()
    np.savez_compressed(os.path.join(OUT, 'val_prehandle.npz'), **out)
    print('val_prehandle.npz written:', {k: v.shape for k, v in out.items()})


def golden_host(pixelssl, sseg_proxy):
    """Host-side API of the reference, as tests/test_host_cpu.py compares the engine with it: algorithm registry and
    sampler stream, task-model state_dict layouts and LR groups, checkpoint keys, parser tables, LR trajectories,
    constructor argument checks, TaskFunc shape hooks and optimizer hyper-parameters."""
    import argparse
    import gzip
    import importlib
    import json
    import func as sseg_func
    import model as sseg_model
    from pixelssl import runner as ref_runner
    from pixelssl.nn import data as ref_data, lrer as ref_lrer, optimizer as ref_optimizer
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import test_host_cpu as T
    np.random.seed(5)
    out = {'register': {'ssl_algorithms': list(pixelssl.ssl_algorithm.SSL_ALGORITHMS),
                        'sampler_seed5': [list(map(int, b)) for b in ref_data.TwoStreamBatchSampler(
                            list(range(9)), list(range(50, 83)), 2, 3)]}}
    out['checkpoint_keys'] = {}
    out['parser_table'] = {}
    for alg in T.SSL_ALGS:
        mod = importlib.import_module('pixelssl.ssl_algorithm.' + alg)
        with open(mod.__file__) as f:
            out['checkpoint_keys'][alg] = T._checkpoint_keys(f.read())
        parser = argparse.ArgumentParser()
        mod.add_parser_arguments(parser)
        out['parser_table'][alg] = T._parser_table(parser)
    parser = ref_runner.create_parser('ssl_null')
    sseg_proxy.add_parser_arguments(parser)
    out['full_parser_table'] = T._parser_table(parser, option_strings=False)
    out['lr_trajectory'] = {n: T._lr_trajectory(ref_lrer, n) for n in T.LR_SCHEDULERS}
    out['constructor_rejects'] = {T._case_id(alg, ov): T._constructor_rejects(
        importlib.import_module('pixelssl.ssl_algorithm.' + alg), alg, ov) for alg, ov in T._CASES}
    out['task_func'] = {}
    for arch in ('deeplabv2', 'pspnet'):
        tf = sseg_func.task_func()(T._task_func_args(arch))
        out['task_func'][arch] = dict({h: getattr(tf, h)() for h in T.SHAPE_HOOKS}, METRIC_STR=tf.METRIC_STR)
    out['optimizer'] = {n: T._optimizer_summary(ref_optimizer, n) for n in ('sgd', 'adam')}
    with open(os.path.join(OUT, 'reference_host.json'), 'w') as f:
        json.dump(out, f, sort_keys=True, indent=1)
        f.write('\n')
    # the state_dict layouts are ~140 kB of JSON: stored compressed
    layouts = {'%s-%s' % (n, b): T._task_model_layout(sseg_model, n, b) for n, b in T.TASK_MODELS}
    with gzip.open(os.path.join(OUT, 'reference_task_models.json.gz'), 'wt') as f:
        json.dump(layouts, f, sort_keys=True)
    print('reference_host.json, reference_task_models.json.gz written:', sorted(out))


def golden_fp64_mid(size=257):
    """fp64 truth of the mid-size MT step (mt_steps_257.npz): same seeds as golden_mt(size=257, steps=1)."""
    D = torch.float64
    names = [n for n, _, _ in O.deeplabv2_param_shapes()]
    rec = {}
    s = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(11, cls_bias_std=0.01), 12), D)
    t = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(21, cls_bias_std=0.01), 22), D)
    mt = O.MTOracle(s, t, lr=0.00025, momentum=0.9, weight_decay=0.0005, max_iters=10,
                    cons_scale=1.0, rampup_steps=1, ema_decay=0.99, cons_for_labeled=False)
    img, lab = O.synthetic_batch(100, 4, 2, size, size)
    out = mt.step(img.to(D), lab.to(D), 2)
    for key in ('s_task_loss', 't_task_loss', 'cons_loss'):
        rec['mt_%s_0' % key] = float(out[key])
    rec['mt_grad_checksum_0'] = checksums([(n, out['grads'][n]) for n in names])
    rec['mt_s_param_checksum_0'] = checksums([(n, mt.s[n]) for n in names])
    rec['mt_t_param_checksum_0'] = checksums([(n, mt.t[n]) for n in names])
    for n in SAMPLE_PARAMS:
        rec['mt_grad_0/%s' % n] = sample_of(out['grads'][n].float())
    np.savez_compressed(os.path.join(OUT, 'fp64_truth_%d.npz' % size), **rec)
    print('fp64 truth (mid-size) written')


def golden_fp64_algs():
    """fp64 oracle evaluation of the Adv / GCT / CCT golden steps (adv_step_65, gct_step_129, cct_step_65): the
    yardstick of the reference's own fp32 noise for the quantities tests/test_gpu_{adv,gct,cct}.py compare."""
    import random
    from oracle import adv_oracle as A, gct_oracle as Gc, cct_oracle as C
    D = torch.float64
    names = [n for n, _, _ in O.deeplabv2_param_shapes()]
    rec = {}

    def td(st):
        return {k: (v.to(D) if v.is_floating_point() else v) for k, v in st.items()}
    # AdvSSL
    s = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(81, cls_bias_std=0.01), 82), D)
    adv = A.AdvOracle(s, td(A.init_fcd(83)), labeled_adv_scale=0.01, unlabeled_adv_scale=0.001, adv_for_labeled=True,
                      discriminator_lr=1e-4, unlabeled_for_discriminator=True, lr=0.00025, momentum=0.9,
                      weight_decay=0.0005, max_iters=10)
    img, lab = O.synthetic_batch(600, 4, 2, 65, 65)
    out = adv.step(img.to(D), lab.to(D), 2)
    for k in ('task_loss', 'labeled_adv_loss', 'unlabeled_adv_loss', 'fake_d_loss', 'real_d_loss'):
        rec['adv_' + k] = float(out[k])
    rec['adv_grad_checksum'] = checksums([(n, out['grads'][n]) for n in names])
    rec['adv_d_grad_checksum'] = checksums([(n, out['d_grads'][n]) for n in adv.d_names])
    print('adv fp64 done')
    # GCT
    lst = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(91, cls_bias_std=0.01), 92), D)
    rst = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(93, cls_bias_std=0.01), 94), D)
    gct = Gc.GctOracle(lst, rst, td(Gc.init_fd(95)), 129, fc_ssl_scale=1.0, dc_ssl_scale=100.0, dc_threshold=0.45,
                       rampup_steps=0, fd_lr=1e-4, fd_scale=10.0, mu=0.5, nu=1)
    img, lab = O.synthetic_batch(700, 4, 2, 129, 129)
    out = gct.step(img.to(D), lab.to(D), 2)
    for k in ('l_task_loss', 'l_fc_loss', 'l_dc_loss', 'r_task_loss', 'r_fc_loss', 'r_dc_loss', 'l_fd_loss', 'r_fd_loss'):
        rec['gct_' + k] = float(out[k])
    for mid in ('l', 'r'):
        rec['gct_%s_grad_checksum' % mid] = checksums([(n, out[mid + '_grads'][n]) for n in names])
    rec['gct_fd_grad_checksum'] = checksums([(n, out['fd_grads'][n]) for n in gct.fd_names])
    print('gct fp64 done')
    # CCT
    st = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(101, cls_bias_std=0.01), 102), D)
    cct = C.CctOracle(st, td(C.init_decoders(103, 7)), C.KINDS, cons_scale=30.0, rampup_steps=0, ad_lr_scale=10.0,
                      lr=0.00025, momentum=0.9, weight_decay=0.0005, max_iters=10)
    img, lab = O.synthetic_batch(800, 4, 2, 65, 65)
    random.seed(7); np.random.seed(8); torch.manual_seed(9)
    out = cct.step(img.to(D), lab.to(D), 2)
    rec['cct_task_loss'], rec['cct_cons_loss'] = float(out['task_loss']), float(out['cons_loss'])
    rec['cct_grad_checksum'] = checksums([(n, out['grads'][n]) for n in names])
    rec['cct_dec_grad_checksum'] = checksums([(n, out['dec_grads'][n]) for n in cct.dec_names])
    np.savez_compressed(os.path.join(OUT, 'fp64_truth_algs.npz'), **rec)
    print('fp64 truth (adv / gct / cct) written')


def golden_fp64():
    """Exact-arithmetic (fp64) evaluation of the SAME steps with the oracle, to measure the
    reference's own fp32 rounding noise on these (ill-conditioned, random-init) networks.  The GPU
    engine is held to that yardstick (tests/test_gpu_model.py).  Needs no reference import."""
    D = torch.float64
    names = [n for n, _, _ in O.deeplabv2_param_shapes()]
    rec = {}
    # forward (deeplabv2_forward_129.npz)
    st = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(31, cls_bias_std=0.01), 32), D)
    img, _ = O.synthetic_batch(200, 2, 2, 129, 129)
    with torch.no_grad():
        logits, latent = O.deeplabv2_forward(img.to(D), st, True)
    rec['fwd_logits'] = logits.float().numpy()
    rec['fwd_latent_checksum'] = checksums([('l', latent)])
    # MT steps (mt_steps_97.npz)
    s = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(11, cls_bias_std=0.01), 12), D)
    t = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(21, cls_bias_std=0.01), 22), D)
    mt = O.MTOracle(s, t, lr=0.00025, momentum=0.9, weight_decay=0.0005, max_iters=10,
                    cons_scale=1.0, rampup_steps=1, ema_decay=0.99, cons_for_labeled=False)
    for k in range(3):
        img, lab = O.synthetic_batch(100 + k, 4, 2, 97, 97)
        out = mt.step(img.to(D), lab.to(D), 2)
        for key in ('s_task_loss', 't_task_loss', 'cons_loss'):
            rec['mt_%s_%d' % (key, k)] = float(out[key])
        rec['mt_grad_checksum_%d' % k] = checksums([(n, out['grads'][n]) for n in names])
        rec['mt_s_param_checksum_%d' % k] = checksums([(n, mt.s[n]) for n in names])
        rec['mt_t_param_checksum_%d' % k] = checksums([(n, mt.t[n]) for n in names])
        for n in SAMPLE_PARAMS:
            rec['mt_grad_%d/%s' % (k, n)] = sample_of(out['grads'][n].float())
    # SupOnly step (null_step_65.npz)
    s = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(41, cls_bias_std=0.01), 42), D)
    sup = O.MTOracle(s, None, lr=0.00025, momentum=0.9, weight_decay=0.0005, max_iters=10)
    img, lab = O.synthetic_batch(300, 2, 2, 65, 65)
    out = sup.step(img.to(D), lab.to(D), 2)
    rec['null_task_loss'] = float(out['s_task_loss'])
    rec['null_grad_checksum'] = checksums([(n, out['grads'][n]) for n in names])
    rec['null_param_checksum'] = checksums([(n, sup.s[n]) for n in names])
    # CutMix step (cutmix_step_65.npz)
    s = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(51, cls_bias_std=0.01), 52), D)
    t = O.to_dtype(O.randomize_bn_affine(O.init_deeplabv2(61, cls_bias_std=0.01), 62), D)
    cm = O.CutMixOracle(s, t, lr=0.00025, momentum=0.9, weight_decay=0.0005, max_iters=10, cons_scale=20.0,
                        rampup_steps=0, ema_decay=0.99, cons_threshold=0.05)
    img, lab = O.synthetic_batch(400, 6, 2, 65, 65)
    out = cm.step(img.to(D), lab.to(D), 2, np.random.RandomState(4321))
    rec['cutmix_task_loss'], rec['cutmix_cons_loss'] = float(out['task_loss']), float(out['cons_loss'])
    rec['cutmix_grad_checksum'] = checksums([(n, out['grads'][n]) for n in names])
    rec['cutmix_s_param_checksum'] = checksums([(n, cm.s[n]) for n in names])
    rec['cutmix_t_param_checksum'] = checksums([(n, cm.t[n]) for n in names])
    np.savez_compressed(os.path.join(OUT, 'fp64_truth.npz'), **rec)
    print('fp64 truth written')


if __name__ == '__main__':
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)                # tests/test_oracle_golden.py GOLDEN_THREADS: fp32 sums depend on it
    pixelssl, sseg_proxy = patch_and_import()
    which = sys.argv[1:] or ['ops', 'forward', 'mt', 'nullcutmix', 'adv', 's4l', 'gct', 'cct', 'pspnet', 'val', 'input',
                             'valprehandle', 'host', 'fp64']
    if which == ['fp64']:
        golden_fp64()
        sys.exit(0)
    if which == ['fp64algs']:
        golden_fp64_algs()
        sys.exit(0)
    if which == ['fp64mid']:
        golden_fp64_mid()
        sys.exit(0)
    if 'mtmid' in which:
        # mid-size step: crosses the 257 -> 129 -> 65 -> 33 -> 17 feature-map sizes (odd tile edges on every level)
        golden_mt(pixelssl, sseg_proxy, size=257, steps=1)
        golden_fp64_mid()
    if 'ops' in which:
        golden_ops(pixelssl, sseg_proxy)
    if 'forward' in which:
        golden_forward(pixelssl)
    if 'mt' in which:
        golden_mt(pixelssl, sseg_proxy)
    if 'nullcutmix' in which:
        golden_null_cutmix(pixelssl, sseg_proxy)
    if 'adv' in which:
        golden_adv(pixelssl, sseg_proxy)
    if 's4l' in which:
        golden_s4l(pixelssl, sseg_proxy)
    if 'gct' in which:
        golden_gct(pixelssl, sseg_proxy)
    if 'cct' in which:
        golden_cct(pixelssl, sseg_proxy)
    if 'pspnet' in which:
        golden_pspnet(pixelssl)
    if 'val' in which:
        golden_val(pixelssl, sseg_proxy)
    if 'input' in which:
        golden_input(pixelssl, sseg_proxy)
    if 'valprehandle' in which:
        golden_val_prehandle(pixelssl, sseg_proxy)
    if 'host' in which:
        golden_host(pixelssl, sseg_proxy)
    if 'fp64' in which:
        golden_fp64()
