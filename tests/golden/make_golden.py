"""Generate tests/golden/hebb_golden.npz + makehebbian_golden.json from the LIVE reference.

Run ONLY in the build container (needs /root/reference, which is not on the GPU
box):  python tests/golden/make_golden.py
The reference modules are imported unchanged under an alias; nothing is copied.
Each case stores what the reference produced (y, argmax winners, delta_w, W
after N optimiser steps), so both the oracle and the CUDA path can be checked
without the reference.  The inputs (x, W, bias) come from one seeded generator
per file and are not stored: tests/helpers.py::load_golden draws them again,
and derives grad after local_update (= -delta_w).
"""
import importlib.util
import io
import json
import os
import sys
import contextlib

import numpy as np
import torch
import torch.nn as nn

REF = os.environ.get('HEBB_REFERENCE', '/root/reference')
HERE = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(HERE))
import helpers  # noqa: E402  (tests/helpers.py: load_golden re-creates the inputs this script does not store)


def load_reference():
    """Import the reference 'hebb' package under the alias 'ref_hebb'."""
    spec = importlib.util.spec_from_file_location(
        'ref_hebb', os.path.join(REF, 'hebb', '__init__.py'),
        submodule_search_locations=[os.path.join(REF, 'hebb')])
    mod = importlib.util.module_from_spec(spec)
    sys.modules['ref_hebb'] = mod
    spec.loader.exec_module(mod)
    mk = importlib.import_module('ref_hebb.makehebbian')
    return mod, mk


CONV_CASES = [
    # name, nd, B, Cin, Cout, kernel, stride, padding, spatial, k, bias
    ('c2d_3x3_p1_k1',      2, 2, 3, 8, 3, 1, 1, (12, 12), 1.0, False),
    ('c2d_3x3_p1_k50',     2, 2, 3, 8, 3, 1, 1, (12, 12), 50.0, False),
    ('c2d_c1_config1',     2, 2, 3, 64, 3, 1, 1, (32, 32), 3.0, False),
    ('c2d_16_16',          2, 2, 16, 16, 3, 1, 1, (20, 24), 50.0, False),
    ('c2d_1x1',            2, 3, 24, 12, 1, 1, 0, (9, 7), 5.0, True),
    ('c2d_stride2_nopad',  2, 2, 3, 16, 3, 2, 0, (15, 15), 10.0, False),
    ('c2d_asym_pad',       2, 1, 4, 6, (3, 3), 1, (2, 1), (8, 10), 2.0, True),
    ('c2d_rect_kernel',    2, 2, 5, 7, (1, 3), 1, (0, 1), (6, 9), 20.0, False),
    ('c3d_3x3x3_p1',       3, 2, 1, 8, 3, 1, 1, (6, 8, 10), 50.0, False),
    ('c3d_8_16',           3, 1, 8, 16, 3, 1, 1, (6, 6, 6), 50.0, False),
    ('c3d_40ch_chunked',   3, 1, 40, 8, 3, 1, 1, (4, 5, 6), 1.0, False),   # > PARALLEL_CHANNELS
    ('c3d_1x1x1',          3, 2, 6, 4, 1, 1, 0, (3, 4, 5), 7.0, True),
]

CONVT_CASES = [
    ('t2d_2x2_s2',  2, 2, 6, 4, 2, 2, (5, 7), 50.0),
    ('t2d_k1',      2, 2, 6, 4, 2, 2, (5, 7), 1.0),
    ('t3d_2x2x2_s2', 3, 2, 8, 4, 2, 2, (3, 4, 5), 50.0),
    ('t3d_40co',    3, 1, 6, 40, 2, 2, (2, 3, 3), 5.0),    # > PARALLEL_CHANNELS out channels
]


def stored(out, redrawn, drawn_again):
    """The arrays of `out` that tests/helpers.py::load_golden does not re-create.  drawn_again: the inputs as
    load_golden draws them (helpers._draw_r1 / _draw_r2), which must equal the ones the reference ran on."""
    mine = {k: v for k, v in out.items() if k.rsplit('/', 1)[1] in ('x', 'w', 'b', 'xs', 'w0')}
    bad = sorted(set(mine) ^ set(drawn_again)) + [k for k in mine if k in drawn_again and
                                                  not np.array_equal(mine[k], drawn_again[k].numpy())]
    if bad:
        raise RuntimeError(f'tests/helpers.py draws other inputs than this script for {bad[:5]}: update its case order')
    return {k: v for k, v in out.items() if k.rsplit('/', 1)[1] not in redrawn}


def main():
    ref, mk = load_reference()
    out = {}
    meta = {}
    g = torch.Generator().manual_seed(20261018)

    def rnd(*shape, scale=1.0):
        return torch.randn(*shape, generator=g) * scale

    for (name, nd, B, Cin, Cout, kernel, stride, padding, spatial, k, bias) in CONV_CASES:
        cls = ref.HebbianConv2d if nd == 2 else ref.HebbianConv3d
        layer = cls(Cin, Cout, kernel, stride=stride, padding=padding, bias=bias,
                    w_nrm=True, mode='swta', k=k, patchwise=True, alpha=1.)
        with torch.no_grad():
            layer.weight.copy_(rnd(*layer.weight.shape, scale=0.3))
            if bias:
                layer.bias.copy_(rnd(Cout, scale=0.1))
        layer.train()
        x = rnd(B, Cin, *spatial)
        y = layer(x)
        dw1 = layer.delta_w.clone()
        y2 = layer(x * 0.5)          # second forward: delta_w must accumulate
        dw2 = layer.delta_w.clone()
        layer.local_update()
        grad = layer.weight.grad.clone()
        out[name + '/x'] = x.numpy()
        out[name + '/w'] = layer.weight.detach().numpy()
        out[name + '/b'] = layer.bias.detach().numpy()
        out[name + '/y'] = y.detach().numpy()
        out[name + '/win'] = y.argmax(dim=1).numpy().astype(np.int32)
        out[name + '/dw1'] = dw1.numpy()
        out[name + '/dw2'] = dw2.numpy()
        out[name + '/grad'] = grad.numpy()
        assert float(layer.delta_w.abs().max()) == 0.0
        meta[name] = dict(kind='conv', nd=nd, B=B, Cin=Cin, Cout=Cout, kernel=kernel, stride=stride,
                          padding=padding, spatial=list(spatial), k=k, bias=bias)

    # HPCA rule (SURVEY 8f row 1; the mode the reference's own test_makehebbian3d exercises)
    for (name, nd, B, Cin, Cout, kernel, padding, spatial, bias) in [
            ('hpca2d_3_8', 2, 2, 3, 8, 3, 1, (10, 12), False), ('hpca2d_16_16', 2, 2, 16, 16, 3, 1, (12, 10), True),
            ('hpca3d_8_16', 3, 1, 8, 16, 3, 1, (5, 6, 7), False), ('hpca3d_40_8', 3, 1, 40, 8, 1, 0, (4, 4, 5), False)]:
        cls = ref.HebbianConv2d if nd == 2 else ref.HebbianConv3d
        layer = cls(Cin, Cout, kernel, stride=1, padding=padding, bias=bias, w_nrm=True, mode='hpca', k=1.,
                    patchwise=True, alpha=1.)
        with torch.no_grad():
            layer.weight.copy_(rnd(*layer.weight.shape, scale=0.3))
            if bias:
                layer.bias.copy_(rnd(Cout, scale=0.1))
        layer.train()
        x = rnd(B, Cin, *spatial)
        y = layer(x)
        out[name + '/x'], out[name + '/w'], out[name + '/b'] = x.numpy(), layer.weight.detach().numpy(), layer.bias.detach().numpy()
        out[name + '/y'], out[name + '/dw1'] = y.detach().numpy(), layer.delta_w.clone().numpy()
        meta[name] = dict(kind='hpca', nd=nd, B=B, Cin=Cin, Cout=Cout, kernel=kernel, stride=1, padding=padding,
                          spatial=list(spatial), bias=bias)

    for (name, nd, B, Cin, Cout, spatial) in [('hpcaT2d_6_4', 2, 2, 6, 4, (5, 7)), ('hpcaT3d_8_4', 3, 1, 8, 4, (3, 4, 5))]:
        cls = ref.HebbianConvTranspose2d if nd == 2 else ref.HebbianConvTranspose3d
        layer = cls(Cin, Cout, 2, stride=2, padding=0, bias=False, w_nrm=True, mode='hpca', k=1., patchwise=True, alpha=1.)
        with torch.no_grad():
            layer.weight.copy_(rnd(*layer.weight.shape, scale=0.3))
        layer.train()
        x = rnd(B, Cin, *spatial)
        y = layer(x)
        out[name + '/x'], out[name + '/w'] = x.numpy(), layer.weight.detach().contiguous().numpy()
        out[name + '/y'], out[name + '/dw1'] = y.detach().numpy(), layer.delta_w.clone().contiguous().numpy()
        meta[name] = dict(kind='hpcaT', nd=nd, B=B, Cin=Cin, Cout=Cout, kernel=2, stride=2, spatial=list(spatial))

    # zero-norm filter + eval()/alpha==0 produce no update
    layer = ref.HebbianConv2d(3, 4, 3, padding=1, bias=False, k=5., alpha=1.)
    with torch.no_grad():
        layer.weight.copy_(rnd(*layer.weight.shape))
        layer.weight[2].zero_()
    x = rnd(2, 3, 6, 6)
    layer.train()
    y = layer(x)
    out['zero_row/x'], out['zero_row/w'] = x.numpy(), layer.weight.detach().numpy()
    out['zero_row/y'], out['zero_row/dw1'] = y.detach().numpy(), layer.delta_w.clone().numpy()
    meta['zero_row'] = dict(kind='conv', nd=2, B=2, Cin=3, Cout=4, kernel=3, stride=1, padding=1,
                            spatial=[6, 6], k=5., bias=False)

    for (name, nd, B, Cin, Cout, kernel, stride, spatial, k) in CONVT_CASES:
        cls = ref.HebbianConvTranspose2d if nd == 2 else ref.HebbianConvTranspose3d
        layer = cls(Cin, Cout, kernel, stride=stride, padding=0, bias=False,
                    w_nrm=True, mode='swta_t', k=k, patchwise=True, alpha=1.)
        with torch.no_grad():
            layer.weight.copy_(rnd(*layer.weight.shape, scale=0.3))
        layer.train()
        x = rnd(B, Cin, *spatial)
        y = layer(x)
        dw1 = layer.delta_w.clone()
        layer.local_update()
        out[name + '/x'] = x.numpy()
        out[name + '/w'] = layer.weight.detach().contiguous().numpy()     # (Cin, Cout, k...)
        out[name + '/y'] = y.detach().numpy()
        out[name + '/win'] = y.argmax(dim=1).numpy().astype(np.int32)
        out[name + '/dw1'] = dw1.contiguous().numpy()
        out[name + '/grad'] = layer.weight.grad.contiguous().numpy()
        meta[name] = dict(kind='convT', nd=nd, B=B, Cin=Cin, Cout=Cout, kernel=kernel, stride=stride,
                          spatial=list(spatial), k=k)

    # multi-step drift: config-1-like layer driven by SGD and Adam for 100 steps
    for opt_name in ('sgd', 'adam'):
        layer = ref.HebbianConv2d(3, 16, 3, padding=1, bias=False, k=10., alpha=1.)
        with torch.no_grad():
            layer.weight.copy_(rnd(*layer.weight.shape, scale=0.3))
        w0 = layer.weight.detach().clone()
        xs = rnd(4, 2, 3, 10, 10)
        opt = (torch.optim.SGD([layer.weight], lr=1e-3) if opt_name == 'sgd'
               else torch.optim.Adam([layer.weight], lr=1e-3))
        layer.train()
        w_after1 = None
        for step in range(100):
            opt.zero_grad()
            layer(xs[step % 4])
            layer.local_update()
            opt.step()
            if step == 0:
                w_after1 = layer.weight.detach().clone()
        out[f'drift_{opt_name}/xs'] = xs.numpy()
        out[f'drift_{opt_name}/w0'] = w0.numpy()
        out[f'drift_{opt_name}/w1'] = w_after1.numpy()
        out[f'drift_{opt_name}/w100'] = layer.weight.detach().numpy()
        meta[f'drift_{opt_name}'] = dict(kind='drift', opt=opt_name, lr=1e-3, k=10., steps=100)

    # contrastive rule (SURVEY 8f row 4; hebb.py:143-172, hebb3d.py:167-197): a loss on the layer output whose
    # weight gradient becomes delta_w.  The rule draws torch.randperm(B) from the global generator: seed it and
    # store the permutation.
    for (name, nd, B, Cin, Cout, spatial, bias, uniformity, contrast) in [
            # (uniformity=True cannot be pinned: the reference's own uniformity branch raises for Cout > 1 --
            #  apply_weights() adds the [Cout] bias to a 1-channel map, hebb.py:75,160)
            #  the 3-D layer cannot either: hebb3d.py:170 calls unfold3d() with a stride of 0 and raises)
            ('ctr2d_3_8', 2, 4, 3, 8, (10, 12), False, False, 1.0), ('ctr2d_16_16', 2, 3, 16, 16, (12, 10), True, False, 0.5),
            ('ctr2d_8_32', 2, 2, 8, 32, (9, 7), True, False, 2.0)]:
        cls = ref.HebbianConv2d if nd == 2 else ref.HebbianConv3d
        layer = cls(Cin, Cout, 3, stride=1, padding=1, bias=bias, w_nrm=True, mode='contrastive', k=1.,
                    contrast=contrast, uniformity=uniformity, alpha=1.)
        with torch.no_grad():
            layer.weight.copy_(rnd(*layer.weight.shape, scale=0.3))
            if bias:
                layer.bias.copy_(rnd(Cout, scale=0.1))
        layer.train()
        x = rnd(B, Cin, *spatial)
        torch.manual_seed(4242)
        perm = torch.randperm(B)
        torch.manual_seed(4242)
        y = layer(x)
        out[name + '/x'], out[name + '/w'], out[name + '/b'] = x.numpy(), layer.weight.detach().numpy(), layer.bias.detach().numpy()
        out[name + '/y'], out[name + '/dw1'] = y.detach().numpy(), layer.delta_w.clone().numpy()
        out[name + '/perm'] = perm.numpy()
        if bias:
            out[name + '/gb'] = layer.bias.grad.detach().numpy()
        meta[name] = dict(kind='contrastive', nd=nd, B=B, Cin=Cin, Cout=Cout, kernel=3, stride=1, padding=1,
                          spatial=list(spatial), bias=bias, uniformity=uniformity, contrast=contrast)

    np.savez_compressed(os.path.join(HERE, 'hebb_golden.npz'), **stored(out, ('x', 'w', 'b', 'xs', 'w0', 'grad'), helpers._draw_r1(meta)))

    # ---- makehebbian structure on the reference test's toy net (tests/test_makehebbian.py:5-39)
    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.down = nn.Sequential(nn.Conv2d(3, 16, 3, stride=2), nn.BatchNorm2d(16), nn.ReLU())
            self.up = nn.Sequential(nn.ConvTranspose2d(16, 20, 3, stride=2), nn.BatchNorm2d(20), nn.ReLU())
            self.clf = nn.Sequential(mk.FlattenLast(2), nn.Linear(20, 16), nn.BatchNorm1d(16), nn.ReLU(),
                                     nn.Dropout(0.5), nn.Linear(16, 10))

        def forward(self, x):
            return self.clf(self.up(self.down(x)))

    def describe(net):
        mods = {n: type(m).__name__ for n, m in net.named_modules()}
        params = {n: [list(p.shape), bool(p.requires_grad), list(p.stride())] for n, p in net.named_parameters()}
        bufs = {n: list(b.shape) for n, b in net.named_buffers()}
        hp = {n: dict(mode=m.mode, k=m.k, alpha=m.alpha, w_nrm=m.w_nrm, patchwise=m.patchwise,
                      kernel_size=list(m.kernel_size), stride=list(m.stride),
                      padding=(m.padding if isinstance(m.padding, int) else list(m.padding)))
              for n, m in net.named_modules() if hasattr(m, 'local_update')}
        return dict(modules=mods, params=params, buffers=bufs, hebb=hp,
                    state_keys=list(net.state_dict().keys()))

    structures = {}
    with contextlib.redirect_stdout(io.StringIO()):
        net = mk.makehebbian(Net(), exclude=['clf.5'], hebb_params={})
        structures['toy_default_params'] = describe(net)
        net = mk.makehebbian(Net(), exclude=['clf.5'],
                             hebb_params={'mode': 'swta_t', 'k': 50., 'w_nrm': True, 'alpha': 1.})
        structures['toy_swta_t'] = describe(net)
        net = mk.makehebbian(Net(), exclude=None, hebb_params=None)
        structures['toy_none'] = describe(net)
    # a checkpoint in the reference's save_snapshot() layout (utils.py:29-55), produced by the reference modules
    torch.manual_seed(7)
    with contextlib.redirect_stdout(io.StringIO()):
        net = mk.makehebbian(Net(), exclude=['clf.5'], hebb_params={'mode': 'swta_t', 'k': 50., 'w_nrm': True, 'alpha': 1.})
    for n_, m_ in net.named_modules():
        if hasattr(m_, 'delta_w'):
            m_.delta_w.normal_()
    torch.save({'model': net.state_dict(), 'threshold': 0.5,
                'hebb_params': {'mode': 'swta_t', 'k': 50., 'w_nrm': True, 'alpha': 1.}, 'excluded_layers': ['clf.5']},
               os.path.join(HERE, 'ref_checkpoint.pth'))
    structures['adjust'] = {
        'swta_t': mk.adjust_hebbian_params({'mode': 'swta_t', 'k': 3}),
        'hpca_t': mk.adjust_hebbian_params({'mode': 'hpca_t'}),
        'swta': mk.adjust_hebbian_params({'mode': 'swta'}),
        'none': mk.adjust_hebbian_params({'k': 2}),
    }
    structures['default_hebb_params'] = {k: (v if not isinstance(v, nn.Module) else type(v).__name__)
                                         for k, v in mk.default_hebb_params.items()}
    with open(os.path.join(HERE, 'makehebbian_golden.json'), 'w') as f:
        json.dump(dict(meta=meta, structures=structures), f, indent=1, sort_keys=True)
    network_goldens(mk)
    print('wrote', len(out), 'arrays;', os.path.getsize(os.path.join(HERE, 'hebb_golden.npz')) // 1024, 'KiB')


def _load_file(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def layer_digest(t, n=48):
    t = t.detach().contiguous().reshape(-1).double()
    idx = torch.linspace(0, t.numel() - 1, min(n, t.numel())).long()
    return dict(sum=float(t.sum()), abssum=float(t.abs().sum()), norm=float(t.norm()),
                idx=idx.tolist(), val=t[idx].tolist())


def network_goldens(mk):
    """Whole-network fixtures: the reference's unet (2-D) and UNet3D (3-D, init_features=4) after
    makehebbian, one training-mode forward + local_update on a small seeded input, dropout off,
    weights from workloads.deterministic_state_.  Also the state_dict key/shape lists that
    tests/test_workloads.py compares the restated topologies with."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    import workloads
    with contextlib.redirect_stdout(io.StringIO()):
        r2 = _load_file(os.path.join(REF, 'models/networks_2d/unet.py'), 'ref_unet2d')
        r3 = _load_file(os.path.join(REF, 'models/networks_3d/unet3d.py'), 'ref_unet3d')
        full2, full3 = r2.unet(3, 2), r3.unet3d(1, 2)
    keys = {'unet2d': [[n, list(v.shape)] for n, v in full2.state_dict().items()],
            'unet3d': [[n, list(v.shape)] for n, v in full3.state_dict().items()]}
    with open(os.path.join(HERE, 'workload_state_keys.json'), 'w') as f:
        json.dump(keys, f)

    res = {}
    hp = {'mode': 'swta_t', 'k': 50., 'w_nrm': True, 'alpha': 1.}
    cases = [('unet2d', lambda: r2.unet(3, 2), workloads.EXCLUDE_2D, (2, 3, 32, 32)),
             ('unet3d_f4', lambda: r3.UNet3D(1, 2, init_features=4), workloads.EXCLUDE_3D, (2, 1, 16, 16, 16))]
    for name, ctor, excl, shape in cases:
        with contextlib.redirect_stdout(io.StringIO()):
            net = ctor()
            mk.makehebbian(net, exclude=excl, hebb_params=hp)
        workloads.deterministic_state_(net)
        workloads.disable_dropout_(net)
        net.train()
        x = torch.randn(*shape, generator=torch.Generator().manual_seed(77))
        out = net(x)
        layers = {}
        for n, m in net.named_modules():
            if hasattr(m, 'local_update'):
                layers[n] = dict(kind=type(m).__name__, delta_w=layer_digest(m.delta_w))
                m.local_update()
                layers[n]['grad'] = layer_digest(m.weight.grad)
        res[name] = dict(shape=list(shape), out=layer_digest(out, 256), layers=layers)
    with open(os.path.join(HERE, 'network_golden.json'), 'w') as f:
        json.dump(res, f)


def round2_goldens():
    """Round-2 fixtures (written to separate files so the round-1 arrays stay byte-identical):
      hebb_golden_r2.npz   100-step weight drift of TENSOR-CORE-shaped layers (Cin = Cout = 64, 3x3 2-D and 3x3x3 3-D)
                           under SGD and Adam, k = 50, plus an act=ReLU layer (the rule sees act(y), hebb.py:80,107)
      network_steps_golden.json   the reference `unet` (2-D) / UNet3D(f=4) driven by the reference training loop
                           (pretrain_hebbian_unsup_2d.py:181-196: zero_grad, forward, loss.backward, local_update of
                           every layer, optimizer.step) for 1 and N steps, Adam with the reference learning rates,
                           dropout off: per-layer digests of W and of the weight movement W_n - W_0."""
    ref, mk = load_reference()
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    import workloads
    out, meta = {}, {}
    g = torch.Generator().manual_seed(20261019)

    def rnd(*shape, scale=1.0):
        return torch.randn(*shape, generator=g) * scale

    for nd, sp, B in ((2, (12, 12), 2), (3, (6, 6, 6), 1)):
        cls = ref.HebbianConv2d if nd == 2 else ref.HebbianConv3d
        w0 = rnd(64, 64, *([3] * nd), scale=(2.0 / (64 * 3 ** nd)) ** 0.5)
        xs = rnd(4, B, 64, *sp)
        out[f'drift64_{nd}d/xs'], out[f'drift64_{nd}d/w0'] = xs.numpy(), w0.numpy()
        idx = torch.linspace(0, w0.numel() - 1, 8192).long()          # W after 1 / 100 steps: 8192 evenly spaced samples
        out[f'drift64_{nd}d/idx'] = idx.numpy()
        for opt_name in ('sgd', 'adam'):
            layer = cls(64, 64, 3, padding=1, bias=False, k=50., alpha=1.)
            with torch.no_grad():
                layer.weight.copy_(w0)
            # SGD: lr 1e-3 (the weights move by ~10 % of their norm in 100 steps).  Adam: lr 1e-5 = the reference's 3-D setting
            # (reproduce_hebbian_unsupervised_pretraining_3d.sh; 10x its 2-D one) -- Adam makes every element move by ~lr per
            # step whatever the update's size, so at lr 1e-3 the weights would travel further than their own magnitude and any
            # two fp32 evaluation orders diverge chaotically
            lr = 1e-3 if opt_name == 'sgd' else 1e-5
            opt = (torch.optim.SGD([layer.weight], lr=lr) if opt_name == 'sgd' else torch.optim.Adam([layer.weight], lr=lr))
            layer.train()
            w1 = None
            for step in range(100):
                opt.zero_grad()
                layer(xs[step % 4])
                layer.local_update()
                opt.step()
                if step == 0:
                    w1 = layer.weight.detach().clone()
            name = f'drift64_{nd}d_{opt_name}'
            out[name + '/w1'] = w1.reshape(-1)[idx].numpy()
            out[name + '/w100'] = layer.weight.detach().reshape(-1)[idx].numpy()
            out[name + '/norms'] = np.array([float(w1.norm()), float(layer.weight.detach().norm())])
            meta[name] = dict(kind='drift64', nd=nd, opt=opt_name, lr=lr, k=50., steps=100, spatial=list(sp), B=B)

    # a layer with a non-Identity activation: the plasticity rule is applied to act(y)
    for (name, Cin, Cout, sp) in [('act_relu_16_16', 16, 16, (12, 10)), ('act_relu_32_64', 32, 64, (9, 11))]:
        layer = ref.HebbianConv2d(Cin, Cout, 3, padding=1, bias=True, w_nrm=True, act=nn.ReLU(), mode='swta', k=5., alpha=1.)
        with torch.no_grad():
            layer.weight.copy_(rnd(*layer.weight.shape, scale=0.3))
            layer.bias.copy_(rnd(Cout, scale=0.1))
        layer.train()
        x = rnd(2, Cin, *sp)
        y = layer(x)
        out[name + '/x'], out[name + '/w'], out[name + '/b'] = x.numpy(), layer.weight.detach().numpy(), layer.bias.detach().numpy()
        out[name + '/y'], out[name + '/dw1'] = y.detach().numpy(), layer.delta_w.clone().numpy()
        meta[name] = dict(kind='act', Cin=Cin, Cout=Cout, spatial=list(sp), k=5., act='relu')
    # mode 'hpca_t' of the transposed layers (hebb.py:266-277, hebb3d.py:291-305); 40 output channels cross the 3-D
    # reference's 32-channel chunking of the triangular decay
    for (name, nd, B, Cin, Cout, sp) in [('hpca_t2d_6_4', 2, 2, 6, 4, (5, 7)), ('hpca_t3d_8_4', 3, 1, 8, 4, (3, 4, 5)),
                                         ('hpca_t3d_6_40', 3, 1, 6, 40, (2, 3, 3))]:
        cls = ref.HebbianConvTranspose2d if nd == 2 else ref.HebbianConvTranspose3d
        layer = cls(Cin, Cout, 2, stride=2, padding=0, bias=False, w_nrm=True, mode='hpca_t', k=1., patchwise=True, alpha=1.)
        with torch.no_grad():
            layer.weight.copy_(rnd(*layer.weight.shape, scale=0.3))
        layer.train()
        x = rnd(B, Cin, *sp)
        y = layer(x)
        out[name + '/x'], out[name + '/w'] = x.numpy(), layer.weight.detach().contiguous().numpy()
        out[name + '/y'], out[name + '/dw1'] = y.detach().numpy(), layer.delta_w.clone().contiguous().numpy()
        meta[name] = dict(kind='hpca_t', nd=nd, B=B, Cin=Cin, Cout=Cout, spatial=list(sp))
    np.savez_compressed(os.path.join(HERE, 'hebb_golden_r2.npz'), **stored(out, ('x', 'w', 'b', 'xs', 'w0'), helpers._draw_r2(meta)))

    with contextlib.redirect_stdout(io.StringIO()):
        r2 = _load_file(os.path.join(REF, 'models/networks_2d/unet.py'), 'ref_unet2d')
        r3 = _load_file(os.path.join(REF, 'models/networks_3d/unet3d.py'), 'ref_unet3d')
    hp = {'mode': 'swta_t', 'k': 50., 'w_nrm': True, 'alpha': 1.}
    res = {}
    # (Adam normalises every element's step to ~lr: its weight movement is sign-like.  The SGD run keeps the
    #  movement linear in the accumulated updates, which makes a strict check of the summed delta_w possible.)
    cases = [('unet2d', lambda: r2.unet(3, 2), workloads.EXCLUDE_2D, (2, 3, 32, 32), 1e-6, 20, 'adam'),
             ('unet3d_f4', lambda: r3.UNet3D(1, 2, init_features=4), workloads.EXCLUDE_3D, (2, 1, 16, 16, 16), 1e-5, 10, 'adam'),
             ('unet2d_sgd', lambda: r2.unet(3, 2), workloads.EXCLUDE_2D, (2, 3, 32, 32), 1e-7, 5, 'sgd')]
    for name, ctor, excl, shape, lr, nsteps, opt_name in cases:
        with contextlib.redirect_stdout(io.StringIO()):
            net = ctor()
            mk.makehebbian(net, exclude=excl, hebb_params=hp)
        workloads.deterministic_state_(net)
        workloads.disable_dropout_(net)
        net.train()
        gg = torch.Generator().manual_seed(78)
        xs = [torch.randn(*shape, generator=gg) for _ in range(2)]
        ms = [torch.randint(0, 2, (shape[0], *shape[2:]), generator=gg) for _ in range(2)]
        opt = torch.optim.Adam(net.parameters(), lr=lr) if opt_name == 'adam' else torch.optim.SGD(net.parameters(), lr=lr)
        w0 = {n: p.detach().clone() for n, p in net.named_parameters() if p.requires_grad}
        snaps = {}
        for step in range(nsteps):
            opt.zero_grad()
            o = net(xs[step % 2])
            loss = workloads.dice_loss(o, ms[step % 2])
            loss.backward()
            for m in net.modules():
                if hasattr(m, 'local_update'):
                    m.local_update()
            opt.step()
            if step in (0, nsteps - 1):
                snaps[str(step + 1)] = dict(
                    loss=float(loss),
                    W={n: layer_digest(p) for n, p in net.named_parameters() if p.requires_grad},
                    move={n: layer_digest((p.detach() - w0[n]) / lr) for n, p in net.named_parameters() if p.requires_grad})
        res[name] = dict(shape=list(shape), lr=lr, steps=nsteps, opt=opt_name, snaps=snaps)
    with open(os.path.join(HERE, 'network_steps_golden.json'), 'w') as f:
        json.dump(dict(meta=meta, nets=res), f)
    print('round-2 goldens written:', os.path.getsize(os.path.join(HERE, 'hebb_golden_r2.npz')) // 1024, 'KiB')


def round2b_goldens():
    """hebb_golden_r2b.npz: anisotropic 3-D kernels / paddings as `unet3d_urpc` builds its blocks
    (models/networks_3d/unet3d_urpc.py:32: kernel (3,3,1), padding (1,1,0)) -- SURVEY 8f row 4.  The reference hands the
    padding tuple to F.pad (hebb3d.py:82-84), which pads from the LAST dimension backwards: (1,1,0) pads W and H by 1 and D
    by 0 while the kernel spans 3 along D and 1 along W, so the output is (D-2, H, W+2).  Parity means reproducing that."""
    ref, mk = load_reference()
    out, meta = {}, {}
    g = torch.Generator().manual_seed(20261020)

    def rnd(*shape, scale=1.0):
        return torch.randn(*shape, generator=g) * scale

    for (name, Cin, Cout, kern, pad, sp) in [('aniso3d_8_16', 8, 16, (3, 3, 1), (1, 1, 0), (7, 9, 10)),
                                             ('aniso3d_32_64', 32, 64, (3, 3, 1), (1, 1, 0), (6, 8, 10)),
                                             ('aniso3d_16_32_k133', 16, 32, (1, 3, 3), (1, 1, 0), (5, 8, 9))]:
        layer = ref.HebbianConv3d(Cin, Cout, kern, padding=pad, bias=True, w_nrm=True, mode='swta', k=5., alpha=1.)
        with torch.no_grad():
            layer.weight.copy_(rnd(*layer.weight.shape, scale=0.3))
            layer.bias.copy_(rnd(Cout, scale=0.1))
        layer.train()
        x = rnd(2, Cin, *sp)
        y = layer(x)
        out[name + '/x'], out[name + '/w'], out[name + '/b'] = x.numpy(), layer.weight.detach().numpy(), layer.bias.detach().numpy()
        out[name + '/y'], out[name + '/dw1'] = y.detach().numpy(), layer.delta_w.clone().numpy()
        meta[name] = dict(kind='aniso3d', Cin=Cin, Cout=Cout, kernel=list(kern), padding=list(pad), spatial=list(sp), k=5.,
                          out_shape=list(y.shape))
    np.savez_compressed(os.path.join(HERE, 'hebb_golden_r2b.npz'), **out)
    with open(os.path.join(HERE, 'hebb_golden_r2b_meta.json'), 'w') as f:
        json.dump(meta, f, indent=1)
    print('wrote hebb_golden_r2b.npz', {k: v['out_shape'] for k, v in meta.items()})


if __name__ == '__main__':
    if '--round2b' in sys.argv:
        round2b_goldens()
    elif '--round2' in sys.argv:
        round2_goldens()
    else:
        main()
