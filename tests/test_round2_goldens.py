"""Round-2 fixtures from the live reference (tests/golden/make_golden.py --round2), held against the CPU oracle:
100-step weight drift of tensor-core-shaped layers, a layer with a non-Identity activation, and the reference
training loop on whole networks for 1 and N optimiser steps (pretrain_hebbian_unsup_2d.py:181-196).  The GPU
twins of these tests live in tests/test_gpu_parity.py."""
import contextlib
import io
import json
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import workloads
from oracle import hebb_oracle as O
from helpers import digest_err, load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G2 = load_golden('hebb_golden_r2.npz')
STEPS = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'network_steps_golden.json')))
G2B = np.load(os.path.join(ROOT, 'tests', 'golden', 'hebb_golden_r2b.npz'))
META2B = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'hebb_golden_r2b_meta.json')))


def sampled_relerr(w, idx, ref_samples):
    got = w.detach().reshape(-1).double().cpu()[torch.from_numpy(idx)]
    ref = torch.from_numpy(ref_samples).double()
    return float((got - ref).norm() / ref.norm())


@pytest.mark.parametrize('opt_name', ['sgd', 'adam'])
@pytest.mark.parametrize('nd', [2, 3])
def test_oracle_drift64_matches_reference(nd, opt_name):
    xs = torch.from_numpy(G2[f'drift64_{nd}d/xs'])
    layer = O.OracleHebbConv(nd, 64, 64, 3, padding=1, bias=False, k=50., alpha=1.)
    with torch.no_grad():
        layer.weight.copy_(torch.from_numpy(G2[f'drift64_{nd}d/w0']))
    lr = STEPS['meta'][f'drift64_{nd}d_{opt_name}']['lr']
    opt = torch.optim.SGD([layer.weight], lr=lr) if opt_name == 'sgd' else torch.optim.Adam([layer.weight], lr=lr)
    layer.train()
    idx = G2[f'drift64_{nd}d/idx']
    for step in range(100):
        opt.zero_grad()
        layer(xs[step % 4])
        layer.local_update()
        opt.step()
        if step == 0:
            assert sampled_relerr(layer.weight, idx, G2[f'drift64_{nd}d_{opt_name}/w1']) < 1e-5
    assert sampled_relerr(layer.weight, idx, G2[f'drift64_{nd}d_{opt_name}/w100']) < 1e-4


@pytest.mark.parametrize('name', ['act_relu_16_16', 'act_relu_32_64'])
def test_oracle_nonidentity_act_matches_reference(name):
    m = STEPS['meta'][name]
    layer = O.OracleHebbConv(2, m['Cin'], m['Cout'], 3, padding=1, bias=True, k=m['k'], alpha=1., act=torch.nn.ReLU())
    with torch.no_grad():
        layer.weight.copy_(torch.from_numpy(G2[name + '/w']))
        layer.bias.copy_(torch.from_numpy(G2[name + '/b']))
    layer.train()
    y = layer(torch.from_numpy(G2[name + '/x']))
    assert float((y - torch.from_numpy(G2[name + '/y'])).norm() / torch.from_numpy(G2[name + '/y']).norm()) < 1e-6
    ref = torch.from_numpy(G2[name + '/dw1'])
    assert float((layer.delta_w - ref).norm() / ref.norm()) < 1e-5


@pytest.mark.parametrize('name', sorted(META2B))
def test_oracle_anisotropic_3d_kernels_match_reference(name):
    """Kernel (3,3,1) / padding (1,1,0) as unet3d_urpc builds its blocks (SURVEY 8f row 4): the reference hands the padding
    tuple to F.pad, which pads from the last dimension backwards -- the output shape is part of the fixture."""
    m = META2B[name]
    layer = O.OracleHebbConv(3, m['Cin'], m['Cout'], tuple(m['kernel']), padding=tuple(m['padding']), bias=True, k=m['k'], alpha=1.)
    with torch.no_grad():
        layer.weight.copy_(torch.from_numpy(G2B[name + '/w']))
        layer.bias.copy_(torch.from_numpy(G2B[name + '/b']))
    layer.train()
    y = layer(torch.from_numpy(G2B[name + '/x']))
    assert list(y.shape) == m['out_shape']
    assert float((y - torch.from_numpy(G2B[name + '/y'])).norm() / torch.from_numpy(G2B[name + '/y']).norm()) < 1e-6
    ref = torch.from_numpy(G2B[name + '/dw1'])
    assert float((layer.delta_w - ref).norm() / ref.norm()) < 1e-5


@pytest.mark.parametrize('name', ['hpca_t2d_6_4', 'hpca_t3d_8_4', 'hpca_t3d_6_40'])
def test_oracle_hpca_t_matches_reference(name):
    m = STEPS['meta'][name]
    x, w = torch.from_numpy(G2[name + '/x']), torch.from_numpy(G2[name + '/w'])
    y = O.convT_activation(x, w, None, (2,) * m['nd'])
    assert float((y - torch.from_numpy(G2[name + '/y'])).norm() / torch.from_numpy(G2[name + '/y']).norm()) < 1e-6
    dw = O.hpca_t_delta(x, y, w, (2,) * m['nd'])
    ref = torch.from_numpy(G2[name + '/dw1'])
    assert float((dw - ref).norm() / ref.norm()) < 1e-5


def build_oracle_net(name):
    if name.startswith('unet2d'):
        net, excl = workloads.unet2d(3, 2), workloads.EXCLUDE_2D
    else:
        net, excl = workloads.UNet3D(1, 2, init_features=4), workloads.EXCLUDE_3D
    O.oracle_makehebbian(net, exclude=excl, k=50., alpha=1.)
    workloads.deterministic_state_(net)
    workloads.disable_dropout_(net)
    return net.train()


def step_inputs(gold):
    gg = torch.Generator().manual_seed(78)
    shape = gold['shape']
    xs = [torch.randn(*shape, generator=gg) for _ in range(2)]
    ms = [torch.randint(0, 2, (shape[0], *shape[2:]), generator=gg) for _ in range(2)]
    return xs, ms


def check_snapshot(net, snap, tol_w, tol_move, lr, w0):
    worst_w = worst_m = 0.0
    for n, p in net.named_parameters():
        if not p.requires_grad:
            continue
        worst_w = max(worst_w, digest_err(p, snap['W'][n]))
        worst_m = max(worst_m, digest_err((p.detach() - w0[n]) / lr, snap['move'][n]))
    assert worst_w < tol_w, worst_w
    assert worst_m < tol_move, worst_m
    return worst_w, worst_m


@pytest.mark.parametrize('name', ['unet2d', 'unet3d_f4', 'unet2d_sgd'])
def test_oracle_training_loop_matches_reference_after_1_and_n_steps(name):
    """The reference loop on the oracle network: W of every trainable tensor after 1 and N steps (norm-wise 1e-4, the
    north-star bound) and the weight MOVEMENT (W_n - W_0)/lr, which Adam makes sign-like and therefore strict."""
    from hebb.step import HebbianStepper
    gold = STEPS['nets'][name]
    net = build_oracle_net(name)
    xs, ms = step_inputs(gold)
    opt = (torch.optim.Adam if gold['opt'] == 'adam' else torch.optim.SGD)(net.parameters(), lr=gold['lr'])
    w0 = {n: p.detach().clone() for n, p in net.named_parameters() if p.requires_grad}
    st = HebbianStepper(net, opt, workloads.dice_loss, allreduce=False)
    for step in range(gold['steps']):
        out, loss = st.step(xs[step % 2], ms[step % 2])
        if str(step + 1) in gold['snaps']:
            snap = gold['snaps'][str(step + 1)]
            assert abs(float(loss) - snap['loss']) < 1e-5
            check_snapshot(net, snap, 1e-6, 5e-2 if step else 1e-3, gold['lr'], w0)


# ---- data-parallel semantics of the stepper on CPU / gloo, world size 2 ----
def _dp_main(rank, world, port, q):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from hebb.step import HebbianStepper
        torch.manual_seed(0)
        # a Hebbian trunk (no BatchNorm: shard statistics would differ from full-batch statistics) + a back-prop head
        net = torch.nn.Sequential(O.OracleHebbConv(2, 3, 8, 3, padding=1, bias=False, k=5., alpha=1.),
                                  torch.nn.ReLU(),
                                  O.OracleHebbConv(2, 8, 8, 3, padding=1, bias=True, k=5., alpha=0.5),
                                  torch.nn.Conv2d(8, 2, 1)).train()
        crit = lambda o, t: ((o - t) ** 2).mean()
        g = torch.Generator().manual_seed(5)
        x, t = torch.randn(4, 3, 8, 8, generator=g), torch.randn(4, 2, 8, 8, generator=g)
        ref = None
        if rank == 0:       # the single-process answer on the full batch
            import copy
            single = copy.deepcopy(net)
            s1 = HebbianStepper(single, torch.optim.SGD(single.parameters(), lr=1e-2), crit, allreduce=False)
            for _ in range(3):
                s1.step(x, t)
            ref = [p.detach().clone() for p in single.parameters()]
        st = HebbianStepper(net, torch.optim.SGD(net.parameters(), lr=1e-2), crit)
        assert st.allreduce and st.world == 2
        for _ in range(3):
            st.step(x[rank * 2:(rank + 1) * 2], t[rank * 2:(rank + 1) * 2])
        mine = [p.detach().clone() for p in net.parameters()]
        gathered = [[torch.zeros_like(p) for _ in range(world)] for p in mine]
        for p, lst in zip(mine, gathered):
            dist.all_gather(lst, p)
        if rank == 0:
            same = all(torch.equal(lst[0], lst[1]) for lst in gathered)
            errs = [float((a - b).norm() / b.norm().clamp_min(1e-30)) for a, b in zip(mine, ref)]
            q.put((same, errs))
    finally:
        dist.destroy_process_group()


def test_data_parallel_step_gloo_world2_replicas_identical_and_equal_full_batch():
    """Two ranks, each on half of the batch: after 3 steps every parameter (Hebbian trunk, a mixed alpha = 0.5 layer,
    the back-prop head) is bit-identical on both ranks and equals the single-process full-batch run (delta_w is summed,
    back-prop gradients of the mean loss are averaged)."""
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29700 + os.getpid() % 200
    procs = [ctx.Process(target=_dp_main, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0
    same, errs = q.get(timeout=5)
    assert same
    assert max(errs) < 1e-5, errs
