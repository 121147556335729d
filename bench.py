#!/usr/bin/env python
"""Benchmark of the Hebbian pretraining step (BASELINE.json metric) — see DESIGN.md §Measurement.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on host cores
    torchrun --nproc-per-node N ... bench.py --gpus N ...    # one rank per GPU (weak scaling)
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed

A "step" is one Hebbian pretraining step of the reference loop (pretrain_hebbian_unsup_2d.py:181-196):
zero_grad -> forward through the makehebbian()-converted UNet (22 Hebbian layers: conv forward +
soft-WTA update) -> Dice loss + backward on the excluded head -> local_update -> optimizer.step().
Default workload = BASELINE.json configs[1]: 2-D UNet, synthetic GlaS-shaped 64 x 3 x 256 x 256 per GPU.
Rank 0 prints ONE JSON line.
"""
import argparse
import contextlib
import io
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'hebbian-bootstraping-semi-supervised-medical-imaging_b200')
for p in (PKG, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import workloads  # noqa: E402

HEBB_PARAMS = {'mode': 'swta_t', 'k': 50., 'w_nrm': True, 'alpha': 1.}   # reproduce_*_2d.sh:18-27 (K=50)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='c2', choices=['c1', 'c2', 'c4', 'c5', 'c6'])
    ap.add_argument('--head-wgrad', type=int, default=64, help='weight gradients of back-prop head convolutions with at most this many filters through hebb_conv_wgrad (0: all cuDNN)')
    ap.add_argument('--aten-backward', action='store_true', help='c6: differentiate with stock ATen ops instead of the native dgrad/wgrad kernels')
    ap.add_argument('--prec', default=os.environ.get('HEBB_PREC', 'bf16x3'), choices=['fp32', 'bf16x3', 'bf16'])
    ap.add_argument('--batch', type=int, default=0, help='per-GPU batch (0 = the workload default)')
    ap.add_argument('--cpu-sample-batch', type=int, default=0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-layer-profile', action='store_true')
    ap.add_argument('--layers-out', default='', help='write the per-layer stage timings to this JSON file')
    ap.add_argument('--no-fuse', action='store_true', help='keep stock BatchNorm/activation/Upsample modules (hebb.fused off)')
    ap.add_argument('--head-nchw', action='store_true', help='keep the stock back-prop head in NCHW (default: channels_last)')
    ap.add_argument('--cudnn-benchmark', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip the companions of the default line (3-D workload, plain drop-in, GPU-eager reference, element-wise kernels)')
    ap.add_argument('--graph', action='store_true', help='replay the step from a CUDA graph (HebbianStepper(capture=True)); the default for c1/c2/c4')
    ap.add_argument('--no-graph', action='store_true', help='launch every step eagerly')
    ap.add_argument('--fused-adam', action='store_true', help='(default) torch.optim.Adam(fused=True): one multi-tensor kernel for the optimiser step')
    ap.add_argument('--no-fused-adam', action='store_true', help='torch.optim.Adam with its default (for-each) implementation')
    ap.add_argument('--dump-outputs', default='', metavar='DIR',
                    help='after the timed steps, write what the last one computed (network output, loss, parameters after the '
                         'update) as DIR/<name>.npy in float32, for comparing two builds output for output')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    return a


WORKLOADS = {
    # name: (description, default per-GPU batch, cpu sample batch)
    'c1': ('single HebbianConv2d 3->64 k3 soft-WTA, 8x3x128x128', 8, 8),
    'c2': ('2D UNet Hebbian pretraining, synthetic GlaS 256x256 RGB', 64, 4),
    'c4': ('3D UNet Hebbian pretraining, synthetic LA 96x96x80', 8, 1),
    # BASELINE configs[4]: forward throughput of the fine-tune-stage network (hebb alpha = 0, nothing updates).  The XNet
    # dual-branch model is not in the reference tree (SURVEY 8d): the same 2-D UNet on a 3-channel image stands in.
    'c5': ('2D UNet forward only, hebb alpha=0 (fine-tune stage), synthetic 256x256 RGB', 64, 4),
    'c6': ('2D UNet fine-tuning step, hebb alpha=0: forward + back-prop through every layer, synthetic 256x256 RGB', 64, 4),
}


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return dict(hbm=float(d['hbm_gbs']), tf=float(d['bf16_tflops']), tf_sustained=float(d.get('bf16_tflops_sustained', d['bf16_tflops'])),
                    source='measured')
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, source='fallback')


DUMP_MAX_ELEMS = 1 << 22        # per array (16 MB in float32); the three arrays of a dump stay under 64 MB


def dump_outputs(path, arrays):
    """Write each tensor as <path>/<name>.npy in float32.  A tensor of more than DUMP_MAX_ELEMS elements is written as
    a fixed sample of them, flattened: the same seeded indices for every run, so two runs compare element for element."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randint(t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, name + '.npy'), t.cpu().numpy())


# ------------------------------------------------------------------------------------------
def build_model(workload, impl_ours, device, fuse=False, head_wgrad=64):
    """Returns (model, make_batch(batch, seed, device), criterion)."""
    if workload == 'c1':
        if impl_ours:
            import hebb
            torch.manual_seed(0)
            layer = hebb.HebbianConv2d(3, 64, 3, stride=1, padding=1, bias=False, w_nrm=True, mode='swta', k=3.,
                                       patchwise=True, alpha=1.)
        else:
            from oracle import hebb_oracle as O
            torch.manual_seed(0)
            layer = O.OracleHebbConv(2, 3, 64, 3, stride=1, padding=1, bias=False, w_nrm=True, k=3., alpha=1.)

        def batch(b, seed, dev):
            g = torch.Generator().manual_seed(seed)
            return torch.randn(b, 3, 128, 128, generator=g).to(dev), None
        return layer.to(device).train(), batch, None
    if workload in ('c2', 'c5', 'c6'):
        net, excl = workloads.unet2d(3, 2), workloads.EXCLUDE_2D

        def batch(b, seed, dev):
            return workloads.glas_batch(b, 256, seed=seed, device=dev)
    else:
        net, excl = workloads.unet3d(1, 2), workloads.EXCLUDE_3D

        def batch(b, seed, dev):
            return workloads.la_batch(b, (96, 96, 80), seed=seed, device=dev)
    alpha = 0. if workload in ('c5', 'c6') else HEBB_PARAMS['alpha']
    with contextlib.redirect_stdout(io.StringIO()):
        if impl_ours:
            from hebb.makehebbian import makehebbian
            makehebbian(net, exclude=excl, hebb_params=dict(HEBB_PARAMS, alpha=alpha))
        else:
            from oracle import hebb_oracle as O
            O.oracle_makehebbian(net, exclude=excl, k=HEBB_PARAMS['k'], alpha=alpha)
    workloads.init_weights_like_reference(net)            # init_weights_unet(model,'kaiming') after surgery
    if impl_ours and fuse:
        from hebb.fused import fuse_norm_act
        fuse_norm_act(net, head_wgrad=head_wgrad)         # BatchNorm(train)+act, 2x up-sampling / max pooling, head weight gradients on our kernels
    if workload == 'c5':
        return net.to(device).eval(), batch, None
    return net.to(device).train(), batch, workloads.dice_loss


def reference_step(model, opt, crit, x, m):
    """The reference loop body, verbatim in structure (pretrain_hebbian_unsup_2d.py:181-196)."""
    if not model.training:                 # c5: inference-style forward of the alpha=0 network
        with torch.no_grad():
            return model(x).sum()
    opt.zero_grad()
    out = model(x)
    loss = None
    if crit is not None:
        loss = crit(out, m)
        loss.backward()
    for mod in model.modules():
        if hasattr(mod, 'local_update'):
            mod.local_update()
    opt.step()
    return loss


def time_cpu_port(workload, sample_batch, steps, warmup):
    """The oracle (a CPU port of the reference algorithm) on the host cores: samples/s."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model, make_batch, crit = build_model(workload, False, 'cpu')
    lr = 1e-6 if workload != 'c4' else 1e-5
    opt = torch.optim.Adam(model.parameters(), lr=lr)
    x, m = make_batch(sample_batch, 0, 'cpu')
    for _ in range(warmup):
        reference_step(model, opt, crit, x, m)
    t0 = time.perf_counter()
    for _ in range(steps):
        reference_step(model, opt, crit, x, m)
    dt = time.perf_counter() - t0
    return dict(value=sample_batch * steps / dt, ms_per_step=dt / steps * 1e3, cores=cores,
                sample=f'{steps} step(s) of batch {sample_batch} (same shapes as the GPU workload), {warmup} warm-up')


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._th = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {}
        for n in dir(nv):
            if n.startswith('nvmlClocksThrottleReason') or n.startswith('nvmlClocksEventReason'):
                v = getattr(nv, n)
                if isinstance(v, int) and v:
                    names[v] = n.replace('nvmlClocksThrottleReason', '').replace('nvmlClocksEventReason', '')
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit and bit & (bit - 1) == 0:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        if self.nv is not None:
            self._th = threading.Thread(target=self._run, daemon=True)
            self._th.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._th is not None:
            self._th.join(2)

    def summary(self):
        s = sorted(self.samples)
        med = s[len(s) // 2] if s else None
        bad = {'HwSlowdown', 'HwThermalSlowdown', 'SwThermalSlowdown'}
        return dict(sm_mhz=med, sm_max_mhz=self.max_mhz, reasons=sorted(r for r in self.reasons if r not in ('None', 'GpuIdle', 'All')),
                    rejected=bool(bad & self.reasons))


# ------------------------------------------------------------------------------------------
def profile_layers(model, x, flush):
    """Per-layer CUDA-event timings in one extra forward pass on each layer's real input: layers on the fused
    small-channel kernel are timed as a whole step (`fused_ms`), layers on the pack / forward / update kernels
    stage by stage (HEBB_F_ONLY_* re-runs one stage alone)."""
    from hebb import _native
    rows = []

    def hook(mod, inp, out):
        xin = inp[0].detach().contiguous()
        desc = mod._desc(xin.shape, True)
        prec = _native.parse_prec(mod.prec)
        base = _native.F_WNRM | _native.F_UPDATE
        path = _native.layer_path(desc, prec, base)
        g = dict(kind=type(mod).__name__, Cin=mod.in_channels, Cout=mod.out_channels, k=list(mod.kernel_size),
                 x=list(xin.shape), y=list(out.shape), tensor_cores=bool(path >= 1), path={0: 'simt', 1: 'tc', 2: 'fused'}[path])
        P = out.numel() // mod.out_channels
        K = mod.in_channels * int(torch.tensor(mod.kernel_size).prod())
        if mod._transposed:
            P = xin.numel() // mod.in_channels
            K = mod.in_channels
            g['flops_one_contraction'] = 2.0 * P * mod.out_channels * K * int(torch.tensor(mod.kernel_size).prod())
        else:
            g['flops_one_contraction'] = 2.0 * P * mod.out_channels * K
        g['bytes_min'] = 4.0 * (xin.numel() + out.numel()) + 12.0 * mod.weight.numel()
        w = mod._raw(mod.weight.detach())
        scratch_dw = torch.zeros_like(w)
        yb = torch.empty_like(out)
        stages = [('full', 0)] + ([('pack', _native.F_ONLY_PACK), ('fwd', _native.F_ONLY_FWD), ('dw', _native.F_ONLY_DW)] if path == 1 else [])
        for name, fl in stages:
            best = None
            for rep in range(3):
                flush()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                _native.conv_step(desc, xin, w, mod.bias.detach(), float(mod.k), yb, None, scratch_dw, base | fl, prec)
                e1.record()
                e1.synchronize()
                t = e0.elapsed_time(e1)
                best = t if best is None else min(best, t)
            g[name + '_ms'] = best
        if path == 2:
            g['fused_ms'] = g['full_ms']
        rows.append(g)

    hs = [m.register_forward_hook(hook) for m in model.modules() if hasattr(m, 'local_update')]
    was = model.training
    model.eval()              # the hook drives the update stages itself; keep delta_w untouched
    with torch.no_grad():
        model(x)
    model.train(was)
    for h in hs:
        h.remove()
    return rows


def roofline_from_rows(rows, prec, pk):
    """Roofline of the dominant kernel class + every class, from the per-layer stage timings."""
    tc = [r for r in rows if r['path'] == 'tc']
    fu = [r for r in rows if r['path'] == 'fused']
    if not tc and not fu:
        return None
    tot = {s: sum(r[s + '_ms'] for r in tc) for s in ('pack', 'fwd', 'dw')} if tc else {}
    if fu:
        tot['fused'] = sum(r['fused_ms'] for r in fu)
    fl_tc = sum(r['flops_one_contraction'] for r in tc)
    fl_fu = sum(r['flops_one_contraction'] for r in fu)
    by_tc = sum(r['bytes_min'] for r in tc)
    by_fu = sum(r['bytes_min'] for r in fu)
    per = {}
    for k in ('fwd', 'dw'):
        if tot.get(k):
            a = fl_tc / (tot[k] / 1e3) / 1e12
            per[{'fwd': 'fwd_swta_kernel', 'dw': 'dw_swta_kernel'}[k]] = dict(bound='tensor', achieved=a, peak=pk['tf'], unit='TFLOP/s', frac=a / pk['tf'],
                                                                           ms=tot[k], launches_per_step=len(tc))
    if tot.get('pack'):
        by = sum(4.0 * torch.tensor(r['x']).prod().item() * 2.0 for r in tc)        # read fp32, write bf16 hi + lo
        a = by / (tot['pack'] / 1e3) / 1e9
        per['pack_x_kernel'] = dict(bound='hbm', achieved=a, peak=pk['hbm'], unit='GB/s', frac=a / pk['hbm'], ms=tot['pack'], launches_per_step=len(tc))
    if tot.get('fused'):
        a = by_fu / (tot['fused'] / 1e3) / 1e9
        t = 2.0 * fl_fu / (tot['fused'] / 1e3) / 1e12
        per['fused_small_kernel'] = dict(bound='hbm', achieved=a, peak=pk['hbm'], unit='GB/s', frac=a / pk['hbm'], ms=tot['fused'],
                                         launches_per_step=len(fu), tensor_view=dict(achieved=t, unit='TFLOP/s', frac=t / pk['tf'],
                                                                                       note='forward + update flops of these layers'),
                                         note='algorithmic bytes (x once + y once + 3 x weights, SURVEY 8d) of the layers on the fused kernel / their '
                                              'summed CUDA-event time (includes the weight-prep and finalize launches of the step)')
    dom_stage = max(tot, key=tot.get)
    dom = {'fwd': 'fwd_swta_kernel', 'dw': 'dw_swta_kernel', 'pack': 'pack_x_kernel', 'fused': 'fused_small_kernel'}[dom_stage]
    roof = dict(per[dom])
    roof['kernel'] = dom
    roof['traffic'] = None
    roof['traffic_note'] = 'DRAM bytes per launch are not measurable inside the run; the ncu capture of this command is profiles/r2_traffic_c2.json'
    roof['peak_source'] = pk['source'] + (' bf16 burst' if roof['bound'] == 'tensor' else ' copy bandwidth')
    roof['precision'] = prec
    roof['stage_ms'] = tot
    roof['per_kernel'] = per
    if 'fwd_swta_kernel' in per or 'dw_swta_kernel' in per:
        roof['per_stage'] = {k: dict(achieved=per[n]['achieved'], frac=per[n]['frac']) for k, n in (('fwd', 'fwd_swta_kernel'), ('dw', 'dw_swta_kernel')) if n in per}
    t_all = sum(tot.values())
    roof['hbm_view'] = dict(algorithmic_bytes=by_tc + by_fu, achieved=(by_tc + by_fu) / (t_all / 1e3) / 1e9, peak=pk['hbm'], unit='GB/s',
                            frac=(by_tc + by_fu) / (t_all / 1e3) / 1e9 / pk['hbm'], stage_ms_total=t_all,
                            note='all Hebbian layers of the step: algorithmic x + y + 3 x weight bytes / summed stage time')
    return roof


def measure(args, workload, prec, B, steps, warmup, dev, world, rank, fuse=True, head_nchw=False, e2e=True, profile=True,
            capture=False, layers_out='', fused_adam=None, dump_dir=''):
    """Build the workload on `dev`, time `steps` steps (HBM-resident inputs, CUDA events per step, L2 flushed between
    steps, max over ranks) and, optionally, the end-to-end loop (pinned host batch in, loss out) and the per-layer profile.
    dump_dir: write the outputs of the last timed step there (dump_outputs)."""
    import torch.distributed as dist
    from hebb import _native
    from hebb.step import HebbianStepper
    import hebb
    hebb.set_precision(prec)
    desc = WORKLOADS[workload][0]
    torch.manual_seed(1234)
    model, make_batch, crit = build_model(workload, True, dev, fuse=fuse, head_wgrad=args.head_wgrad)
    if (not head_nchw) and hasattr(model, 'out_conv') and workload == 'c2':
        model.out_conv.to(memory_format=torch.channels_last)
        # hand the head its input already in channels_last: cuDNN would otherwise convert the NCHW activation once
        # in the forward and once more (from the saved NCHW tensor) for the weight gradient
        model.out_conv.register_forward_pre_hook(lambda mod, a: (a[0].contiguous(memory_format=torch.channels_last),))
    lr = 1e-6 if workload != 'c4' else 1e-5
    params = [p for p in model.parameters()]
    if fused_adam is None:
        fused_adam = not args.no_fused_adam
    opt = torch.optim.Adam(params, lr=lr, capturable=bool(capture), fused=True if fused_adam else None) if params else None
    stepper = HebbianStepper(model, opt, crit, capture=capture)
    x_host, m_host = make_batch(B, 100 + rank, 'cpu')
    x_pin = x_host.pin_memory()
    m_pin = m_host.pin_memory() if m_host is not None else None
    x = x_pin.to(dev)
    m = m_pin.to(dev) if m_pin is not None else None
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def flush():
        flush_buf.fill_(1)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(warmup, 3)):
        stepper.step(x, m)
    sync_all()

    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    n0, g0 = _native.launch_count(), stepper.graph_launches
    with ClockSampler(dev.index or 0) as clk:
        sync_all()
        t_wall0 = time.perf_counter()
        last = None
        for e0, e1 in evs:
            flush()
            if dump_dir:
                last = None               # the previous step's outputs do not stay allocated through this step
                e0.record()
                last = stepper.step(x, m)
            else:
                e0.record()
                stepper.step(x, m)
            e1.record()
        sync_all()
        t_wall = time.perf_counter() - t_wall0
    if dump_dir and rank == 0:
        out, loss = last
        arrays = {'out': out} if loss is None else {'out': out, 'loss': loss}
        arrays['params'] = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
        dump_outputs(dump_dir, arrays)
        del out, loss, arrays
    del last
    launches = _native.launch_count() - n0 + (stepper.graph_launches - g0)
    dev_ms = sum(e0.elapsed_time(e1) for e0, e1 in evs)
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    res = dict(workload=f'{workload}: {desc}', prec=prec, B=B, lr=lr, value=B * world * steps / (dev_ms / 1e3), ms_per_step=dev_ms / steps,
               launches=int(launches), clocks=clk.summary(), wall_s=t_wall, steps=steps,
               graph=stepper._graph is not None, fused_adam=bool(fused_adam))

    if e2e:
        # The public-API loop a user writes: every step's batch is copied from pinned host memory (on a side
        # stream, double-buffered so step i+1's copy overlaps step i's compute) and the loss is read back.
        copy_stream = torch.cuda.Stream(device=dev)
        bufs = [(x, m), (torch.empty_like(x), torch.empty_like(m) if m is not None else None)]
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        freed = [torch.cuda.Event(), torch.cuda.Event()]

        def prefetch(i):
            xb, mb = bufs[i % 2]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[i % 2])          # the step that last read this buffer is done
                xb.copy_(x_pin, non_blocking=True)
                if mb is not None:
                    mb.copy_(m_pin, non_blocking=True)
                ready[i % 2].record(copy_stream)

        sync_all()
        cur = torch.cuda.current_stream(dev)
        for ev in freed:
            ev.record(cur)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        last = 0.0
        prefetch(0)
        for i in range(steps):
            if i + 1 < steps:
                prefetch(i + 1)
            cur.wait_event(ready[i % 2])
            xb, mb = bufs[i % 2]
            out, loss = stepper.step(xb, mb)
            freed[i % 2].record(cur)
            last = float(loss.item()) if loss is not None else float(out.flatten()[0].item())
        s1.record()
        sync_all()
        t = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
        h2d = x_pin.numel() * x_pin.element_size() + (m_pin.numel() * m_pin.element_size() if m_pin is not None else 0)
        res['e2e'] = {'value': B * world * steps / (e2e_ms / 1e3), 'unit': 'samples/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4,
                      'ms_per_step': e2e_ms / steps, 'last_loss': last}

    res['roofline'] = None
    if profile and rank == 0:
        if workload == 'c1':
            class _W(torch.nn.Module):
                def __init__(s, l):
                    super().__init__(); s.l = l

                def forward(s, z):
                    return s.l(z)
            rows = profile_layers(_W(model), x, flush)
        else:
            rows = profile_layers(model, x, flush)
        res['roofline'] = roofline_from_rows(rows, prec, peaks())
        if layers_out:
            with open(layers_out, 'w') as f:
                json.dump(dict(workload=workload, prec=prec, batch=B, layers=rows), f, indent=1)
    stepper.release()
    del stepper, model, opt, x, m, flush_buf
    _native.release_workspaces()
    torch.cuda.empty_cache()
    return res


def time_gpu_eager(workload, B, dev, steps=2, warmup=1):
    """The reference's own formulation on the GPU: the oracle port's modules (materialised unfold + matmul + softmax in
    stock PyTorch ops, i.e. cuDNN / cuBLAS) run eagerly on the B200 -- SURVEY 8d's "bar on the box" -- with TF32 off and
    on, at a reduced batch (the unfold of the widest layer needs ~0.6 GB per sample); reported per sample."""
    out = {}
    model, make_batch, crit = build_model(workload, False, dev)
    lr = 1e-6 if workload != 'c4' else 1e-5
    opt = torch.optim.Adam(model.parameters(), lr=lr)
    x, m = make_batch(B, 0, dev)
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        for name, tf32 in (('fp32', False), ('tf32', True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            for _ in range(warmup):
                reference_step(model, opt, crit, x, m)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                reference_step(model, opt, crit, x, m)
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[name] = dict(value=B / (ms / 1e3), ms_per_step=ms)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    out['unit'] = 'samples/s'
    out['batch'] = B
    out['kind'] = 'port (oracle modules on cuda: unfold + cuBLAS/cuDNN eager ops)'
    del model, opt, x, m
    torch.cuda.empty_cache()
    return out


def elementwise_gbs(dev, pk):
    """Achieved HBM GB/s of the element-wise kernels of the path (north-star: "achieved HBM GB/s for the elementwise and
    normalisation stages"): normalize() (hebb_wnorm), local_update() (hebb_local_update_multi) on a weight set shaped like
    the 3-D network's (90 M weights, 361 MB) and on the 2-D network's (1.8 M)."""
    from hebb import _native
    res = {}
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for tag, shapes in (('c4_weights', [(1024, 1024, 27), (1024, 512, 27), (512, 512, 27), (512, 512, 27), (512, 256, 27), (256, 256, 27), (256, 256, 27)]),
                        ('c2_weights', [(256, 256, 9), (256, 128, 9), (128, 256, 9), (128, 128, 9), (128, 128, 9), (64, 128, 9), (64, 64, 9)])):
        ws = [torch.randn(s, device=dev) for s in shapes]
        n = sum(w.numel() for w in ws)
        # normalize(): read W, write W/|W| (8 B per weight)
        best = None
        for rep in range(3):
            flush_buf.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for w in ws:
                _native.wnorm(w, w.shape[0], w[0].numel(), 1, 0, w[0].numel())
            e1.record(); e1.synchronize()
            best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
        a = 8.0 * n / (best / 1e3) / 1e9
        res[f'wnorm_kernel/{tag}'] = dict(achieved=a, unit='GB/s', frac=a / pk['hbm'], ms=best, bytes=8.0 * n)
        # local_update(): read grad and delta_w, write grad and zero delta_w (16 B per weight; 12 B when grad is not read)
        grads = [torch.randn_like(w) for w in ws]
        dws = [torch.randn_like(w) for w in ws]
        best = None
        for rep in range(3):
            flush_buf.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _native.local_update_multi(grads, dws, [1.0] * len(ws), [False] * len(ws))
            e1.record(); e1.synchronize()
            best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
        a = 12.0 * n / (best / 1e3) / 1e9
        res[f'local_update_kernel/{tag}'] = dict(achieved=a, unit='GB/s', frac=a / pk['hbm'], ms=best, bytes=12.0 * n)
    res['peak'] = pk['hbm']
    res['peak_source'] = pk['source'] + ' copy bandwidth'
    return res


def run_ours(args):
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    if args.aten_backward:
        os.environ['HEBB_ATEN_BACKWARD'] = '1'
    if args.cudnn_benchmark:
        torch.backends.cudnn.benchmark = True
    desc, dflt_b, cpu_b = WORKLOADS[args.workload]
    B = args.batch or dflt_b
    cpu_b = args.cpu_sample_batch or cpu_b

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = time_cpu_port(args.workload, cpu_b, 2 if args.workload != 'c4' else 1, 1 if args.workload != 'c4' else 0)

    def want_graph(workload):
        return bool(args.graph or (not args.no_graph and workload in ('c1', 'c2', 'c4')))

    graph_error = None
    try:
        main = measure(args, args.workload, args.prec, B, args.steps, args.warmup, dev, world, rank, fuse=not args.no_fuse,
                       head_nchw=args.head_nchw, e2e=True, profile=not args.no_layer_profile, capture=want_graph(args.workload),
                       layers_out=args.layers_out, dump_dir=args.dump_outputs)
    except Exception as e:
        if not want_graph(args.workload):
            raise
        # recording the step failed: say so and measure the eagerly launched step instead
        graph_error = f'{type(e).__name__}: {str(e)[:300]}'
        print(f'[bench] CUDA-graph capture failed ({graph_error}); falling back to eager launches', file=sys.stderr, flush=True)
        torch.cuda.synchronize()
        main = measure(args, args.workload, args.prec, B, args.steps, args.warmup, dev, world, rank, fuse=not args.no_fuse,
                       head_nchw=args.head_nchw, e2e=True, profile=not args.no_layer_profile, capture=False, layers_out=args.layers_out,
                       dump_dir=args.dump_outputs)

    # ---- companions of the headline (single GPU, default workload only): the 3-D half of BASELINE's metric, the plain
    # drop-in number, the reference formulation on this GPU, the element-wise kernels ----
    extras = {}
    if world == 1 and rank == 0 and args.workload == 'c2' and not args.no_extras:
        pk = peaks()
        try:
            plain = measure(args, 'c2', args.prec, B, 3, 3, dev, world, rank, fuse=False, head_nchw=True, e2e=False, profile=False,
                            capture=False, fused_adam=False)
            extras['value_plain_dropin'] = dict(value=plain['value'], ms_per_step=plain['ms_per_step'], unit='samples/s',
                                                note='same step with the stock module tree, launched eagerly: no hebb.fused pass, back-prop head in NCHW, for-each Adam (bench.py --no-fuse --head-nchw --no-graph --no-fused-adam)')
        except Exception as e:          # an extra must never take the headline down
            extras['value_plain_dropin'] = dict(error=str(e)[:200])
        c4 = {}
        for prec in ('bf16x3', 'bf16'):
            try:
                r = measure(args, 'c4', prec, WORKLOADS['c4'][1], 3, 3, dev, world, rank, e2e=True, profile=True, capture=want_graph('c4'),
                            layers_out=(args.layers_out.replace('.json', f'_c4_{prec}.json') if args.layers_out else ''))
                roof = r['roofline'] or {}
                c4[prec] = dict(value=r['value'], unit='samples/s', ms_per_step=r['ms_per_step'], e2e=r.get('e2e'), clocks=r['clocks'],
                                gpu_launches=r['launches'], steps=r['steps'], cuda_graph=r['graph'],
                                roofline=dict(per_stage=roof.get('per_stage'), per_kernel={k: dict(achieved=v['achieved'], unit=v['unit'], frac=v['frac'], ms=v['ms'])
                                                                                             for k, v in (roof.get('per_kernel') or {}).items()},
                                              peak=pk['tf'], peak_source=pk['source'] + ' bf16 burst',
                                              note='dw = the update contraction of all 22 layers: algorithmic 2*P*Cout*K flops / summed CUDA-event time '
                                                   f'({"3-4 MMAs per product (split operands)" if prec == "bf16x3" else "1 MMA per product"})'))
            except Exception as e:
                c4[prec] = dict(error=str(e)[:200])
        c4['config'] = {'workload': 'c4: ' + WORKLOADS['c4'][0], 'per_gpu_batch': WORKLOADS['c4'][1], 'optimizer': 'adam lr=1e-05'}
        extras['c4'] = c4
        try:
            eager = {'c2': time_gpu_eager('c2', 8, dev), 'c4': time_gpu_eager('c4', 1, dev, steps=1, warmup=1)}
            eager['c2']['ours_over_eager_fp32'] = main['value'] / eager['c2']['fp32']['value']
            eager['c2']['ours_over_eager_tf32'] = main['value'] / eager['c2']['tf32']['value']
            if 'value' in c4.get('bf16x3', {}):
                eager['c4']['ours_over_eager_fp32'] = c4['bf16x3']['value'] / eager['c4']['fp32']['value']
                eager['c4']['ours_over_eager_tf32'] = c4['bf16x3']['value'] / eager['c4']['tf32']['value']
            extras['gpu_eager_baseline'] = eager
        except Exception as e:
            extras['gpu_eager_baseline'] = dict(error=str(e)[:200])
        try:
            extras['elementwise'] = elementwise_gbs(dev, pk)
        except Exception as e:
            extras['elementwise'] = dict(error=str(e)[:200])

    if rank == 0:
        lr = main['lr']
        line = {
            'metric': 'hebbian_pretrain_samples_per_sec', 'value': main['value'], 'unit': 'samples/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': main['ms_per_step'], 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': {'fp32': 'f32', 'bf16x3': 'bf16x3 (fp32-equivalent split)', 'bf16': 'bf16'}[args.prec],
            'data': 'synthetic',
            'config': {'workload': f'{args.workload}: {desc}', 'per_gpu_batch': B, 'global_batch': B * world,
                       'hebb_params': HEBB_PARAMS if args.workload != 'c1' else {'mode': 'swta', 'k': 3.0, 'alpha': 1.0},
                       'optimizer': f'adam lr={lr}' + (' (torch.optim.Adam(fused=True))' if main['fused_adam'] else ''), 'precision_mode': args.prec,
                       'fused_norm_act_upsample': (not args.no_fuse) and args.workload != 'c1',
                       'fused_ops': 'BatchNorm(train)+act(+the Dropout behind it) with statistics from the conv epilogue, 2x up-sampling, 2x max pooling, bias+ReLU+dropout of the back-prop head (own Philox dropout stream)' if ((not args.no_fuse) and args.workload != 'c1') else 'none',
                       'head_weight_gradient': ('hebb_conv_wgrad (fp32-equivalent split) for <= %d filters: the fused kernel in weight-gradient mode for 16->64 and 64->32, the tcgen05 update kernel for the 2-class layer' % args.head_wgrad) if ((not args.no_fuse) and args.head_wgrad and args.workload != 'c1') else 'cuDNN',
                       'backward': 'stock ATen' if args.aten_backward else 'native dgrad/wgrad on the tcgen05 kernels where the planner takes the layer',
                       'backprop_head_memory_format': 'nchw' if (args.head_nchw or args.workload != 'c2') else 'channels_last (input converted once, by a forward pre-hook)', 'l2': 'flushed between timed steps (256 MB fill)',
                       'cuda_graph': bool(main['graph']),
                       'cuda_graph_note': ('the whole step (zero-grad, forward, both all-reduces, loss, backward, local_update, Adam) is recorded once by HebbianStepper(capture=True) and replayed; gpu_launches counts the replayed kernel nodes of this library'
                                           if main['graph'] else (f'capture failed: {graph_error}' if graph_error else 'eager launches')),
                       'parallelism': f'dp{world} (batch shards; delta_w summed by one all-reduce issued after the forward, back-prop gradients of the head averaged by a second one)'},
            'e2e': main.get('e2e'),
            'gpu_launches': main['launches'],
            'clocks': main['clocks'],
            'wall_s_timed_region': main['wall_s'],
            'roofline': main['roofline'],
            'cpu_baseline': (dict(value=cpu['value'], unit='samples/s', cores=cpu['cores'], kind='port', sample=cpu['sample'],
                                  ms_per_step=cpu['ms_per_step']) if cpu else None),
        }
        line.update(extras)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_reference(args):
    """The reference's algorithm on the box's host cores (oracle port: /root/reference is not on the box)."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    desc, dflt_b, cpu_b = WORKLOADS[args.workload]
    cpu_b = args.cpu_sample_batch or cpu_b
    r = time_cpu_port(args.workload, cpu_b, args.steps, args.warmup)
    line = {
        'impl': 'reference', 'metric': 'hebbian_pretrain_samples_per_sec', 'value': r['value'], 'unit': 'samples/s',
        'n_gpus': int(os.environ.get('WORLD_SIZE', 1)), 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': r['ms_per_step'],
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': f'{args.workload}: {desc}', 'per_step_sample_batch': cpu_b,
                   'note': 'CPU PyTorch restatement of the reference path (oracle/), all host threads'},
        'cpu_baseline': {'value': r['value'], 'unit': 'samples/s', 'cores': r['cores'], 'kind': 'port', 'sample': r['sample']},
        'e2e': {'value': r['value'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


if __name__ == '__main__':
    a = parse_args()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
