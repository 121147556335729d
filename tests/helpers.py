"""Helpers shared by the test modules."""
import json
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')

# The inputs of the reference runs behind hebb_golden.npz and hebb_golden_r2.npz (weights, biases, images) came from
# one seeded generator per file (tests/golden/make_golden.py), in the case order below.  They are drawn again here
# instead of being stored, which keeps each fixture file under 1 MB; make_golden.py checks that these draws equal its own.
R1_SEED, R2_SEED = 20261018, 20261019
R1_ORDER = ['c2d_3x3_p1_k1', 'c2d_3x3_p1_k50', 'c2d_c1_config1', 'c2d_16_16', 'c2d_1x1', 'c2d_stride2_nopad', 'c2d_asym_pad',
            'c2d_rect_kernel', 'c3d_3x3x3_p1', 'c3d_8_16', 'c3d_40ch_chunked', 'c3d_1x1x1',
            'hpca2d_3_8', 'hpca2d_16_16', 'hpca3d_8_16', 'hpca3d_40_8', 'hpcaT2d_6_4', 'hpcaT3d_8_4', 'zero_row',
            't2d_2x2_s2', 't2d_k1', 't3d_2x2x2_s2', 't3d_40co', 'drift_sgd', 'drift_adam', 'ctr2d_3_8', 'ctr2d_16_16', 'ctr2d_8_32']
R2_ORDER = ['drift64_2d', 'drift64_3d', 'act_relu_16_16', 'act_relu_32_64', 'hpca_t2d_6_4', 'hpca_t3d_8_4', 'hpca_t3d_6_40']


def _draw_r1(meta):
    g = torch.Generator().manual_seed(R1_SEED)
    rnd = lambda *shape, scale=1.0: torch.randn(*shape, generator=g) * scale
    out = {}
    for name in R1_ORDER:
        m = meta[name]
        if m['kind'] == 'drift':
            out[name + '/w0'] = rnd(16, 3, 3, 3, scale=0.3)
            out[name + '/xs'] = rnd(4, 2, 3, 10, 10)
            continue
        kern = list(m['kernel']) if isinstance(m['kernel'], (list, tuple)) else [m['kernel']] * m['nd']
        if name == 'zero_row':                                   # a filter of norm 0
            w = rnd(m['Cout'], m['Cin'], *kern)
            w[2].zero_()
        elif m['kind'] in ('convT', 'hpcaT'):                    # transposed layers: (Cin, Cout, k...)
            w = rnd(m['Cin'], m['Cout'], *kern, scale=0.3)
        else:
            w = rnd(m['Cout'], m['Cin'], *kern, scale=0.3)
        out[name + '/w'] = w
        if m['kind'] in ('conv', 'hpca', 'contrastive') and name != 'zero_row':
            out[name + '/b'] = rnd(m['Cout'], scale=0.1) if m['bias'] else torch.zeros(m['Cout'])
        out[name + '/x'] = rnd(m['B'], m['Cin'], *m['spatial'])
    return out


def _draw_r2(meta):
    g = torch.Generator().manual_seed(R2_SEED)
    rnd = lambda *shape, scale=1.0: torch.randn(*shape, generator=g) * scale
    out = {}
    for name in R2_ORDER:
        if name.startswith('drift64'):
            m = meta[name + '_sgd']
            out[name + '/w0'] = rnd(64, 64, *[3] * m['nd'], scale=(2.0 / (64 * 3 ** m['nd'])) ** 0.5)
            out[name + '/xs'] = rnd(4, m['B'], 64, *m['spatial'])
            continue
        m = meta[name]
        if m['kind'] == 'act':
            out[name + '/w'] = rnd(m['Cout'], m['Cin'], 3, 3, scale=0.3)
            out[name + '/b'] = rnd(m['Cout'], scale=0.1)
            out[name + '/x'] = rnd(2, m['Cin'], *m['spatial'])
        else:                                                    # hpca_t: transposed k = 2 layers
            out[name + '/w'] = rnd(m['Cin'], m['Cout'], *[2] * m['nd'], scale=0.3)
            out[name + '/x'] = rnd(m['B'], m['Cin'], *m['spatial'])
    return out


def load_golden(fname):
    """{name: array} of tests/golden/<fname> (hebb_golden.npz or hebb_golden_r2.npz) together with the inputs of its
    reference runs, drawn again from the fixture's generator seed.  For hebb_golden.npz also the weight gradient the
    reference left after local_update() where the fixture pins it: -delta_w, exactly (alpha = 1)."""
    arrays = dict(np.load(os.path.join(GOLDEN, fname)))
    if fname != 'hebb_golden.npz':
        meta = json.load(open(os.path.join(GOLDEN, 'network_steps_golden.json')))['meta']
        arrays.update({k: v.numpy() for k, v in _draw_r2(meta).items()})
        return arrays
    meta = json.load(open(os.path.join(GOLDEN, 'makehebbian_golden.json')))['meta']
    arrays.update({k: v.numpy() for k, v in _draw_r1(meta).items()})
    for name, m in meta.items():
        if name + '/dw2' in arrays:                       # conv cases: two forwards, then local_update()
            arrays[name + '/grad'] = -arrays[name + '/dw2']
        elif m['kind'] == 'convT':                        # transposed cases: one forward, then local_update()
            arrays[name + '/grad'] = -arrays[name + '/dw1']
    return arrays


def digest_err(t, dg):
    t = t.detach().contiguous().reshape(-1).double().cpu()
    idx = torch.tensor(dg['idx'])
    val = torch.tensor(dg['val'], dtype=torch.float64)
    scale = max(dg['norm'] / max(t.numel(), 1) ** 0.5, 1e-30)
    e_samples = float((t[idx] - val).abs().max() / scale)
    e_norm = abs(float(t.norm()) - dg['norm']) / max(dg['norm'], 1e-30)
    e_sum = abs(float(t.sum()) - dg['sum']) / max(dg['abssum'], 1e-30)
    return max(e_samples, e_norm, e_sum)


# ---- parity report: every GPU parity test records its measured errors; conftest dumps them ----
REPORT = {}


def record(test, case, **vals):
    REPORT.setdefault(test, {})[case] = {k: (float(v) if not isinstance(v, (int, str)) else v) for k, v in vals.items()}
