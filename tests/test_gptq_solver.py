"""SURVEY.md 8(f) rank 4: the GPTQ solver (`gptq.GPTQ`, drop-in for the reference module) against what the reference's own `gptq.py`
computes on the same layers and calibration batches: scales, zeros, g_idx and the on-grid weights must agree.  The reference's results are
stored in tests/golden/solver_ref.npz (written by tests/golden/make_solver_golden.py from the unmodified reference); CPU."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'solver_ref.npz')
CASES = [(256, 96, 4, 64, False), (256, 96, 4, 128, True), (192, 64, 3, -1, False), (256, 64, 8, 128, False), (256, 96, 2, 32, True)]
H_SAMPLES = 2048  # Hessian entries stored per case, spread over the K x K matrix


def case_name(K, N, bits, groupsize, actorder):
    return f'K{K}_N{N}_b{bits}_g{groupsize}' + ('_act' if actorder else '')


def run_solver(gptq_cls, K, N, bits, groupsize, actorder):
    """One seeded layer + calibration set through `gptq_cls` (ours or the reference's GPTQ, same interface).  Returns the Hessian, the
    fasterquant outputs and the layer's on-grid weights."""
    g = torch.Generator().manual_seed(K + N + bits)
    lin = nn.Linear(K, N, bias=True)
    lin.weight.data = torch.randn(N, K, generator=g) * 0.05
    # correlated calibration inputs with a few dominant (and one dead) features, so that act-order actually reorders
    mix = torch.randn(K, K, generator=g) * 0.2 + torch.eye(K)
    gain = torch.rand(K, generator=g) * 3 + 0.1
    gain[5] = 0.0
    batches = [(torch.randn(2, 24, K, generator=g) @ mix) * gain for _ in range(3)]
    s = gptq_cls(lin)
    s.quantizer.configure(bits, perchannel=True, sym=False, mse=False)
    for x in batches:
        s.add_batch(x, None)
    H = s.H.clone()
    scale, zero, g_idx, err = s.fasterquant(blocksize=128, percdamp=.01, groupsize=groupsize, actorder=actorder, name='t')
    return dict(H=H, scale=scale.cpu(), zero=zero.cpu(), g_idx=g_idx.cpu(), W=lin.weight.data.clone(), err=err, x=batches[0].reshape(-1, K))


def h_sample_index(K):
    return torch.arange(H_SAMPLES) * 7919 % (K * K)  # stride coprime with K * K: distinct entries


def grid_codes(r):
    """The on-grid weights as integer codes: W = scale[:, g] * (q - zero[:, g]) for column k in group g = g_idx[k]."""
    g = r['g_idx'].long()
    return torch.round(r['W'] / r['scale'][:, g] + r['zero'][:, g])


@pytest.fixture(scope='module')
def reference():
    return dict(np.load(GOLDEN))


@pytest.mark.parametrize('K,N,bits,groupsize,actorder', CASES)
def test_solver_matches_reference_gptq(reference, K, N, bits, groupsize, actorder):
    import gptq as ours_mod
    assert 'gptq-for-llama_b200' in ours_mod.__file__
    name = case_name(K, N, bits, groupsize, actorder)
    ref = {k[len(name) + 1:]: v for k, v in reference.items() if k.startswith(name + '/')}
    r = run_solver(ours_mod.GPTQ, K, N, bits, groupsize, actorder)
    assert torch.allclose(torch.from_numpy(ref['H_sample']), r['H'].flatten()[h_sample_index(K)], rtol=1e-5, atol=1e-6)
    sa, za, ga = (torch.from_numpy(ref[k]) for k in ('scale', 'zero', 'g_idx'))
    sb, zb, gb, eb = r['scale'], r['zero'], r['g_idx'], r['err']
    assert torch.equal(ga, gb) and sa.shape == sb.shape and za.shape == zb.shape
    if actorder:
        assert not torch.equal(gb, (torch.arange(K) // (groupsize if groupsize != -1 else K)).int())  # the fixture really exercises the permutation
    # the same algorithm in fp32 with a different operation order: scales / zeros agree closely, a handful of weights may land on a neighbouring grid point
    assert torch.allclose(sa, sb, rtol=1e-4, atol=1e-7)
    assert (za != zb).float().mean().item() < 0.01
    ga = ga.long()
    Wa = sa[:, ga] * (torch.from_numpy(ref['codes']).float() - za[:, ga])
    Wb = r['W']
    step = sb.mean().item()
    differing = ((Wa - Wb).abs() > 0.5 * step).float().mean().item()
    assert differing < 0.01, f'{differing:.2%} of the quantised weights differ'
    ea = float(ref['err'])
    assert abs(ea - eb) <= 0.02 * abs(ea) + 1e-9
    # and the point of the exercise: the layer output error stays small and comparable
    x = r['x']
    assert torch.allclose(x @ Wa.t(), x @ Wb.t(), rtol=0, atol=0.05 * (x @ Wa.t()).abs().mean().item() + 1e-6)
    sys.modules.pop('gptq', None)


def test_quantize_linears_drives_a_block_with_bias_layers():
    """OPT / GPT-NeoX wiring (opt.py:249-285, neox.py:234-273): their blocks are nn.Linear WITH bias; the generic sequential recipe quantises them
    through forward hooks and leaves on-grid weights behind for QuantLinear.pack."""
    import gptq as ours_mod
    torch.manual_seed(0)

    class Block(nn.Module):
        def __init__(self):
            super().__init__()
            self.fc1, self.fc2 = nn.Linear(64, 128, bias=True), nn.Linear(128, 64, bias=True)

        def forward(self, x):
            return self.fc2(torch.relu(self.fc1(x)))

    blk = Block()
    before = {n: p.detach().clone() for n, p in blk.named_parameters()}
    res = ours_mod.quantize_linears(blk, [torch.randn(4, 16, 64) for _ in range(2)], wbits=4, groupsize=32, act_order=False)
    assert set(res) == {'fc1', 'fc2'}
    for n, (scale, zero, g_idx, err) in res.items():
        lin = getattr(blk, n)
        K = lin.in_features
        assert scale.shape == (lin.out_features, K // 32) and zero.shape == scale.shape and g_idx.shape == (K, ) and err >= 0
        assert torch.equal(before[n + '.bias'], lin.bias.detach())  # biases are untouched (they travel as fp16 buffers of QuantLinear)
        # every weight sits on its group's grid: w = scale * (q - zero), q integer in [0, 15]
        q = lin.weight.data / scale.repeat_interleave(32, dim=1) + zero.repeat_interleave(32, dim=1)
        assert torch.allclose(q, q.round(), atol=1e-3) and q.min() >= -1e-3 and q.max() <= 15 + 1e-3
        assert (lin.weight.data - before[n + '.weight']).abs().mean() < scale.mean()  # moved by quantisation + error compensation, not destroyed
    sys.modules.pop('gptq', None)
