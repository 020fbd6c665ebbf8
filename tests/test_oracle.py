"""CPU tests: pin the oracle restatement (oracle/pgt_oracle.py) against outputs of the
reference itself, stored as golden vectors under tests/golden/ (oracle/make_golden.py)."""
import json
import os

import pytest
import torch

from conftest import ROOT, load_golden
from oracle import pgt_oracle as O
from oracle.make_golden import golden_input

TOL = 2e-5      # fp32 summation-order noise between two CPU formulations (measured 5e-6)


def test_spec_matches_reference_state_dict(arch_spec):
    _, spec = arch_spec
    ref = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'state_dict_spec.json')))
    assert len(spec) == len(ref) == 961
    for k, (shape, dtype) in ref.items():
        assert k in spec, k
        assert list(spec[k][0]) == shape and 'torch.' + spec[k][2] == dtype, k


def test_synth_weights_deterministic(arch_spec):
    from pgtformer_b200.weights import synth_state_dict, relative_position_index
    _, spec = arch_spec
    sub = {k: spec[k] for k in list(spec)[:40]}
    a, b = synth_state_dict(sub, 0), synth_state_dict(sub, 0)
    assert all(torch.equal(a[k], b[k]) for k in a)
    idx = relative_position_index()
    assert idx.shape == (48, 48) and idx.min() == 0 and idx.max() == 244 and idx[0, 0] == 2 * 49 + 3 * 7 + 3


@pytest.mark.parametrize('fixture', ['pgtformer_ref_b1_128_seed1.pt', 'pgtformer_ref_b2_128_seed2.pt'])
def test_oracle_matches_reference_golden(arch_spec, synth_sd, fixture):
    arch, _ = arch_spec
    g = load_golden(fixture)
    x = golden_input(g['seed'], g['b'], g['H'])
    with torch.no_grad():
        out, logits, lq = O.pgtformer_forward(synth_sd, arch, x, w=g['w'], adain_on=g['adain'])
    assert (out - g['out']).abs().max() < TOL * 10
    assert (logits - g['logits']).abs().max() < TOL
    assert (lq - g['lq_feat']).abs().max() < TOL
    assert torch.equal(logits.argmax(-1), g['logits'].argmax(-1))


def test_oracle_vq_path_matches_reference_golden(arch_spec, synth_sd):
    arch, _ = arch_spec
    g = load_golden('pgtformer_ref_b1_128_seed1.pt')
    x = golden_input(g['seed'], g['b'], g['H'])
    with torch.no_grad():
        out, loss, codes = O.tdcrqvae3_forward(synth_sd, arch, x)
    assert torch.equal(codes, g['vq_codes'])
    assert (out - g['vq_out']).abs().max() < TOL * 10
    assert abs(loss.item() - g['vq_loss'].mean().item()) < 1e-4


def test_l2_argmin_exact_agrees_with_fp32_formula(synth_sd):
    cb = synth_sd['quantizer.codebooks.0.weight']
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 8, 8, 512, generator=g)
    a = O.l2_argmin(cb, x)
    b, d = O.l2_argmin_exact(cb, x)
    top2 = d.topk(2, dim=1, largest=False).values
    safe = ((top2[:, 1] - top2[:, 0]) > 1e-4).reshape(a.shape)
    assert torch.equal(a[safe], b[safe]) and safe.float().mean() > 0.99
    assert int(a.max()) < 1024            # padding row excluded


def test_shift_mask_census():
    """4 distinct window patterns per layer; values {0,-100} (SURVEY App. C step 5)."""
    for hw in (8, 32):
        m = O.shift_mask(hw, hw)
        assert set(m.unique().tolist()) == {0.0, -100.0}
        assert len({tuple(w.flatten().tolist()) for w in m}) == 4


def test_oracle_matches_reference_golden_64(arch_spec, synth_sd):
    """At 64^2: every code index and a strided sample of out, logits and lq_feat of the reference (oracle/make_golden.py
    --tiny)."""
    arch, _ = arch_spec
    g = load_golden('pgtformer_ref_b1_64_seed7_strided.pt')
    x = golden_input(g['seed'], g['b'], g['H'])
    with torch.no_grad():
        out, logits, lq = O.pgtformer_forward(synth_sd, arch, x, w=g['w'], adain_on=g['adain'])
    assert torch.equal(logits.argmax(-1), g['codes'].long())
    for name, t in (('out', out), ('logits', logits), ('lq_feat', lq)):
        assert list(t.shape) == g[name + '_shape'], name
        assert (t.reshape(-1)[::g['stride']] - g[name]).abs().max() < TOL * 10, name


def test_oracle_matches_full_size_reference_golden(arch_spec, synth_sd):
    """512^2 is the unpatched reference's native size: the oracle restatement against the compact fixture minted from
    it (every code index, sampled logit rows, lq_feat and the middle output frame stored as fp16)."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    from oracle import pgt_oracle as O
    from oracle.make_golden import golden_input as gi_oracle
    from parity_check import golden_input, load_compact
    g = load_compact(512)
    x = golden_input(g['seed'], g['b'], g['H'])
    assert torch.equal(x, gi_oracle(g['seed'], g['b'], g['H']))
    arch, _ = arch_spec
    with torch.no_grad():
        out, logits, lq = O.pgtformer_forward(synth_sd, arch, x, 1.0, True)
    lo = logits.reshape(-1, logits.shape[-1])
    assert torch.equal(lo.argmax(-1), g['codes'].long().reshape(-1))
    rows = g['logit_rows_idx'].long()
    assert (lo[rows] - g['logit_rows']).abs().max().item() < 2e-5 * g['logits_absmax'] + 1e-5
    assert (lq - g['lq_feat'].float()).abs().max().item() < 1.5e-3 * g['lq_absmax']          # fp16 storage of the fixture
    assert (out[1::3] - g['out_mid'].float()).abs().max().item() < 1.5e-3 * g['out_absmax']
