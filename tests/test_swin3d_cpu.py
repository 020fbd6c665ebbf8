"""Video-Swin BasicLayer (SURVEY 8(f) #4): the oracle restatement against fixtures minted from the reference's own
`modules/swin.py` (oracle/make_golden.py --swin), and the drop-in's state-dict layout against the reference module's."""
import pytest
import torch

from conftest import load_golden
from oracle import swin3d_oracle as S


def _oracle_layer(case):
    from modules.swin import BasicLayer                   # this repo's drop-in: used here only for its state-dict layout
    c = S.SWIN_CASES[case]
    shell = BasicLayer(c['dim'], c['depth'], c['heads'], c['window'])
    sd = S.synth_state(shell.state_dict(), c['seed'])
    return c, sd


@pytest.mark.parametrize('case', ['a', 'b'])
def test_oracle_matches_reference_golden(case):
    c, sd = _oracle_layer(case)
    g = load_golden('swin3d_%s.pt' % case)
    with torch.no_grad():
        y = S.basic_layer(sd, '', S.case_input(case), c['depth'], c['heads'], c['window'])
    assert y.shape == g['out'].shape
    assert (y - g['out'].float()).abs().max().item() < 1.5e-3 * g['out_absmax']      # fp16 storage of the fixture


def test_dropin_state_dict_is_reference_compatible():
    """Same parameter / buffer names, shapes and dtypes as the reference's BasicLayer, and the same relative position
    index (recorded from the reference module by oracle/make_golden.py --swin-spec)."""
    from modules.swin import BasicLayer
    ours = BasicLayer(256, 4, 8, (5, 5, 5)).state_dict()
    assert len(ours) == 52 and ours['blocks.1.attn.relative_position_bias_table'].shape == (729, 8)
    ref = load_golden('swin3d_basic_layer_state_spec.pt')
    assert set(ours) == set(ref['spec'])
    assert all(list(ours[k].shape) == shape and str(ours[k].dtype) == dtype for k, (shape, dtype) in ref['spec'].items())
    assert torch.equal(ours['blocks.0.attn.relative_position_index'], ref['relative_position_index'].long())
