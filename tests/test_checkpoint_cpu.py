"""Checkpoint formats of the drop-in class (SURVEY 8f #3): HF `config.json + model.safetensors` directories
(`PGTFormer.from_pretrained`, inference.py:118) and BasicSR `.pth` files with `params_ema` (inference_cn.py:124-126),
including the layout of a directory written by the REFERENCE class itself."""
import gzip
import json
import os
import struct

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _model(network_g):
    from archs.pgtformer_arch import PGTFormer
    kw = dict(network_g)
    kw.pop('type', None)
    return PGTFormer(**kw)


def _perturb(model):
    """Make the weights differ from what the constructor synthesises, so a no-op load cannot pass."""
    sd = model.state_dict()
    g = torch.Generator().manual_seed(5)
    for i, (k, v) in enumerate(sd.items()):
        if v.dtype.is_floating_point and i % 7 == 0:
            v.mul_(0.5).add_(torch.randn(v.shape, generator=g) * 0.01)
    return {k: v.clone() for k, v in sd.items()}


def test_hf_directory_round_trip(network_g, tmp_path):
    from archs.pgtformer_arch import PGTFormer
    m = _model(network_g)
    want = _perturb(m)
    m.save_pretrained(str(tmp_path))
    assert {'config.json', 'model.safetensors'} <= set(os.listdir(tmp_path))
    m2 = PGTFormer.from_pretrained(str(tmp_path))
    got = m2.state_dict()
    assert list(got) == list(want) and len(got) == 961
    for k in want:
        assert got[k].dtype == want[k].dtype and torch.equal(got[k], want[k]), k
    assert m2.arch.__dict__ == m.arch.__dict__            # ctor keywords survive config.json
    assert m2.__dict__.get('_engine') is None             # kernel-layout caches are rebuilt lazily after a load


def test_basicsr_params_ema_pth(network_g, tmp_path):
    m = _model(network_g)
    want = _perturb(m)
    path = os.path.join(str(tmp_path), 'net_g_latest.pth')
    torch.save({'params': {k: torch.zeros_like(v) for k, v in want.items()}, 'params_ema': want}, path)
    m2 = _model(network_g)
    state = torch.load(path, map_location='cpu')
    missing = m2.load_state_dict(state['params_ema'], strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    for k, v in m2.state_dict().items():
        assert torch.equal(v, want[k]), k


def test_directory_written_by_the_reference_class_loads(tmp_path):
    """What `PGTFormer.from_pretrained("kepeng/pgtformer-base")` downloads is a directory the reference class wrote.
    config.json and the model.safetensors header are the reference's own, byte for byte (oracle/make_golden.py
    --checkpoint); the tensor payload at the recorded offsets is seeded, so a no-op load cannot pass."""
    from archs.pgtformer_arch import PGTFormer
    with gzip.open(os.path.join(ROOT, 'tests', 'golden', 'reference_checkpoint_layout.json.gz'), 'rt') as f:
        layout = json.load(f)
    (tmp_path / 'config.json').write_text(layout['config.json'])
    header = layout['model.safetensors header'].encode()
    entries = sorted(((k, v) for k, v in json.loads(header).items() if k != '__metadata__'),
                     key=lambda kv: kv[1]['data_offsets'][0])
    g = torch.Generator().manual_seed(11)
    want = {}
    with open(tmp_path / 'model.safetensors', 'wb') as f:
        f.write(struct.pack('<Q', len(header)) + header)
        pos = 0
        for k, v in entries:
            assert v['data_offsets'][0] == pos, k
            if v['dtype'] == 'F32':
                t = torch.randn(v['shape'], generator=g)
            else:
                assert v['dtype'] == 'I64', k
                t = torch.randint(0, 1000, v['shape'], generator=g)
            f.write(t.numpy().tobytes())
            pos = v['data_offsets'][1]
            want[k] = t
    ours = PGTFormer.from_pretrained(str(tmp_path))
    osd = ours.state_dict()
    assert set(want) == set(osd) and len(osd) == 961        # registration order differs, names do not
    for k in want:
        assert osd[k].dtype == want[k].dtype and torch.equal(osd[k], want[k]), k


def test_submodule_load_and_refresh_drop_the_packed_engine(network_g):
    """The packed-weight engine is a derived cache: loading into a submodule (the reference loads the face-parsing
    weights into `conditionnet` separately) or calling refresh() must invalidate it."""
    from archs.pgtformer_arch import PGTFormer
    kw = dict(network_g)
    kw.pop('type')
    m = PGTFormer(**kw)
    marker = object()
    m.__dict__['_engine'] = marker
    m.conditionnet.load_state_dict(m.conditionnet.state_dict())
    assert m.__dict__['_engine'] is None
    m.__dict__['_engine'] = marker
    m.encoder.down.load_state_dict(m.encoder.down.state_dict())
    assert m.__dict__['_engine'] is None
    m.__dict__['_engine'] = marker
    assert m.refresh() is m and m.__dict__['_engine'] is None
