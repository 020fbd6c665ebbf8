"""TEST INFRASTRUCTURE ONLY — mints tests/golden/* by running the UNMODIFIED reference
(/root/reference, imported through oracle/reference_loader.py) on seeded inputs with the
deterministic synthetic checkpoint (pgtformer_b200.weights.synth_state_dict, seed 0).

Run in the build container (the reference does not exist on the GPU box):
    python -m oracle.make_golden            # 128^2 fixtures (full tensors)
    python -m oracle.make_golden --full     # 512^2 (the reference's native size, NO size patch) and 1024^2 (size patch)
    python -m oracle.make_golden --video    # first 8 frames of assets/inputdemovideo.mp4 through inference.py's loop
    python -m oracle.make_golden --swin     # the Video-Swin BasicLayer of modules/swin.py (TDRQVAE) on stand-in weights
    python -m oracle.make_golden --tiny     # 64^2 (strided sample of every output)
    python -m oracle.make_golden --swin-spec --checkpoint   # BasicLayer state-dict layout; save_pretrained layout
Inputs are not stored: `golden_input(seed, b, H)` regenerates them bit-exactly.

The full-size fixtures are stored compactly (the raw outputs are 50-200 MB): every code index (int16), the top-2
logit values of every token (the margin that decides whether a code flip is a real error), full logit rows for a
seeded sample of tokens, lq_feat as fp16 (at 1024^2: every other token in y and x), the middle output frame as fp16
(that is what `inference.py:15` consumes), the L2-argmin codes of `TDCRQVAE3.get_codes`, and per-tensor max|ref|.
"""
import argparse
import os
import sys
import time

import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
OPT = os.path.join(ROOT, 'options', 'release_test_stage_IIII_dont_need_align_version.yml')
DEMO_VIDEO = 'assets/inputdemovideo.mp4'          # relative to the reference root
N_LOGIT_ROWS = 384
SAMPLE_STRIDE = 11


def load_network_g():
    with open(OPT) as f:
        return yaml.safe_load(f)['network_g']


def golden_input(seed, b, H):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(b * 3, 3, H, H, generator=g)


def sampled_rows(T, seed):
    """Token rows whose full logit vectors a compact fixture keeps."""
    g = torch.Generator().manual_seed(1000 + seed)
    return torch.randperm(T, generator=g)[:N_LOGIT_ROWS].sort().values


def _reference_model():
    from oracle.reference_loader import build_reference_model
    from pgtformer_b200.spec import build_spec
    from pgtformer_b200.weights import synth_state_dict
    opt = load_network_g()
    arch, spec = build_spec(opt)
    sd = synth_state_dict(spec, 0)
    torch.set_num_threads(os.cpu_count())
    return build_reference_model(opt, sd)


def small():
    from oracle.reference_loader import reference_forward, import_reference, generalise_size
    m = _reference_model()
    ref_mod = import_reference()
    for (seed, b, H) in ((1, 1, 128), (2, 2, 128)):
        x = golden_input(seed, b, H)
        out, logits, lq = reference_forward(m, x, w=1.0, adain=True)
        rec = {'out': out, 'logits': logits, 'lq_feat': lq.contiguous(), 'seed': seed, 'b': b, 'H': H,
               'w': 1.0, 'adain': True}
        # the registered TDCRQVAE3.forward (L2-argmin path) on the same module / weights
        vq = []
        with torch.no_grad():
            for i in range(b):
                generalise_size(m, H, H)
                vq.append(ref_mod.TDCRQVAE3.forward(m, x[i * 3:(i + 1) * 3]))
        rec['vq_out'] = torch.cat([v[0] for v in vq], 0)
        rec['vq_loss'] = torch.stack([v[1] for v in vq])
        rec['vq_codes'] = torch.cat([v[2] for v in vq], 0)
        path = os.path.join(GOLDEN, 'pgtformer_ref_b%d_%d_seed%d.pt' % (b, H, seed))
        torch.save(rec, path)
        print('wrote', path, {k: tuple(v.shape) for k, v in rec.items() if torch.is_tensor(v)})


def compact_record(out, logits, lq, seed, H, lq_stride):
    Fr = out.shape[0]
    T = logits.numel() // logits.shape[-1]
    lo = logits.reshape(T, -1)
    top2 = lo.topk(2, dim=-1)
    rows = sampled_rows(T, seed)
    return {'seed': seed, 'b': Fr // 3, 'H': H, 'w': 1.0, 'adain': True, 'compact': True,
            'codes': lo.argmax(-1).to(torch.int16).view(Fr, H // 16, H // 16),
            'top2': top2.values.float().view(Fr, H // 16, H // 16, 2).contiguous(),
            'logit_rows_idx': rows.to(torch.int32), 'logit_rows': lo[rows].float().contiguous(),
            'logits_absmax': lo.abs().max().item(),
            'lq_feat': lq[:, ::lq_stride, ::lq_stride].to(torch.float16).contiguous(), 'lq_stride': lq_stride,
            'lq_absmax': lq.abs().max().item(),
            'out_mid': out[1::3].to(torch.float16).contiguous(), 'out_absmax': out.abs().max().item()}


def full():
    """512^2 through the UNPATCHED reference (its native size); 1024^2 through `generalise_size`."""
    from oracle.reference_loader import generalise_size, import_reference
    ref_mod = import_reference()
    for (seed, H, lq_stride) in ((3, 512, 1), (4, 1024, 2)):
        m = _reference_model()                          # fresh module: the 512^2 run sees no run-time patch at all
        if H != 512:
            generalise_size(m, H, H)
        x = golden_input(seed, 1, H)
        t0 = time.time()
        with torch.no_grad():
            out, logits, lq = m(x, w=1.0, adain=True)
            vq_codes = ref_mod.TDCRQVAE3.get_codes(m, x)
        rec = compact_record(out, logits, lq, seed, H, lq_stride)
        rec['vq_codes'] = vq_codes.to(torch.int16).view(3, H // 16, H // 16)
        rec['patched'] = H != 512
        path = os.path.join(GOLDEN, 'pgtformer_ref_b1_%d_seed%d_compact.pt' % (H, seed))
        torch.save(rec, path)
        print('wrote %s in %.0f s (%.1f MB)' % (path, time.time() - t0, os.path.getsize(path) / 1e6),
              {k: tuple(v.shape) for k, v in rec.items() if torch.is_tensor(v)})


def read_demo_frames(n):
    """First n frames of the reference's demo video as rgb24 (cv2 decodes BGR)."""
    import cv2
    import numpy as np
    from oracle.reference_loader import REFERENCE_ROOT
    cap = cv2.VideoCapture(os.path.join(REFERENCE_ROOT, DEMO_VIDEO))
    frames = []
    while len(frames) < n:
        ok, f = cap.read()
        if not ok:
            break
        frames.append(cv2.cvtColor(f, cv2.COLOR_BGR2RGB))
    cap.release()
    return np.stack(frames)


def video(n=8):
    """`inference.py:12-19,37-76` on the first n frames of assets/inputdemovideo.mp4 with the reference model (CPU): the
    input frames and the reference's uint8 outputs are stored, so the GPU test needs neither the video nor the reference."""
    import numpy as np
    from oracle import video_oracle as VO
    m = _reference_model()
    frames = read_demo_frames(n)

    def apply_window(win):                               # apply_net_to_frames without the .cuda()
        x = torch.from_numpy(VO.rgbnp2tensor(win))
        with torch.no_grad():
            mid = m(x, w=1.0)[0][1]                      # adain comes from the yml (True), as in inference.py:15
        return VO.tensor2rgb(mid.numpy())

    t0 = time.time()
    restored = np.stack(VO.restore_frames(list(frames), apply_window))
    path = os.path.join(GOLDEN, 'demo_video_first%d.npz' % n)
    np.savez_compressed(path, frames=frames, restored=restored)
    print('wrote %s in %.0f s (%.1f MB)' % (path, time.time() - t0, os.path.getsize(path) / 1e6), frames.shape, restored.shape)


def _reference_swin_module():
    """The reference's `modules/swin.py`, imported with the mmcv / basicsr / timm shims."""
    import importlib.util
    from oracle.reference_loader import REFERENCE_ROOT, _ensure_paths
    _ensure_paths()
    spec = importlib.util.spec_from_file_location('_pgt_reference.modules.swin', os.path.join(REFERENCE_ROOT, 'modules', 'swin.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def swin():
    """The reference's Video-Swin `BasicLayer` (`modules/swin.py:326-405`, imported with the mmcv / basicsr / timm shims)
    on the deterministic stand-in weights of oracle/swin3d_oracle.py: outputs stored as fp16."""
    from oracle import swin3d_oracle as S
    mod = _reference_swin_module()
    for name, c in S.SWIN_CASES.items():
        layer = mod.BasicLayer(c['dim'], c['depth'], c['heads'], c['window']).eval()
        layer.load_state_dict(S.synth_state(layer.state_dict(), c['seed']), strict=True)
        x = S.case_input(name)
        with torch.no_grad():
            y = layer(x)
        path = os.path.join(GOLDEN, 'swin3d_%s.pt' % name)
        torch.save({'case': name, 'out': y.to(torch.float16), 'out_absmax': y.abs().max().item()}, path)
        print('wrote', path, tuple(y.shape), '%.1f KB' % (os.path.getsize(path) / 1e3))


def tiny(seed=7, H=64):
    """The reference's forward at 64^2: every code index and every SAMPLE_STRIDE-th element of out, logits and
    lq_feat (flattened, fp32).  The stride is prime, so the sample walks through every channel of the
    power-of-two-wide tensors."""
    from oracle.reference_loader import reference_forward
    m = _reference_model()
    out, logits, lq = reference_forward(m, golden_input(seed, 1, H), w=1.0, adain=True)
    rec = {'seed': seed, 'b': 1, 'H': H, 'w': 1.0, 'adain': True, 'stride': SAMPLE_STRIDE,
           'codes': logits.argmax(-1).to(torch.int16)}
    for k, v in (('out', out), ('logits', logits), ('lq_feat', lq)):
        rec[k] = v.reshape(-1)[::SAMPLE_STRIDE].clone()
        rec[k + '_shape'] = list(v.shape)
    path = os.path.join(GOLDEN, 'pgtformer_ref_b1_%d_seed%d_strided.pt' % (H, seed))
    torch.save(rec, path)
    print('wrote %s (%.1f KB)' % (path, os.path.getsize(path) / 1e3))


def swin_spec():
    """Parameter / buffer names, shapes and dtypes of the reference's `BasicLayer(256, 4, 8, (5, 5, 5))`, and its
    relative_position_index (values < 729, stored as int16): the state-dict layout `modules/swin.py` reproduces."""
    sd = _reference_swin_module().BasicLayer(256, 4, 8, (5, 5, 5)).state_dict()
    path = os.path.join(GOLDEN, 'swin3d_basic_layer_state_spec.pt')
    torch.save({'spec': {k: (list(v.shape), str(v.dtype)) for k, v in sd.items()},
                'relative_position_index': sd['blocks.0.attn.relative_position_index'].to(torch.int16)}, path)
    print('wrote %s: %d entries (%.1f KB)' % (path, len(sd), os.path.getsize(path) / 1e3))


def checkpoint_layout():
    """What the reference class's `save_pretrained` writes, the layout of a Hub checkpoint such as
    kepeng/pgtformer-base: config.json and the model.safetensors header, both verbatim.  The 500 MB tensor payload is
    not kept; the loader test fills the recorded offsets with seeded values."""
    import gzip
    import json
    import struct
    import tempfile
    from oracle.reference_loader import build_reference_model
    ref = build_reference_model(load_network_g())
    with tempfile.TemporaryDirectory() as d:
        ref.save_pretrained(d)
        with open(os.path.join(d, 'config.json')) as f:
            config = f.read()
        with open(os.path.join(d, 'model.safetensors'), 'rb') as f:
            header = f.read(struct.unpack('<Q', f.read(8))[0]).decode()
    path = os.path.join(GOLDEN, 'reference_checkpoint_layout.json.gz')
    with open(path, 'wb') as f, gzip.GzipFile(fileobj=f, mode='wb', mtime=0) as z:
        z.write(json.dumps({'config.json': config, 'model.safetensors header': header}).encode())
    print('wrote %s (%.1f KB)' % (path, os.path.getsize(path) / 1e3))


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--full', action='store_true')
    ap.add_argument('--video', action='store_true')
    ap.add_argument('--swin', action='store_true')
    ap.add_argument('--tiny', action='store_true')
    ap.add_argument('--swin-spec', action='store_true')
    ap.add_argument('--checkpoint', action='store_true')
    a = ap.parse_args()
    if a.full:
        full()
    if a.video:
        video()
    if a.swin:
        swin()
    if a.tiny:
        tiny()
    if a.swin_spec:
        swin_spec()
    if a.checkpoint:
        checkpoint_layout()
    if not (a.full or a.video or a.swin or a.tiny or a.swin_spec or a.checkpoint):
        small()
