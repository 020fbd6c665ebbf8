#!/usr/bin/env python
"""bench.py — clips/s of the PGTFormer forward path (BASELINE.json metric) on N B200s.

A "step" is one `PGTFormer.forward` over `--clips` synthetic 3-frame 512x512 clips per GPU
(default 16 = BASELINE configs[2] at N=1, configs[3] at N=8: weak scaling, clips are independent).
  value       whole-job clips/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e         the same metric through the drop-in `PGTFormer.__call__` with HOST (pinned) inputs:
              H2D copy of the clips and D2H copy of `out` every step inside the timed region (on their own
              streams, overlapping the neighbouring step's compute as a serving loop would)
  roofline    dominant kernel (tcgen05 implicit-GEMM conv / GEMM): algorithmic FLOPs / live per-launch
              device time (CUDA events on the launching stream, separate profiled pass of the same steps)
  cpu_baseline  the CPU oracle (port of the reference's PyTorch path) on the host cores, N=1 rank 0 only
`--impl reference` times that CPU path alone (the reference has no CUDA code of its own and cannot
travel to the GPU box; `oracle/pgt_oracle.py` is pinned to it by tests/golden/).
`--dump-outputs DIR` writes what the last timed step computed, from inputs that are the same on every run, so two
builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOPS_PER_CLIP = {128: 236.8e9, 256: None, 512: 3952.0e9, 1024: 17895.0e9}     # SURVEY 8(d), 2*MAC


def config_label(b, H, world):
    """Which BASELINE.json config this run is (configs[2] / [3] are the ones the metric is quoted on)."""
    if H == 512 and b == 16:
        return 'BASELINE configs[2]' if world == 1 else 'BASELINE configs[3] shape: 16 clips/GPU, weak scaling'
    if H == 512 and b == 1 and world == 1:
        return 'BASELINE configs[1]'
    if H == 1024:
        return 'BASELINE configs[4] shape (1024x1024 clips)'
    return 'custom size, not a BASELINE config'


def flops_per_clip(H):
    s = H / 512.0
    return (3952.0e9 - 173.9e9) * s * s + 173.9e9 * s ** 4


def load_network_g():
    import yaml
    with open(os.path.join(ROOT, 'options', 'release_test_stage_IIII_dont_need_align_version.yml')) as f:
        return yaml.safe_load(f)['network_g']


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d, 'measured'
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback'


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons every 200 ms while the timed region runs."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, col in (('hw_slowdown', 5), ('hw_thermal_slowdown', 6), ('sw_thermal_slowdown', 7),
                                  ('sw_power_cap', 8)):
                    if r[col].lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


def cpu_oracle_clips_per_s(H, warmup, steps):
    """Times the CPU oracle (port of the reference forward) one clip per step; returns (clips/s, cores)."""
    import torch
    from oracle import pgt_oracle as O
    from pgtformer_b200.spec import build_spec
    from pgtformer_b200.weights import synth_state_dict
    # all the host threads that help: on the 2x32-core GPU boxes oneDNN/OpenMP is fastest at 16-32 threads and
    # collapses (100x slower) at 128 — measured with tools/cpu_threads.py (256^2 clip: 1.5 s @16-32, 2.5 s @64, 118 s @128)
    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    arch, spec = build_spec(load_network_g())
    sd = synth_state_dict(spec, 0)
    x = torch.rand(3, 3, H, H, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        for _ in range(warmup):
            O.pgtformer_forward(sd, arch, x, 1.0, True)
        t0 = time.perf_counter()
        for _ in range(steps):
            O.pgtformer_forward(sd, arch, x, 1.0, True)
        dt = time.perf_counter() - t0
    return steps / dt, torch.get_num_threads()


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel class, from the committed ncu
    capture of this command (profiles/r2_traffic.json, written by tools/summarize_profiles.py); None if absent."""
    p = os.path.join(ROOT, 'profiles', 'r2_traffic.json')
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def parity_block(model, dev):
    """Golden-vector parity of THIS process's model (same weights, same kernels as the timed steps): the reference's
    own 512^2 outputs and its inference.py loop on the demo video (tools/parity_check.py; fixtures in tests/golden)."""
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    out = {}
    try:
        import parity_check as P
        out['golden_512'] = P.check_compact(model, 512, dev)
        out['demo_video_first8'] = P.check_demo_video(model)
    except Exception as e:                                     # never lose the throughput line to the checker
        out['error'] = repr(e)
    return out


def north_star_kernels(b, H, dev, peaks):
    """Window attention (largest level of the workload) and the nearest-codebook L2 argmin at the workload's token
    count, timed alone: achieved HBM GB/s and tensor TFLOP/s against the measured peaks (burst figures: kernels timed
    in isolation)."""
    import torch
    from pgtformer_b200 import ops
    from pgtformer_b200.weights import relative_position_index
    res = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run(fn, cls, iters=8):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ops.profile_begin()
        for _ in range(iters):
            flush.zero_()
            fn()
        pr = ops.profile_end()
        return pr[cls][1] / max(pr[cls][2], 1)

    try:
        g = torch.Generator().manual_seed(5)
        C, heads, hw = 256, 8, H // 4                           # decoder / encoder level 2: the largest attention level
        T = b * 3 * hw * hw
        qkv = torch.randn(T, 3 * C, generator=g).bfloat16().to(dev)
        bias = (0.02 * torch.randn(245, heads, generator=g))[relative_position_index().view(-1)].view(48, 48, heads)
        tab = ops.window_tables(bias.permute(2, 0, 1).contiguous().to(dev))
        o = torch.empty(T, C, dtype=torch.bfloat16, device=dev)
        ms = run(lambda: ops.window_attention_tc(qkv, b, hw, hw, C, heads, 2, tab, o), 'window_attn')
        by = T * 4 * C * 2
        res['window_attention'] = {'shape': '%d windows of 48 tokens, C=256, 8 heads, shifted' % (T // 48), 'kernel_ms': ms,
                                   'algorithmic_bytes': by, 'achieved_hbm_gbs': by / ms / 1e6,
                                   'hbm_frac': by / ms / 1e6 / peaks['hbm_gbs'],
                                   'achieved_tflops': 4.0 * 48 * 48 * C * (T // 48) / ms / 1e9}
        Tq = b * 3 * (H // 16) ** 2
        cb = torch.randn(1025, 512, generator=g).to(dev)
        z = torch.randn(Tq, 512, generator=g).to(dev)
        idx = torch.empty(Tq, dtype=torch.int64, device=dev)
        pack = ops.codebook_pack(cb, 1024)
        ms = run(lambda: ops.l2_argmin_tc(z, cb, pack, 1024, idx, None), 'l2_argmin')
        fl, by = 2.0 * Tq * 1024 * 512, Tq * 512 * 4 + 1024 * 512 * 4 + Tq * 8
        res['l2_argmin'] = {'shape': 'T=%d tokens x 1024 codes x 512 (random z: the small-margin regime)' % Tq, 'kernel_ms': ms,
                            'achieved_tflops': fl / ms / 1e9, 'tensor_frac': fl / ms / 1e9 / peaks['bf16_tflops'],
                            'algorithmic_bytes': by, 'achieved_hbm_gbs': by / ms / 1e6,
                            'hbm_frac': by / ms / 1e6 / peaks['hbm_gbs'],
                            'exhaustive_fallback_tokens': ops.last_l2_argmin_fallbacks()}
    except Exception as e:
        res['error'] = repr(e)
    return res


DUMP_MAX_ELEMENTS = 4 << 20            # per array: three fp32 arrays stay under 64 MB


def dump_outputs(outputs, directory):
    """Writes each output as <directory>/<name>.npy in float32.  An output with more than DUMP_MAX_ELEMENTS elements is
    replaced by the elements at a fixed seeded sample of flat indices (sorted; the same for every run of one shape), so
    two builds can be compared output for output.  Returns {name: {'shape', 'stored', 'sampled'}}."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    info = {}
    for name, t in outputs.items():
        stored = t
        if t.numel() > DUMP_MAX_ELEMENTS:
            idx = torch.randint(t.numel(), (DUMP_MAX_ELEMENTS,), generator=torch.Generator().manual_seed(0))
            stored = t.reshape(-1)[idx.sort().values.to(t.device)]
        np.save(os.path.join(directory, name + '.npy'), stored.float().cpu().numpy())
        info[name] = {'shape': list(t.shape), 'stored': stored.numel(), 'sampled': stored is not t}
    return info


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path (oracle port), host cores only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    warm = min(args.warmup, 1)
    val, cores = cpu_oracle_clips_per_s(args.size, warm, args.steps)
    sample = '%d steps x 1 clip (3x%dx%d), %d warm-up, fp32 PyTorch CPU' % (args.steps, args.size, args.size, warm)
    line = {'impl': 'reference', 'metric': 'clips_per_s', 'value': val, 'unit': 'clips/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': warm, 'ms_per_step': 1000.0 / val, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'PGTFormer.forward, 1 clip/step of 3x%dx%d on host CPU' % (args.size, args.size),
                       'size': args.size, 'clips_per_step': 1},
            'cpu_baseline': {'value': val, 'unit': 'clips/s', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': val, 'unit': 'clips/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--clips', type=int, default=16, help='clips per GPU per step')
    ap.add_argument('--size', type=int, default=512)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--graph', action='store_true', help='replay the forward from a CUDA graph')
    ap.add_argument('--gather', default='middle_u8', choices=['middle_u8', 'full'],
                    help='N > 1: what the end-of-step all-gather carries (restored middle frames as rgb24, or every fp32 frame)')
    ap.add_argument('--no-parity', action='store_true', help='skip the golden-vector parity block of the JSON line')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last timed step returned (out: the step result, '
                         'logits, lq_feat) as DIR/<name>.npy in float32; arrays over %d elements as a fixed seeded '
                         'sample' % DUMP_MAX_ELEMENTS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from archs.pgtformer_arch import PGTFormer
    from pgtformer_b200 import ops

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    warmup = max(args.warmup, 3)

    opt = load_network_g()
    kw = dict(opt)
    kw.pop('type')
    model = PGTFormer(**kw).to(dev)
    model.eval()
    model.cuda_graph = bool(args.graph)
    b, H = args.clips, args.size
    g = torch.Generator().manual_seed(1 + rank)
    x_host = torch.rand(b * 3, 3, H, H, generator=g).pin_memory()
    x_dev = x_host.to(dev)
    out_host = torch.empty(b * 3, 3, H, H, dtype=torch.float32).pin_memory()
    from pgtformer_b200.parallel import gather_frames, gather_restored

    def collective(out):
        # the path's one collective (SURVEY 8e), NCCL: the restored middle frames as rgb24 — what the consumer of the
        # path keeps (inference.py:15-19) — or, with --gather full, every fp32 output frame
        if world == 1:
            return out
        return gather_frames(out, world * b) if args.gather == 'full' else gather_restored(out, world * b)

    last = {}

    def step_resident():
        out, last['logits'], last['lq_feat'] = model(x_dev, w=1, adain=True)
        last['out'] = collective(out)
        return last['out']

    # end to end as a serving loop would run it: the pinned-host -> device copy of step k+1 and the device -> host copy
    # of step k's result ride their own streams and overlap the compute of the neighbouring step; every step still does
    # both copies inside the timed region (finish_e2e joins the side streams before the closing event)
    main_stream = torch.cuda.current_stream(dev)
    h2d_stream, d2h_stream = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def step_e2e():
        with torch.cuda.stream(h2d_stream):
            xd = x_host.to(dev, non_blocking=True)
        main_stream.wait_stream(h2d_stream)
        xd.record_stream(main_stream)
        out = model(xd, w=1, adain=True)[0]
        if model.cuda_graph:
            out = out.clone()                                   # the graph's static output is rewritten by the next replay
        gathered = collective(out)                              # N > 1: the collective is part of the end-to-end step too
        d2h_stream.wait_stream(main_stream)
        with torch.cuda.stream(d2h_stream):
            out_host.copy_(out, non_blocking=True)
        out.record_stream(d2h_stream)
        return gathered

    def finish_e2e():
        main_stream.wait_stream(h2d_stream)
        main_stream.wait_stream(d2h_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, finish=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if finish is not None:
            finish()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    # kernels per forward, counted by the library on an eager forward (a graph replay launches the same kernels without
    # passing through the C ABI's launch counter)
    model.cuda_graph = False
    ops.reset_launch_count()
    model(x_dev, w=1, adain=True)
    launches_per_forward = ops.launch_count()
    model.cuda_graph = bool(args.graph)
    for _ in range(warmup):
        step_resident()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.reset_launch_count()
    ms = timed(step_resident, args.steps)
    launches = ops.launch_count() if not args.graph else launches_per_forward * args.steps
    clocks = sampler.stop() if rank == 0 else None
    value = world * b * args.steps / (ms / 1000.0)
    # before the e2e pass: with --graph the outputs are static tensors the next replay rewrites
    dumped = dump_outputs(last, args.dump_outputs) if rank == 0 and args.dump_outputs else None

    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps, finish_e2e)
    e2e_val = world * b * args.steps / (ms_e2e / 1000.0)

    # roofline of the dominant kernel: separate profiled pass (events around every launch of the class)
    torch.cuda.synchronize()
    model.cuda_graph = False                                   # the profiler brackets individual launches
    ops.profile_begin()
    for _ in range(args.steps):
        model(x_dev, w=1, adain=True)
    prof = ops.profile_end()
    peaks, peak_kind = measured_peaks()

    # the two north_star kernels that are not the dominant class, measured on their own at this workload's shapes
    # (events around each launch inside the library; L2 flushed between launches)
    ns_kernels = north_star_kernels(b, H, dev, peaks) if rank == 0 else None
    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_block(model, dev)

    if rank == 0:
        work, pms, n = prof['gemm_tc']
        achieved = work / (pms / 1000.0) / 1e12 if pms > 0 else 0.0
        peak = float(peaks.get('bf16_tflops_sustained', 1400.0))
        total_ms = sum(v[1] for v in prof.values())
        breakdown = {k: {'ms_per_step': v[1] / args.steps, 'launches_per_step': v[2] / args.steps,
                         'work_per_step': v[0] / args.steps} for k, v in prof.items() if v[2] > 0}
        line = {
            'metric': 'clips_per_s', 'value': value, 'unit': 'clips/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
            'config': {'workload': 'PGTFormer.forward on %d clips/GPU of 3x%dx%d (%s), w=1, adain, '
                                   'random-init pgtformer-base' % (b, H, H, config_label(b, H, world)),
                       'clips_per_gpu': b, 'size': H, 'global_clips': world * b, 'parallelism': 'dp%d' % world,
                       'l2_policy': 'inputs and activations (GBs per step) exceed the 126 MB L2; no flush needed',
                       'flops_per_clip': flops_per_clip(H), 'cuda_graph': bool(args.graph)},
            'e2e': {'value': e2e_val, 'unit': 'clips/s', 'ms_per_step': ms_e2e / args.steps,
                    'h2d_bytes_per_step': x_host.numel() * 4, 'd2h_bytes_per_step': out_host.numel() * 4},
            'gpu_launches': launches,
            'clocks': clocks,
            'roofline': {'bound': 'tensor', 'kernel': 'gemm_tc_kernel (tcgen05 implicit-GEMM conv / GEMM)',
                         'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak,
                         'peak_kind': peak_kind + ' bf16_tflops_sustained', 'traffic': None,
                         'launches_per_step': n / args.steps, 'kernel_ms_per_step': pms / args.steps,
                         'share_of_profiled_kernel_time': pms / total_ms if total_ms > 0 else None,
                         'pass': 'separate profiled pass of the same %d steps' % args.steps,
                         'end_to_end_frac': value / world * flops_per_clip(H) / (peak * 1e12)},
            'kernel_breakdown': breakdown,
            'north_star_kernels': ns_kernels,
            'parity': parity,
        }
        if dumped is not None:
            line['dumped_outputs'] = {'dir': args.dump_outputs, 'arrays': dumped}
        tr = load_traffic()
        if tr is not None:
            line['roofline']['traffic'] = tr.get('dram_bytes_per_launch')
            line['roofline']['traffic_source'] = tr.get('source')
            line['roofline']['algorithmic_bytes_per_launch'] = tr.get('algorithmic_bytes_per_launch')
        if world > 1:
            line['config']['collective'] = ('all_gather of the restored middle frames (rgb24, %d B/rank)' % (b * H * H * 3)
                                            if args.gather == 'middle_u8' else
                                            'all_gather of every fp32 output frame (%d B/rank)' % (b * 9 * H * H * 4))
        if world == 1 and not args.no_cpu_baseline:
            try:
                v, cores = cpu_oracle_clips_per_s(H, 1, 1)
                line['cpu_baseline'] = {'value': v, 'unit': 'clips/s', 'cores': cores, 'kind': 'port',
                                        'sample': '1 clip (3x%dx%d) timed once after 1 warm-up, fp32 PyTorch CPU oracle' % (H, H)}
            except Exception as e:                     # never lose the GPU line to a CPU-side problem
                line['cpu_baseline'] = {'value': None, 'unit': 'clips/s', 'cores': os.cpu_count(), 'kind': 'port',
                                        'sample': 'failed: %r' % (e,)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
