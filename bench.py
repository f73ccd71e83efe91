"""bench.py — headline benchmark of the render + SR hot path (BASELINE.json: rendered frames/sec @512^2, 64^2 NeRF, 48 samples/ray).

One "step" = one batch of `--batch` frames per GPU: resident tri-planes -> fused render (64x64 rays x 48 samples) -> SR to 512^2 -> frames.
N = 1 is BASELINE configs[2]; N > 1 is configs[3]: the clip's frames are sharded over the ranks (steps x batch frames per GPU, weak scaling),
every step's frames are exchanged inside the timed region and the clip is complete on rank 0 when the clock stops.
Prints ONE JSON line on rank 0; DESIGN.md §5 explains every field.  The same line carries, under roofline.extra.configs, short measurements
of BASELINE configs[1] (render only) and configs[4] (48+48 samples + the torso/background SR head) so that one driver run records them.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes the frames the last timed step returned to DIR/frames.npy, so that two builds run with the same arguments (and
therefore the same seeded inputs) can be compared output for output.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR_GFLOP_PER_FRAME = 197.63          # SURVEY.md §8d (FlopCounter probe of the reference SR, exact)
SAMPLE_BYTES_PER_FRAME = 103.0e6     # stand-alone sample_from_planes op, S=48 (SURVEY.md §8d)
RENDER_BYTES_PER_FRAME = 26.51e6     # fused render, S=48: planes 25.17 MB + jitter 0.79 MB + outputs 0.56 MB (SURVEY.md §8d)
RENDER_GFLOP_PER_FRAME = 1.84        # decoder 1.636 GFLOP + ~0.2 GFLOP interpolation / composite (SURVEY.md §8d)
WARP_CONV_GFLOP_PER_FRAME = 782.0    # torso head conv stack without the torso warper (SURVEY.md §8d); 685 with the per-clip cache
METRIC = 'rendered frames/sec @512^2 (64^2 NeRF, 48 samples/ray)'
DUMP_BYTES = 64 * 10 ** 6            # --dump-outputs budget: larger outputs keep a seeded selection of whole frames


def dump_frames(out_dir, frames):
    """frames [F,...] (fp32 or uint8) -> out_dir/frames.npy in float32.  Above DUMP_BYTES a fixed seeded selection of whole frames is kept
    (in frame order), the same selection for every run with the same arguments."""
    a = frames.detach().float().cpu()
    per_frame = a[0].numel() * a.element_size()
    if a.numel() * a.element_size() > DUMP_BYTES:
        keep = torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:max(1, DUMP_BYTES // per_frame)]
        a = a[keep.sort().values]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'frames.npy'), a.numpy())


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return {'hbm_gbs': d['hbm_gbs'], 'tf_burst': d['bf16_tflops'], 'tf_sustained': d.get('bf16_tflops_sustained', d['bf16_tflops']),
                'src': 'measured'}
    return {'hbm_gbs': 6650.0, 'tf_burst': 1590.0, 'tf_sustained': 1400.0, 'src': 'fallback'}


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/ncu_traffic.json); None when the
    kernel source changed since the capture (stale numbers are not reported)."""
    p = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if not os.path.exists(p):
        return None, 'no capture committed'
    d = json.load(open(p))
    sha = hashlib.sha256(open(os.path.join(ROOT, 'real3dportrait_b200', 'csrc', 'sr_tc.cu'), 'rb').read()).hexdigest()[:16]
    if d.get('sr_tc_cu_sha16') != sha:
        return None, f"stale: captured at {d.get('commit')} for sr_tc.cu {d.get('sr_tc_cu_sha16')}, source is now {sha}"
    return d['bytes_per_launch'], f"{d.get('what')}; captured at commit {d.get('commit')} ({d.get('file')})"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region (B200_PROFILING.md recipe).  Read through NVML in-process (what nvidia-smi
    itself calls) every 20 ms: spawning `nvidia-smi` several times a second from a side thread stalled the driver long enough to cost
    the PCIe-bound e2e loop a quarter of its H2D rate.  Falls back to the nvidia-smi query if NVML cannot be loaded."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows, self.source = index, threading.Event(), [], 'nvml'
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            pr = torch.cuda.get_device_properties(index)
            self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(f'{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0')
            self.max_sm = int(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml, self.source = None, 'nvidia-smi'

    def _sample_nvml(self):
        n = self.nvml
        sm = int(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        try:
            mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
            mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        self.rows.append([str(sm), str(self.max_sm)] + [('Active' if mask & bit else 'Not Active') for bit in (0x8, 0x40, 0x20, 0x4)])

    def run(self):
        while not self.stop_flag.is_set():
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    out = subprocess.run(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-i', str(self.index)],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.split(',')])
            except Exception:
                pass
            self.stop_flag.wait(0.02 if self.nvml is not None else 0.5)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith('active')})
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_min_mhz': sm[0] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(self.rows), 'source': self.source}


def host_threads():
    """Threads the CPU baseline may really use: min(cpu_count, affinity mask, cgroup cpu quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = max(1, min(n, int(float(q) / float(per))))
    except Exception:
        pass
    return n


# ---- CPU baseline: the reference's own modules (oracle/_ref, staged by oracle/make_ref.py) or, if they are absent, the oracle port ----------
def cpu_frame_fn(n_frames, workload='frame'):
    """-> (callable running `n_frames` frames of the workload on the host, kind)."""
    from real3dportrait_b200 import synthetic as syn
    from oracle import ref_runner
    fine = 48 if workload == 'torso' else 0
    planes, cam = syn.make_planes(n_frames, seed=0), syn.make_cameras(n_frames, seed=1)
    u_c, u_f = syn.make_jitter(n_frames, 4096, 48, fine, seed=2)
    mlp = syn.make_decoder_params(seed=4)
    srp = syn.make_sr_warp_params(seed=6) if workload == 'torso' else syn.make_sr_params(seed=5)
    cond = syn.make_warp_inputs(n_frames, seed=7) if workload == 'torso' else None
    if ref_runner.available():
        head = ref_runner.Head(mlp, srp, S=48, S_imp=fine, torso=workload == 'torso', warp_hparams=syn.WARP_HPARAMS, torso_model=syn.StubTorsoModel())
        return (lambda: head.frame(planes, cam, u_c, u_f, cond=cond, sr=workload != 'render')), 'reference'
    from oracle import real3d_oracle as orc
    c2w, K = syn.split_camera(cam)

    def run():
        with torch.no_grad():
            if workload == 'render':
                o, d = orc.gen_rays(c2w, K, 64)
                return orc.render(planes, mlp, o, d, S=48, u_coarse=u_c, lib=True)[0]
            if workload == 'torso':
                o, d = orc.gen_rays(c2w, K, 64)
                feat, _, wsum, _ = orc.render(planes, mlp, o, d, S=48, S_imp=48, u_coarse=u_c, u_fine=u_f, lib=True)
                fimg, wimg = orc.feature_image(feat, 64), orc.feature_image(wsum, 64)
                return orc.superres_warp(fimg[:, :3], fimg, torch.ones(n_frames, 14, 512), cond['ref_torso_rgb'], cond['ref_bg_rgb'], wimg, cond['segmap'],
                                         cond['kp_s'], cond['kp_d'], srp, syn.StubTorsoModel())[0]
            return orc.frame(planes, mlp, srp, c2w, K, u_coarse=u_c, lib=True)['image']
    return run, 'port'


def time_cpu(n_frames, reps, warm=1, budget_s=45.0, workload='frame'):
    """Median frames/s on the host.  Tries the full thread count and (if that is > 32) 32 threads, because torch's CPU convolutions often
    run SLOWER when heavily over-threaded; reports the best, with the count used."""
    fn, kind = cpu_frame_fn(n_frames, workload)
    best = None
    cands = [host_threads()] + ([32] if host_threads() > 32 else [])
    for nt in cands:
        torch.set_num_threads(nt)
        t_start = time.perf_counter()
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            t = time.perf_counter(); fn(); ts.append(time.perf_counter() - t)
            if time.perf_counter() - t_start > budget_s / len(cands):
                break
        ts.sort()
        fps = n_frames / ts[len(ts) // 2]
        if best is None or fps > best[0]:
            best = (fps, ts, nt, kind)
    return best


def workload_text(args, world):
    base = (f'batch={args.batch} frames/step/GPU, 64x64 rays x 48 samples on 3x32x256x256 fp32 tri-planes + SR 64^2->512^2 '
            f'(197.63 GFLOP/frame), random-init weights')
    if world == 1:
        return 'BASELINE configs[2]: ' + base
    return (f'BASELINE configs[3]: synthetic clip sharded over {world} GPUs ({args.steps} steps x {args.batch} = {args.steps * args.batch} frames per GPU, '
            f'weak scaling), frames exchanged every step and the clip reassembled on rank 0 inside the timed region; per GPU: ' + base)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of this workload on the host cores (oracle/_ref = the reference's unmodified
    modules staged by oracle/make_ref.py; the oracle port only if they are absent).  Same frames per step and step counts as the GPU arm,
    bounded so the run ends within a few minutes."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    B = args.batch
    t_probe = time.perf_counter()
    fn, kind = cpu_frame_fn(B)
    torch.set_num_threads(host_threads())
    fn()                                                            # first call: lazy initialisation + a timing probe
    probe = time.perf_counter() - t_probe
    steps = max(1, min(args.steps, int(150.0 / max(probe, 1e-3))))  # ~150 s of timed work at most
    warm = max(0, min(args.warmup, 1)) if probe > 20 else max(1, min(args.warmup, 2))
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(steps):
        t = time.perf_counter(); fn(); ts.append(time.perf_counter() - t)
    tot = sum(ts)
    fps = B * len(ts) / tot
    nthr = host_threads()
    line = {'impl': 'reference', 'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus, 'steps': len(ts), 'warmup': warm + 1,
            'ms_per_step': 1e3 * tot / len(ts), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': workload_text(args, args.gpus), 'frames_per_step_per_gpu': B, 'samples_per_ray': 48, 'render_res': 64, 'out_res': 512},
            'setup': {'note': f'each step = the same batch of {B} frames on the host CPU (rank 0 only; the frames of one GPU\'s step); steps bounded to ~150 s of work '
                              f'({len(ts)} of the requested {args.steps})'},
            'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': nthr, 'kind': kind,
                             'sample': f'{len(ts)} steps x {B} frames (render 64^2x48 + SR) through '
                                       + ('the reference\'s unmodified modules (oracle/_ref)' if kind == 'reference' else 'the oracle port')
                                       + f', torch CPU threads={nthr}'},
            'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


# ---- helpers for the GPU arm ---------------------------------------------------------------------------------------------------------------
def timed_loop(fn, steps, warmup, barrier, dist, dev, after=None):
    """warm-up, barrier + sync, `steps` calls between CUDA events on the current stream, barrier + sync; returns max-over-ranks ms."""
    for i in range(warmup):
        fn(i)
    if after is not None:
        after()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(warmup + i)
    if after is not None:
        after()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


class GraphPool:
    """One CUDA graph per resident input batch for a plain callable (used by the render-only and torso mini-benchmarks)."""

    def __init__(self, fn, n):
        self.graphs = []
        pool = None
        for i in range(n):
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                fn(i); fn(i)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool):
                out = fn(i)
            pool = pool or g.pool()
            self.graphs.append((g, out))

    def __call__(self, i):
        g, out = self.graphs[i % len(self.graphs)]
        g.replay()
        return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=32)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--batch', type=int, default=4)
    ap.add_argument('--pool', type=int, default=32, help='distinct resident frames per GPU (32 x 25 MB = 805 MB > L2)')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--sr-mode', default=None, choices=[None, 'fp32', 'tc', 'tc_exact'])
    ap.add_argument('--planes', default='cl', choices=['cl', 'nchw'],
                    help="resident tri-plane layout: 'cl' = channels-last as the producer's conv emits them (no repack in the step); "
                         "'nchw' = the reference's [N,3,32,256,256] (repacked every step)")
    ap.add_argument('--exchange', default='auto', choices=['auto', 'allgather', 'p2p'], help='N > 1: how the frames reach the clip')
    ap.add_argument('--frames-f32', action='store_true', help='exchange fp32 NCHW frames instead of uint8 HWC video frames')
    ap.add_argument('--sustain-seconds', type=float, default=2.0, help='extra back-to-back run of this length for the sustained (power-capped) number; 0 = skip')
    ap.add_argument('--no-extra-configs', action='store_true', help='skip the configs[1] / configs[4] mini-benchmarks')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='launch every kernel from Python instead of replaying one CUDA graph per step')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write the frames of the last timed step to DIR/frames.npy '
                                                          '(float32; above 64 MB a seeded selection of whole frames)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the frames of the GPU path; it does not apply to --impl reference')
    args.warmup = max(args.warmup, 3)
    if args.impl == 'reference':
        return run_reference(args)

    import real3dportrait_b200 as r3
    from real3dportrait_b200 import _capi, synthetic as syn, engine, renderer as ren

    rank, world, local = int(os.environ.get('RANK', '0')), int(os.environ.get('WORLD_SIZE', '1')), int(os.environ.get('LOCAL_RANK', '0'))
    assert world == args.gpus, f'--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    L = _capi.lib()
    _capi.check(L.r3dp_device_info(None, None, None))

    sr_mode = args.sr_mode or engine.default_sr_mode()
    u8 = (world > 1) and not args.frames_f32 and sr_mode in ('tc', 'tc_exact')
    exchange = 'none' if world == 1 else ('p2p' if args.exchange in ('auto', 'p2p') else 'allgather')
    exchange_note = ''

    def make_engine(exch):
        e = engine.FrameEngine(batch=args.batch, sr_mode=sr_mode, device=dev, world=world, rank=rank, dist=dist, use_graph=not args.no_graph,
                               hp={'num_samples_fine': 0}, out_uint8=u8, exchange=exch)
        e.load_params(syn.make_decoder_params(seed=4), syn.make_sr_params(seed=5))
        return e

    eng = make_engine(exchange)
    B, P = args.batch, max(args.pool, args.batch)
    nb = P // B
    # resident inputs: every rank owns its own shard of the clip (different seeds per rank)
    planes = syn.make_planes(P, seed=100 + rank).to(dev)
    cams = syn.make_cameras(P, seed=200 + rank).to(dev)
    u_c = syn.make_jitter(P, 4096, 48, 0, seed=300 + rank)[0].to(dev)
    sl = lambda i: slice((i % nb) * B, (i % nb) * B + B)                     # P/B distinct resident batches, cycled
    planes_cl_all = ren.planes_to_channels_last(planes).data                 # [P,3,256,256,32]: what a channels-last producer leaves in HBM
    torch.cuda.synchronize()
    res_nchw = [(planes[sl(i)], cams[sl(i)], u_c[sl(i)]) for i in range(nb)]
    res_cl = [(ren.PlanesCL(planes_cl_all[sl(i)]), cams[sl(i)], u_c[sl(i)]) for i in range(nb)]
    resident = res_cl if args.planes == 'cl' else res_nchw

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    if exchange == 'p2p':
        try:
            eng.open_clip(args.steps * B)
        except Exception as e:                                               # noqa: BLE001  (no CUDA IPC between these processes: fall back)
            flag = torch.tensor([1], device=dev)
            exchange_note = f'p2p unavailable ({type(e).__name__}: {e}); '
        else:
            flag = torch.tensor([0], device=dev)
        dist.all_reduce(flag)
        if int(flag.item()) > 0:
            exchange = 'allgather'
            eng = make_engine(exchange)
            exchange_note += 'fell back to the NCCL all-gather'
    eng.prepare(resident)                                                    # one step graph per resident batch: inputs are read in place

    last = [None]                                                            # what the last step returned (the engine reuses the buffer)

    def step(i):
        last[0] = eng.step(*resident[i % nb], frame_index=((i - args.warmup) % args.steps) * B if i >= args.warmup else 0)
        return last[0]

    sampler = ClockSampler(local); sampler.start()
    launches0 = L.r3dp_launch_count()
    ms = timed_loop(step, args.steps, args.warmup, barrier, dist, dev, after=eng.wait_gather)
    launches = L.r3dp_launch_count() - launches0
    if eng.graph is not None or eng.inplace:        # kernels replayed from the captured graph are not re-counted by the library
        launches = eng.launches_per_step * args.steps
    if args.dump_outputs and rank == 0:
        dump_frames(args.dump_outputs, last[0])
    if exchange == 'p2p':
        eng.close_clip()
    fps = world * B * args.steps / (ms / 1e3)

    # ---- sustained run: the same loop back to back for --sustain-seconds (power-capped regime)
    sustained = None
    if args.sustain_seconds > 0:
        k = max(args.steps, int(args.sustain_seconds * 1e3 / (ms / args.steps)))
        eng.exchange_saved, eng.exchange = eng.exchange, ('none' if eng.exchange == 'p2p' else eng.exchange)     # the clip holds only `steps` steps
        ms_s = timed_loop(lambda i: eng.step(*resident[i % nb]), k, 1, barrier, dist, dev, after=eng.wait_gather)
        eng.exchange = eng.exchange_saved
        sustained = {'seconds': ms_s / 1e3, 'steps': k, 'value': world * B * k / (ms_s / 1e3), 'ms_per_step': ms_s / k}

    # ---- the other resident layout, for comparison (same engine, same kernels except the repack)
    other = res_nchw if args.planes == 'cl' else res_cl
    eng_o = make_engine('none')
    eng_o.prepare(other)
    ms_o = timed_loop(lambda i: eng_o.step(*other[i % nb]), args.steps, 3, barrier, dist, dev)
    del eng_o

    # ---- dominant kernel live timing (SR convolutions) over the same steps, CUDA events on the launching stream
    prof_eng = make_engine('none')
    prof = prof_eng.profile_steps(lambda i: resident[i % nb], args.warmup, args.steps)
    del prof_eng
    barrier()

    # ---- end-to-end through the public call with HOST buffers (pinned, the reference's NCHW plane layout), H2D + D2H inside the timed region
    numa = {}
    e2e_eng = make_engine('none')
    with engine.gpu_local_cpus(torch.cuda.current_device(), report=numa):      # pinned staging buffers on the GPU's NUMA node
        h_planes = planes[:B].cpu().pin_memory(); h_cams = cams[:B].cpu().pin_memory(); h_u = u_c[:B].cpu().pin_memory()
        h_out = torch.empty((B,) + e2e_eng.frame_shape(), dtype=e2e_eng.frame_dtype()).pin_memory()
    ksteps = max(8, min(args.steps, 32))
    t_host0 = time.perf_counter()
    ms_e = timed_loop(lambda i: e2e_eng.step_host(h_planes, h_cams, h_u, h_out), ksteps, 3, barrier, dist, dev, after=e2e_eng.sync_host)
    e2e_wall_ms = (time.perf_counter() - t_host0) * 1e3
    del e2e_eng
    clocks = sampler.summary()                    # sampled from the start of the timed region to the end of the e2e region (GPU busy throughout)
    e2e_fps = world * B * ksteps / (ms_e / 1e3)
    h2d = h_planes.numel() * 4 + h_cams.numel() * 4 + h_u.numel() * 4
    d2h = h_out.numel() * h_out.element_size()

    # ---- BASELINE configs[1]: render only (rays -> fused render), one CUDA graph per resident batch
    extra_cfg = {}
    if not args.no_extra_configs:
        head = eng.head
        sampler_mod = r3.RaySampler()

        def render_only(i):
            pl, cm, uu = res_cl[i % nb]
            o, d = sampler_mod(cm[:, :16].reshape(-1, 4, 4), cm[:, 16:25].reshape(-1, 3, 3), 64)
            return head.renderer(pl, head.decoder, o, d, dict(head.rendering_kwargs, u_coarse=uu))[0]
        gp = GraphPool(render_only, nb) if not args.no_graph else render_only
        ms_r = timed_loop(gp, args.steps, 3, barrier, dist, dev)
        us_frame = 1e3 * ms_r / args.steps / B
        extra_cfg['configs[1] render only'] = {
            'value': world * B * args.steps / (ms_r / 1e3), 'unit': 'frames/s (64x64x48 feature images)', 'us_per_frame': us_frame, 'ms_per_step': ms_r / args.steps,
            'kernel': 'render_stream_kernel (gather || tcgen05 decode || march) + ray generation, limits, depth clamp',
            'hbm_GBps_algorithmic': RENDER_BYTES_PER_FRAME / (us_frame * 1e-6) / 1e9, 'hbm_frac_of_peak': RENDER_BYTES_PER_FRAME / (us_frame * 1e-6) / 1e9 / peaks()['hbm_gbs'],
            'decoder_TFLOPs_algorithmic': RENDER_GFLOP_PER_FRAME / us_frame * 1e3,
            'note': '26.51 MB / 1.84 GFLOP per frame (SURVEY.md §8d): the HBM floor is loose here, the bound is L2->SM gather traffic + MUFU (DESIGN.md §4)'}
        del gp

        # ---- BASELINE configs[4]: 48 + 48 samples/ray + SuperresolutionHybrid8XDC_Warp (stub torso warper), per-clip constants cached
        if sr_mode == 'tc':
            hp5 = dict(syn.WARP_HPARAMS, num_samples_fine=48)
            head5 = r3.RenderHead(hp=hp5, torso_model=syn.StubTorsoModel())
            sd = {'decoder.' + k: v for k, v in syn.make_decoder_params(seed=4).items()}
            sd.update({'superresolution.' + k: v for k, v in syn.make_sr_warp_params(seed=6).items()})
            head5.load_state_dict(sd, strict=True)
            head5 = head5.to(dev).eval()
            u_f = syn.make_jitter(P, 4096, 48, 48, seed=300 + rank)[1].to(dev)
            inp = {k: v.to(dev) for k, v in syn.make_warp_inputs(1, seed=7).items()}
            kp_d = (torch.rand(P, 68, 3, generator=torch.Generator().manual_seed(9)) * 2 - 1).to(dev)
            cond_static = {'ref_torso_img': inp['ref_torso_rgb'].expand(B, -1, -1, -1).contiguous(), 'bg_img': inp['ref_bg_rgb'].expand(B, -1, -1, -1).contiguous(),
                           'segmap': inp['segmap'].expand(B, -1, -1, -1).contiguous(), 'kp_s': inp['kp_s'].expand(B, -1, -1).contiguous()}
            sr5 = head5.superresolution
            sr5.assume_shared_styles = True
            res5 = {}
            for cached in (False, True):
                if cached:
                    sr5.begin_clip(inp['ref_torso_rgb'], inp['ref_bg_rgb'])

                def torso_step(i):
                    pl, cm, uu = res_cl[i % nb]
                    s = sl(i)
                    cond = dict(cond_static, kp_d=kp_d[s])
                    return head5.synthesis(pl, cm, cond=cond, u_coarse=uu, u_fine=u_f[s.start * 4096:s.stop * 4096])['image']
                gp5 = GraphPool(torso_step, min(nb, 4)) if not args.no_graph else torso_step
                k5 = max(6, args.steps // 2)
                res5[cached] = timed_loop(gp5, k5, 3, barrier, dist, dev) / k5
                del gp5
            sr5.end_clip()
            ms5 = res5[True]
            extra_cfg['configs[4] torso+head, 96 samples/ray'] = {
                'value': world * B / (ms5 / 1e3), 'unit': 'frames/s', 'ms_per_step': ms5, 'ms_per_step_uncached': res5[False],
                'conv_stack_TFLOPs_algorithmic': WARP_CONV_GFLOP_PER_FRAME * B / res5[False], 'frames_per_step_per_gpu': B,
                'note': 'render 48+48 (two-pass kernel) + SuperresolutionHybrid8XDC_Warp fuse mode v2 on the tcgen05 conv kernels; torso warper = '
                        'synthetic.StubTorsoModel (the real warper is the caller\'s PyTorch child, out of scope); cached = begin_clip() hoists '
                        'bg_encoder(ref_bg) and the 512->256 resizes (sr_with_ref.py:77-90); TFLOP/s counts the reference\'s 782 GFLOP/frame conv stack over the UNCACHED step'}
            del head5

    # ---- the fp32-grade tensor-core SR (sr_mode='tc_exact': split fp16 operands, three MMAs per product) on the same step, beside the fp16 headline
    if not args.no_extra_configs and sr_mode == 'tc':
        ex = engine.FrameEngine(batch=B, sr_mode='tc_exact', device=dev, world=world, rank=rank, dist=dist, use_graph=not args.no_graph,
                                hp={'num_samples_fine': 0}, exchange='none')
        ex.load_params(syn.make_decoder_params(seed=4), syn.make_sr_params(seed=5))
        ex.prepare(resident[:min(nb, 4)])
        kx = max(6, args.steps // 2)
        ms_x = timed_loop(lambda i: ex.step(*resident[i % min(nb, 4)]), kx, 3, barrier, dist, dev) / kx
        extra_cfg["sr_mode='tc_exact' (fp32-grade SR on tcgen05)"] = {
            'value': world * B / (ms_x / 1e3), 'unit': 'frames/s', 'ms_per_step': ms_x,
            'note': 'same step as the headline with split fp16 operands in every SR convolution (x_hi*w_hi + x_lo*w_hi + x_hi*w_lo, fp32 accumulation): '
                    'image within 1e-3*range of the fp32 reference (tests/test_gpu_parity.py::test_sr_full_tc_exact_vs_reference) instead of 2.3e-3 absolute'}
        del ex

    # ---- north_star's HBM roofline: the stand-alone sample_from_planes op on one step's render samples (L2 flushed between iterations)
    hbm = None
    if rank == 0:
        pcl = ren.PlanesCL(planes_cl_all[:B])
        ro, rd = r3.RaySampler()(cams[:B, :16].reshape(-1, 4, 4), cams[:B, 16:25].reshape(-1, 3, 3), 64)
        depth_mid = 2.15 + 1.1 * (torch.arange(48, device=dev).view(1, 1, 48, 1) + u_c[:B]) / 47.0            # samples spread through the box
        coords = (ro.unsqueeze(-2) + depth_mid * rd.unsqueeze(-2)).reshape(B, -1, 3).contiguous()
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
        ts = []
        for it in range(13):
            flush.zero_()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(); ren.sample_from_planes(None, pcl, coords, box_warp=1.0); a1.record()
            torch.cuda.synchronize()
            if it >= 3:
                ts.append(a0.elapsed_time(a1))
        ts.sort()
        t_ms = ts[len(ts) // 2]
        hbm = {'kernel': 'triplane_sample_kernel (sample_from_planes contract, mean NOT fused)', 'ms': t_ms, 'algorithmic_bytes': SAMPLE_BYTES_PER_FRAME * B,
               'achieved': SAMPLE_BYTES_PER_FRAME * B / (t_ms * 1e-3) / 1e9, 'unit': 'GB/s'}
        del flush
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    pk = peaks()
    hbm.update({'peak': pk['hbm_gbs'], 'frac': hbm['achieved'] / pk['hbm_gbs'], 'peak_source': pk['src'] + ' copy bandwidth', 'bound': 'hbm',
                'timing': '10 timed iterations, L2 flushed (256 MB write) before each, CUDA events, median'})
    # dominant kernel = the tensor-core conv (4 launches/step); its time is measured by CUDA-event pairs around every launch (library hook)
    if prof.get('conv_kernel_ms'):
        k_ms_per_step, k_launches = prof['conv_kernel_ms'] / args.steps, prof['conv_launches'] / args.steps
    else:
        k_ms_per_step, k_launches = prof['sr_conv_ms'] / args.steps, None
    sr_ms_per_step = prof['sr_conv_ms'] / args.steps
    sr_tflops = SR_GFLOP_PER_FRAME * B / k_ms_per_step                   # GFLOP / ms == TFLOP/s  (algorithmic: the reference's 197.63 GFLOP/frame)
    timed_window_s = ms / 1e3
    use_burst = timed_window_s < 1.0                                     # the kernel is timed inside a short step train at boost clocks: burst peak
    peak = pk['tf_burst'] if use_burst else pk['tf_sustained']
    traffic, traffic_note = ncu_traffic() if (sr_mode == 'tc' and B == 4) else (None, 'capture is for batch 4 on the tensor-core path')
    share = k_ms_per_step / (prof['total_ms'] / args.steps)
    stage = {k: v / args.steps for k, v in prof['stages'].items()}
    rextra = {'stage_ms_per_step': stage, 'hbm_sample_op': hbm, 'frac_of_sustained_peak': sr_tflops / pk['tf_sustained'],
              'sr_stage_ms_per_step': sr_ms_per_step, 'sr_stage_TFLOPs': SR_GFLOP_PER_FRAME * B / sr_ms_per_step,
              'whole_step_TFLOPs_per_gpu': SR_GFLOP_PER_FRAME * B / (ms / args.steps),
              'other_planes_layout': {'layout': 'nchw' if args.planes == 'cl' else 'cl', 'ms_per_step': ms_o / args.steps,
                                      'value': world * B * args.steps / (ms_o / 1e3)},
              'configs': extra_cfg}
    if sustained:
        sustained['conv_TFLOPs_estimate'] = SR_GFLOP_PER_FRAME * B / (sustained['ms_per_step'] * share)
        sustained['frac_of_sustained_peak'] = sustained['conv_TFLOPs_estimate'] / pk['tf_sustained']
        sustained['note'] = 'same step loop back to back; conv time estimated as this run\'s ms/step x the conv share measured in the profiled pass'
        rextra['sustained'] = sustained
    line = {
        'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32 render (decoder GEMMs: split-fp16 operands on tcgen05, f32 accumulate, f32-grade results); SR ' + {'tc': 'f16 operands / f32 accumulate (tcgen05)', 'tc_exact': 'split-f16 operands (3 products) / f32 accumulate (tcgen05), f32-grade results'}.get(sr_mode, 'f32'),
        'data': 'synthetic',
        # `config` = the workload (the same keys and values in the reference arm) + the L2 policy / timing statements the timing rules ask for;
        # how this arm runs the workload is under `setup`
        'config': {'workload': workload_text(args, world), 'frames_per_step_per_gpu': B, 'samples_per_ray': 48, 'render_res': 64, 'out_res': 512,
                   'l2_policy': f'inputs larger than L2: {P} distinct resident frames/GPU ({P * 25.2:.0f} MB) cycled',
                   'timing': 'CUDA events on the launch stream, barrier+sync both sides, max over ranks'},
        'setup': {'parallelism': f'frames sharded over {world} GPU(s); no data-path collective, one frame exchange per step',
                   'planes_layout': ("channels-last [N,3,256,256,32] resident in HBM, as the producer's channels_last conv emits them (sampled in place, no repack)"
                                     if args.planes == 'cl' else 'reference [N,3,32,256,256], repacked to channels-last inside every step'),
                   'exchange': (exchange_note + {'none': 'single GPU: none', 'p2p': 'copy-engine peer pushes of each step\'s frames into the clip on rank 0 (CUDA IPC), overlapped with the next step',
                                                  'allgather': 'NCCL all_gather_into_tensor of each step\'s frames on a side stream, overlapped with the next step'}[exchange]),
                   'frames': 'uint8 HWC video frames (real3d_infer.py:519 conversion fused into the last SR epilogue)' if u8 else 'fp32 NCHW in [-1,1] (clamp fused into the last SR epilogue)',
                   'sr_mode': sr_mode, 'cuda_graph': not args.no_graph},
        'clocks': clocks, 'gpu_launches': int(launches),
        'e2e': {'value': e2e_fps, 'unit': 'frames/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'steps': ksteps,
                'host_wall_ms': e2e_wall_ms, 'h2d_GBps': h2d * ksteps / (ms_e * 1e6), 'pinned_buffers': numa,
                'note': 'step_host(): pinned host in/out (reference NCHW plane layout), copies of step i+1 overlap compute of step i; the H2D of the fp32 planes (PCIe) bounds it'},
        'roofline': {'bound': 'tensor', 'achieved': sr_tflops, 'peak': peak, 'unit': 'TFLOP/s', 'frac': sr_tflops / peak,
                     'traffic': traffic, 'traffic_note': traffic_note,
                     'kernel': prof['sr_kernel'], 'launches_per_step': k_launches, 'kernel_ms_per_step': k_ms_per_step,
                     'peak_source': pk['src'] + (' bf16 burst (kernel timed per launch inside a %.0f ms step train)' % (ms) if use_burst else ' bf16 sustained'),
                     'algorithmic': f'{SR_GFLOP_PER_FRAME} GFLOP/frame x {B} frames/step', 'share_of_step': share, 'extra': rextra},
    }
    if not args.no_cpu_baseline:
        cpu_fps, ts, nthr, kind = time_cpu(1, 5, 1)
        torch.set_num_threads(1)                                   # SURVEY.md §8d: also report the 1-thread figure (one frame, no warm-up repeat)
        fn1, _ = cpu_frame_fn(1)
        t1 = time.perf_counter(); fn1(); one_thread_fps = 1.0 / (time.perf_counter() - t1)
        torch.set_num_threads(nthr)
        line['cpu_baseline'] = {'value': cpu_fps, 'unit': 'frames/s', 'cores': nthr, 'kind': kind, 'one_thread_value': one_thread_fps,
                                'sample': f'{len(ts)} x 1 frame of the same workload through '
                                          + ("the reference's unmodified modules (oracle/_ref)" if kind == 'reference' else 'the oracle port')
                                          + f', {nthr} torch threads of {host_threads()} usable, median'}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
