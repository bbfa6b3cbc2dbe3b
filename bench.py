#!/usr/bin/env python
"""Benchmark of the HMMR video->SMPL hot path (BASELINE.json metric: frames/sec through
ResNet-v2-50 -> f_movie -> IEF -> SMPL LBS -> projection).

  python bench.py --gpus N --steps K --warmup W            our CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference ...                     the reference path restated on the host CPU cores
                                                           (TF 1.8 cannot be installed here: oracle port)

Prints ONE JSON line (rank 0).  Workloads: hmmr (BASELINE config 3: 32 clips x T=20, the default; weak-scaled
to 32 clips per GPU = config 4 at 8 GPUs), single_frame (config 2: batch 64), smpl (config 5: 65536 poses).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# algorithmic work per unit (SURVEY.md 8d / DESIGN.md): dense FLOPs as the reference computes them
FLOP_RESNET_FRAME = 6.960e9
FLOP_FMOVIE_FRAME = 0.146e9
FLOP_IEF_FRAME_3HEADS = 59.4e6
FLOP_SMPL_POSE = 16.5e6
BYTES_SMPL_POSE = 84384


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {'hbm_gbs': d['hbm_gbs'], 'bf16_tflops': d['bf16_tflops'], 'bf16_tflops_sustained': d['bf16_tflops_sustained'],
                'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                          '-lms', '50'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, smax, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        time.sleep(0.15)
        inside = [ln for ts, ln in self.lines if (t0 is None or ts >= t0) and (t1 is None or ts <= t1 + 0.1)]
        for ln in (inside if len(inside) >= 2 else [ln for _, ln in self.lines]):
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax = float(f[1])
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': smax, 'samples': len(sm), 'reasons': sorted(reasons)}


# --------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port of the reference path on the host cores
# --------------------------------------------------------------------------------------------------------
PARITY_KEYS = ('omegas', 'verts', 'kps', 'joints', 'poses', 'omegas_delta', 'verts_delta', 'kps_delta')
PARITY_TOL = 1e-4          # BASELINE.json north_star: outputs within 1e-4 rel FP32 of the reference graph


def cpu_reference_run(workload, steps, warmup, clips_per_step=1, T=20, images=None, keep=None):
    """Times the oracle port on the host cores.  `images` (optional, hmmr / single_frame): run on exactly these frames
    instead of a fresh synthetic sample; `keep` (a dict) then receives the oracle's outputs of the last step, which is how
    bench.py parity-checks the run it has just timed (the checker, never the thing measured as ours)."""
    import torch
    from human_dynamics_b200 import synthetic
    from oracle import nets_ref
    # measured on this pool's 128-core host (tools/cpu_threads.py): the torch-CPU port peaks at 16-32 threads (51 frames/s
    # for the ResNet part) and collapses beyond 64 (<1 frame/s at 128), so the reference arm uses min(cores, 32) threads.
    cores = min(os.cpu_count() or 1, int(os.environ.get('HD_CPU_THREADS', '32')))
    torch.set_num_threads(cores)
    w = synthetic.make_synthetic_weights(seed=1)
    smpl = synthetic.make_synthetic_smpl(seed=2)
    times = []
    if workload == 'smpl':
        from oracle.smpl_ref import SMPLRef, batch_orth_proj_idrot
        n = 256
        beta, theta = synthetic.make_smpl_inputs(n, seed=0)
        cam = np.ones((n, 3), np.float32)
        ref = SMPLRef(smpl)
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            v, j, _ = ref(beta, theta, get_skin=True)
            batch_orth_proj_idrot(j, cam)
            if it >= warmup:
                times.append(time.perf_counter() - t0)
        units, sample = n, '%d poses per step (numpy float32 port of batch_smpl.py)' % n
    elif workload == 'single_frame':
        img = synthetic.make_images(8, seed=0) if images is None else images
        n = img.shape[0]
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            r = nets_ref.single_frame_predict(img, w, smpl)
            if it >= warmup:
                times.append(time.perf_counter() - t0)
        if keep is not None:
            keep.update(r)
        units, sample = n, '%d frames per step (torch-CPU float32 port, reference op order)' % n
    else:
        img = synthetic.make_images(clips_per_step * T, seed=0).reshape(clips_per_step, T, 224, 224, 3) if images is None else images
        clips_per_step = img.shape[0]
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            r = nets_ref.hmmr_predict(img, w, smpl)
            if it >= warmup:
                times.append(time.perf_counter() - t0)
        if keep is not None:
            keep.update(r)
        units = clips_per_step * T
        sample = '%d clip(s) x T=%d frames per step (torch-CPU float32 port of the TF1 graph, reference op order)' % (clips_per_step, T)
    sec = float(np.mean(times))
    return units / sec, sec, cores, sample


def _cpu_worker(workload, steps, warmup, threads, idx, start_evt, q):
    """One process of the multi-process reference arm: `threads` torch threads on its own clip."""
    os.environ['HD_CPU_THREADS'] = str(threads)
    import torch
    torch.set_num_threads(threads)
    from human_dynamics_b200 import synthetic
    from oracle import nets_ref
    w = synthetic.make_synthetic_weights(seed=1)
    smpl = synthetic.make_synthetic_smpl(seed=2)
    if workload == 'single_frame':
        img = synthetic.make_images(8, seed=50 + idx)
        fn, units = (lambda: nets_ref.single_frame_predict(img, w, smpl)), 8
    else:
        img = synthetic.make_images(20, seed=50 + idx).reshape(1, 20, 224, 224, 3)
        fn, units = (lambda: nets_ref.hmmr_predict(img, w, smpl)), 20
    for _ in range(warmup):
        fn()
    q.put(('ready', idx))
    start_evt.wait()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    q.put(('done', idx, units * steps, time.perf_counter() - t0))


def cpu_reference_run_multi(workload, steps, warmup):
    """The reference arm with all the host threads it can use: the torch-CPU port stops scaling beyond ~32 threads per process
    (tools/cpu_threads.py), so the box's cores are split into processes of 32 threads, each running the path on its own clip;
    throughput = all frames / the slowest process's time (all processes start together)."""
    import multiprocessing as mp
    total = os.cpu_count() or 1
    threads = min(total, int(os.environ.get('HD_CPU_THREADS', '32')))
    procs = max(1, min(int(os.environ.get('HD_CPU_PROCS', str(total // threads))), 8))
    if workload == 'smpl' or procs == 1:
        return cpu_reference_run(workload, steps, warmup) + (1,)
    ctx = mp.get_context('spawn')
    q, evt = ctx.Queue(), ctx.Event()
    ps = [ctx.Process(target=_cpu_worker, args=(workload, steps, warmup, threads, i, evt, q)) for i in range(procs)]
    for pr in ps:
        pr.start()
    ready = 0
    while ready < procs:
        if q.get(timeout=600)[0] == 'ready':
            ready += 1
    evt.set()
    res = [q.get(timeout=900) for _ in range(procs)]
    for pr in ps:
        pr.join(timeout=60)
    units = sum(r[2] for r in res)
    sec = max(r[3] for r in res)
    per = 20 if workload != 'single_frame' else 8
    sample = ('%d processes x %d threads, each %s per step on its own input (torch-CPU float32 port of the TF1 graph, reference op order)'
              % (procs, threads, '1 clip x T=20 frames' if workload != 'single_frame' else '8 frames'))
    return units / sec, sec / steps, procs * threads, sample, procs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='hmmr', choices=['hmmr', 'single_frame', 'smpl'])
    ap.add_argument('--clips', type=int, default=32, help='clips per GPU (hmmr) / frames per GPU x 1 (single_frame: 64)')
    ap.add_argument('--mode', default=os.environ.get('HD_IMPL', 'auto'), choices=['auto', 'tc3h', 'tc3', 'simt', 'tc1'],
                    help='auto/tc3h = tcgen05 fp16 head+remainder split x3 (FP32-class parity mode, the headline); tc3 = 3xTF32 (also FP32-class); '
                         'tc1 = single-pass TF32 (fails parity); simt = exact FP32 CUDA cores')
    ap.add_argument('--frame-chunk', type=int, default=int(os.environ.get('HD_FRAME_CHUNK', '160')))
    ap.add_argument('--late-chunk', type=int, default=int(os.environ.get('HD_LATE_CHUNK', '640')))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the C2 / C5 sub-results of the default line')
    ap.add_argument('--graph', type=int, default=int(os.environ.get('HD_GRAPH', '1')),
                    help='1 = replay the device-resident step from a CUDA graph (one graph launch per step), 0 = eager launches')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB in '
                         'all: larger arrays are cut to a fixed seeded sample along their longest axis); inputs are seeded, so runs '
                         'with the same arguments can be compared output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.warmup < 3 and args.impl == 'ours':
        args.warmup = 3

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    unit_name = 'poses/sec' if args.workload == 'smpl' else 'frames/sec'
    metric = 'frames/sec (ResNet->f_movie->SMPL LBS)' if args.workload == 'hmmr' else (
        'frames/sec (ResNet->IEF->SMPL, single frame)' if args.workload == 'single_frame' else 'poses/sec (SMPL LBS)')

    if args.impl == 'reference':
        if rank != 0:
            return 0
        # the port stops scaling past ~32 threads, and several 32-thread processes fight over memory bandwidth (measured on this
        # pool's 128-core hosts: 4 x 32 threads = 17.6 frames/s in total vs 23.4 for one process): time both, report the better
        v1, sec1, cores1, sample1 = cpu_reference_run(args.workload, args.steps, args.warmup)
        vm, secm, coresm, samplem, procs = cpu_reference_run_multi(args.workload, args.steps, args.warmup)
        if procs > 1 and vm > v1:
            v, sec, cores, sample = vm, secm, coresm, samplem + ' [one 32-thread process: %.1f %s]' % (v1, unit_name)
        else:
            v, sec, cores, sample = v1, sec1, cores1, sample1 + (' [%d processes x 32 threads together: %.1f %s]' % (procs, vm, unit_name) if procs > 1 else '')
        line = {'impl': 'reference', 'metric': metric, 'value': v, 'unit': unit_name, 'n_gpus': args.gpus, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f32', 'data': 'synthetic',
                'config': {'workload': workload_name(args), 'note': 'TF 1.8 cannot be installed here; restated reference on host CPU'},
                'cpu_baseline': {'value': v, 'unit': unit_name, 'cores': cores, 'kind': 'port', 'sample': sample},
                'e2e': {'value': v, 'unit': unit_name, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'gpu_launches': 0}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from human_dynamics_b200 import synthetic, HMMRConfig, _lib
    from human_dynamics_b200.engine import HMMREngine
    from human_dynamics_b200.dist import OutputGatherer

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    dev = torch.device('cuda', local_rank)
    peaks = load_peaks()
    w = synthetic.make_synthetic_weights(seed=1)
    smpl = synthetic.make_synthetic_smpl(seed=2)
    T = 20

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.workload == 'smpl':
        from human_dynamics_b200.smpl import SMPLConstants
        N = 65536
        consts = SMPLConstants(smpl, device=dev)
        beta, theta = synthetic.make_smpl_inputs(N, seed=rank)
        b_d, t_d = torch.from_numpy(beta).to(dev), torch.from_numpy(theta).to(dev)
        cam = torch.ones((N, 3), device=dev)
        outs = consts.forward(b_d, t_d, cam=cam)

        def step():
            consts.forward(b_d, t_d, cam=cam, out=outs)
        units_per_step, B = N, None
        gather_keys = ()
    else:
        single = args.workload == 'single_frame'
        B = 64 if single and args.clips == 32 else args.clips
        Tw = 1 if single else T
        cfg = HMMRConfig(batch_size=B, sequence_length=Tw, frame_chunk=args.frame_chunk, late_chunk=args.late_chunk)
        eng = HMMREngine(w, smpl, cfg, device=dev, impl=args.mode)
        img_host = torch.from_numpy(synthetic.make_images(B * Tw, seed=100 + rank)).view(B, Tw, 224, 224, 3).pin_memory()
        img_dev = img_host.to(dev)
        units_per_step = B * Tw
        gather_keys = ('omegas', 'verts', 'kps')          # per-clip outputs named by BASELINE config 4 / SURVEY 8e
        last = {}

        gatherer = OutputGatherer(B * world, dst=0) if world > 1 else None

        def step():
            if world > 1:
                # eager launches so that the dt=0 outputs start travelling to rank 0 (side stream, point-to-point over NVLink)
                # while the delta heads still compute; the delta-independent keys need nothing else
                def main_ready(o):
                    gatherer.start({k: o[k] for k in gather_keys if k in o})
                if args.graph and not single:       # two graph launches per step, the gather starts between them
                    out, last['nodes'] = eng.predict_graphed_split(img_dev, main_ready)
                else:
                    out = eng.predict(img_dev, single_frame=single, on_main_ready=main_ready)
                rest = {k: out[k] for k in gather_keys if k.endswith('_delta')}
                if rest:
                    gatherer.start(rest)
                last['g'] = gatherer.wait()
            elif args.graph:
                out, last['nodes'] = eng.predict_graphed(img_dev, single_frame=single)
            else:
                out = eng.predict(img_dev, single_frame=single)
            last['out'] = out

        # end to end through the reference-named API: src.evaluation.tester.Tester.predict on a PLAIN numpy array (pageable memory,
        # page-locked in place on first sight), numpy results back.  The single-frame workload has no Tester wiring in the
        # reference (SURVEY 3.3): it goes through HMMREngine.predict_host with the same copies.
        from src.evaluation.tester import Tester
        tester = Tester(cfg, engine=eng)
        img_np = np.array(img_host.numpy(), copy=True)
        FR = 256                                          # synthetic uint8 "video frames" for the process_image leg
        rng = np.random.RandomState(7 + rank)
        frames_u8 = rng.randint(0, 256, size=(B, Tw, FR, FR, 3), dtype=np.uint8)
        boxes = np.stack([rng.uniform(100, 156, B * Tw), rng.uniform(100, 156, B * Tw), rng.uniform(0.9, 1.2, B * Tw)], axis=1).reshape(B, Tw, 3)

        def step_e2e():
            if world > 1:      # N GPUs: the end-to-end step includes the gather of the per-clip outputs onto rank 0 (device tensors there)
                def main_ready(o):
                    gatherer.start({k: o[k] for k in gather_keys if k in o})
                host, h2d, d2h = eng.predict_host(img_host, single_frame=single, on_main_ready=main_ready)
                last['g'] = gatherer.wait()
                torch.cuda.current_stream().synchronize()
                return h2d, d2h
            if single:
                host, h2d, d2h = eng.predict_host(img_host, single_frame=True)
                torch.cuda.current_stream().synchronize()
                return h2d, d2h
            res = tester.predict(img_np)
            return img_np.nbytes, sum(v.nbytes for v in res.values())

        def step_e2e_u8():
            res = tester.predict_frames(frames_u8, boxes)
            return frames_u8.nbytes + B * Tw * 16, sum(v.nbytes for v in res.values())

    # ------------------------------------------------------------------ device-resident timing (value)
    sampler = ClockSampler(local_rank)
    sampler.start()                    # started before warm-up so nvidia-smi is already looping when the timed region begins
    for _ in range(args.warmup):
        step()
    barrier()
    _lib.lib.hd_launch_count_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = sampler.mark()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    t_end = sampler.mark()
    launches = int(_lib.lib.hd_launch_count())
    # results of the LAST TIMED step for the clips / frames the oracle will check (the later end-to-end legs reuse the output buffers)
    timed_out = None
    if args.workload != 'smpl':
        sel_idx = [0, B - 1]
        timed_out = {k: last['out'][k][sel_idx].float().cpu().numpy() for k in PARITY_KEYS if k in last['out']}
    dumped = None
    if args.dump_outputs and rank == 0:
        # what a caller of the timed path receives: the fetch keys (not the '_'-prefixed inspection buffers) / the SMPL outputs
        res = outs if args.workload == 'smpl' else last['out']
        dumped = dump_outputs({k: v for k, v in res.items() if not k.startswith('_') and v is not None}, args.dump_outputs)
    gather_ok = None
    if world > 1 and rank == 0 and last.get('g') is not None:
        # gathered tensors must contain rank 0's own clips bit for bit (the N-GPU == 1-GPU identity is tests/test_multi_gpu.py);
        # checked here, before the end-to-end legs reuse the output buffers
        torch.cuda.synchronize()
        gather_ok = bool(all(torch.equal(last['g'][k][:B], last['out'][k]) for k in gather_keys))
    graph_nodes = None
    if args.workload != 'smpl' and args.graph and last.get('nodes'):
        graph_nodes = int(last['nodes'])
        launches = graph_nodes * args.steps          # kernels executed inside the timed region (submitted as `steps` graph launches)
    clocks = sampler.stop(t_begin, t_end)
    ms = e0.elapsed_time(e1) / args.steps
    if world > 1:
        tms = torch.tensor([ms], device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    value = units_per_step * world / (ms * 1e-3)

    # ------------------------------------------------------------------ end-to-end through the public API (host buffers)
    e2e = None
    if args.workload != 'smpl':
        for _ in range(2):
            step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            h2d, d2h = step_e2e()
        torch.cuda.synchronize()
        sec = (time.perf_counter() - t0) / args.steps
        if world > 1:
            ts = torch.tensor([sec], device=dev)
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
            sec = float(ts.item())
        e2e = {'value': units_per_step * world / sec, 'unit': unit_name, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
               'ms_per_step': sec * 1e3,
               'api': ('HMMREngine.predict_host(pinned float32 frames), single_frame=True' if single else
                       'src.evaluation.tester.Tester.predict(np.ndarray float32 (B,T,224,224,3)) -> dict of 14 numpy arrays; the '
                       "caller's pageable array is page-locked in place once (cudaHostRegister), H2D in 32-frame pieces overlapped with "
                       'the ResNet, results are views of a 2-deep ring of pinned buffers (copy=False)')}
        if not single:
            for _ in range(2):
                step_e2e_u8()
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                h2d8, d2h8 = step_e2e_u8()
            torch.cuda.synchronize()
            sec8 = (time.perf_counter() - t0) / args.steps
            if world > 1:
                ts = torch.tensor([sec8], device=dev)
                dist.all_reduce(ts, op=dist.ReduceOp.MAX)
                sec8 = float(ts.item())
            # streaming: the same copies, but window i+1 is uploaded / computed while window i's results travel to the host
            stream_n = args.steps + 2
            for _ in tester.predict_stream([img_np] * 2):
                pass
            barrier()
            t0 = time.perf_counter()
            got = 0
            for res in tester.predict_stream([img_np] * stream_n):
                got += 1
            torch.cuda.synchronize()
            secs = (time.perf_counter() - t0) / stream_n
            if world > 1:
                ts = torch.tensor([secs], device=dev)
                dist.all_reduce(ts, op=dist.ReduceOp.MAX)
                secs = float(ts.item())
            e2e['streaming'] = {'value': units_per_step * world / secs, 'unit': unit_name, 'ms_per_step': secs * 1e3, 'windows': stream_n,
                                'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                                'api': 'Tester.predict_stream(iterable of numpy windows): same H2D / D2H per window, the device->host copies of '
                                       'window i overlap window i+1 (2 device input buffers, 2 result slots)'}
            e2e['uint8_frames'] = {'value': units_per_step * world / sec8, 'unit': unit_name, 'h2d_bytes_per_step': int(h2d8),
                                   'd2h_bytes_per_step': int(d2h8), 'ms_per_step': sec8 * 1e3,
                                   'api': 'Tester.predict_frames(uint8 (B,T,%d,%d,3) video frames + bbox [cx,cy,scale]): process_image '
                                          '(run_video.py:56-107) on the GPU feeding conv1 directly, then the same path' % (FR, FR)}

    # ------------------------------------------------------------------ roofline of the dominant kernel (instrumented extra pass)
    roofline = None
    if rank == 0:
        roofline = measure_roofline(args, peaks, locals())

    # ------------------------------------------------------------------ cpu_baseline + parity of the run just timed
    # The oracle port runs on the FIRST and LAST clip (frame) of this very benchmark input; its outputs double as the
    # checker of the last timed step's results (clips / frames are independent, so a 2-clip oracle run checks them exactly).
    cpu_baseline, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if args.workload == 'smpl':
            v, sec, cores, sample = cpu_reference_run(args.workload, 2, 1)
        else:
            sel = [0, B - 1]
            sub = img_host[sel].numpy() if not single else img_host[sel].numpy().reshape(2, 224, 224, 3)
            ref = {}
            v, sec, cores, sample = cpu_reference_run(args.workload, 2, 1, images=sub, keep=ref)
            torch.cuda.synchronize()
            worst, per = 0.0, {}
            for k in PARITY_KEYS:
                if k not in ref or k not in timed_out:
                    continue
                g = timed_out[k].reshape(ref[k].shape).astype(np.float64)
                e = float(np.abs(g - ref[k]).max() / max(float(np.abs(ref[k]).max()), 1e-12))
                per[k] = e
                worst = max(worst, e)
            parity = {'parity_max_rel': worst, 'tolerance': PARITY_TOL, 'per_key': per,
                      'checked': 'last timed step, %s {0, %d} of %d vs the float32 oracle port' % ('frames' if single else 'clips', B - 1, B)}
            sample += ' = %s {0, %d} of the timed input' % ('frames' if single else 'clips', B - 1)
        cpu_baseline = {'value': v, 'unit': unit_name, 'cores': cores, 'kind': 'port', 'sample': sample}
    if gather_ok is not None:
        parity = {'gather_own_shard_bit_identical': gather_ok}

    # ------------------------------------------------------------------ the other single-GPU BASELINE configs, device-resident
    extra = None
    if rank == 0 and world == 1 and args.workload == 'hmmr' and not args.no_extra:
        extra = measure_extra_configs(args, peaks, w, smpl, dev)

    if rank == 0:
        line = {'metric': metric, 'value': value, 'unit': unit_name, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
                'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f32 (SMPL; blend GEMM on tcgen05 with the fp16 head/remainder split)' if args.workload == 'smpl' else {'auto': 'f32 (tcgen05 3x fp16 head/remainder split, fp32 two-level accumulate)', 'tc3h': 'f32 (tcgen05 3x fp16 head/remainder split, fp32 two-level accumulate)',
                          'tc3': 'f32 (tcgen05 3xTF32 split, fp32 two-level accumulate)', 'simt': 'f32', 'tc1': 'tf32'}[args.mode],
                'data': 'synthetic',
                'config': {'workload': workload_name(args), 'mode': args.mode, 'frame_chunk': args.frame_chunk, 'late_chunk': args.late_chunk,
                           'l2': 'inputs larger than L2 (%.0f MB of frames per step vs 126 MB)' % (units_per_step * 224 * 224 * 3 * 4 / 1e6)
                           if args.workload != 'smpl' else 'outputs larger than L2 (5.4 GB of vertices per step)',
                           'parallelism': 'dp%d (clips sharded, gather of %s to rank 0)' % (world, '/'.join(gather_keys)) if world > 1 else 'single GPU',
                           'peaks': peaks['source']},
                'clocks': clocks, 'gpu_launches': launches,
                'gpu_launches_per_step': launches / max(1, args.steps)}
        if graph_nodes:
            line['cuda_graph'] = {'graph_launches_per_step': 1 if world == 1 else 2, 'kernel_nodes_per_step': graph_nodes}
        if e2e:
            line['e2e'] = e2e
        if roofline:
            line['roofline'] = roofline
        if cpu_baseline:
            line['cpu_baseline'] = cpu_baseline
        if extra:
            line['extra'] = extra
        if dumped is not None:
            line['dumped_outputs'] = {'dir': args.dump_outputs, 'shapes': dumped}
        if parity:
            line['parity'] = parity
            if 'parity_max_rel' in parity:
                line['parity_max_rel'] = parity['parity_max_rel']
        print(json.dumps(line))
        if parity and parity.get('parity_max_rel', 0.0) > PARITY_TOL:
            sys.stderr.write('bench.py: PARITY FAILURE %r\n' % (parity,))
            return 3
        if parity and parity.get('gather_own_shard_bit_identical') is False:
            sys.stderr.write('bench.py: gathered outputs differ from the local shard\n')
            return 3
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_BYTES = 60 << 20       # --dump-outputs: array data in all; with the .npy headers the files stay under 64 MB (64e6 bytes)


def dump_outputs(outs, path, budget=DUMP_BYTES):
    """Writes each output tensor as path/<name>.npy in float32.  Smaller arrays are written whole; the budget left over is shared
    among the larger ones, each cut down, while over its share, along its longest axis to a sorted sample of indices drawn with a
    fixed seed.  The sample depends only on the shapes, so two builds run with the same arguments write comparable files."""
    import torch
    os.makedirs(path, exist_ok=True)
    items = sorted(outs.items(), key=lambda kv: (kv[1].numel(), kv[0]))
    left, written = budget, {}
    for i, (name, t) in enumerate(items):
        share = left // (len(items) - i)
        t = t.detach()
        rng = np.random.RandomState(0)
        while t.numel() * 4 > share:
            ax = max(range(t.dim()), key=lambda d: t.shape[d])
            keep = max(1, t.shape[ax] * share // (t.numel() * 4))
            idx = np.sort(rng.choice(t.shape[ax], keep, replace=False))
            t = t.index_select(ax, torch.from_numpy(idx).to(t.device))
        a = t.float().cpu().numpy()
        np.save(os.path.join(path, name + '.npy'), a)
        left -= a.nbytes
        written[name] = list(a.shape)
    return written


def workload_name(args):
    if args.workload == 'hmmr':
        return 'BASELINE configs[2] (configs[3] per GPU at N=8): full HMMR, T=20 window, %d clips per GPU, 224x224x3' % args.clips
    if args.workload == 'single_frame':
        return 'BASELINE configs[1]: single-frame ResNet-50 + 3-iter IEF + SMPL, batch 64'
    return 'BASELINE configs[4]: SMPL LBS microbench, 65536 poses -> 6890 verts'


def measure_extra_configs(args, peaks, w, smpl, dev):
    """BASELINE configs[1] (single-frame, batch 64) and configs[4] (SMPL LBS microbench, 65536 poses) timed device-resident with
    CUDA events so that the default bench line carries them too (same code as --workload single_frame / smpl)."""
    import torch
    from human_dynamics_b200 import synthetic, HMMRConfig
    from human_dynamics_b200.engine import HMMREngine
    from human_dynamics_b200.smpl import SMPLConstants
    out = {}

    def timed(fn, steps, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps
    # C2
    n = 64
    eng = HMMREngine(w, smpl, HMMRConfig(batch_size=n, sequence_length=1), device=dev, impl=args.mode)
    img = torch.from_numpy(synthetic.make_images(n, seed=300)).to(dev).view(n, 1, 224, 224, 3)
    ms = timed(lambda: eng.predict_graphed(img, single_frame=True) if args.graph else eng.predict(img, single_frame=True), 10)
    fl = n * (FLOP_RESNET_FRAME + FLOP_IEF_FRAME_3HEADS / 3 + FLOP_SMPL_POSE)
    out['C2_single_frame_batch64'] = {'value': n / (ms * 1e-3), 'unit': 'frames/sec', 'ms_per_step': ms,
                                      'roofline': {'bound': 'tensor', 'achieved': fl / (ms * 1e-3) / 1e12, 'peak': peaks['bf16_tflops_sustained'],
                                                   'unit': 'TFLOP/s', 'frac': fl / (ms * 1e-3) / 1e12 / peaks['bf16_tflops_sustained']},
                                      'note': 'one 64-frame pass: 49..392 tiles per late layer on 148 SMs (wave quantisation), L2-resident inputs'}
    del eng
    # C5
    N = 65536
    consts = SMPLConstants(smpl, device=dev)
    beta, theta = synthetic.make_smpl_inputs(N, seed=0)
    b_d, t_d = torch.from_numpy(beta).to(dev), torch.from_numpy(theta).to(dev)
    cam = torch.ones((N, 3), device=dev)
    outs = consts.forward(b_d, t_d, cam=cam)
    ms = timed(lambda: consts.forward(b_d, t_d, cam=cam, out=outs), 5)
    ach = N * BYTES_SMPL_POSE / (ms * 1e-3) / 1e9
    out['C5_smpl_lbs_65536'] = {'value': N / (ms * 1e-3), 'unit': 'poses/sec', 'ms_per_step': ms,
                                'roofline': {'bound': 'hbm', 'achieved': ach, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': ach / peaks['hbm_gbs'],
                                             'algorithmic_bytes_per_step': N * BYTES_SMPL_POSE},
                                'note': 'pose + blend GEMM (tcgen05, 3 MMAs per product in the parity mode: %.1f TFLOP-equivalents, the '
                                        'tensor pipe bounds this config before HBM does) + tensor-core skinning + keypoints' % (N * 256 * 20672 * 2 * 3 / 1e12)}
    del outs, consts
    torch.cuda.empty_cache()
    return out


def measure_roofline(args, peaks, env):
    """Instrumented extra pass (NOT part of `value`): CUDA events around every launch of the dominant kernel."""
    import torch
    if args.workload == 'smpl':
        # one fused blend+skin kernel dominates: HBM-bound target
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        step = env['step']
        torch.cuda.synchronize()
        e0.record(); step(); e1.record(); torch.cuda.synchronize()
        t = e0.elapsed_time(e1) * 1e-3
        ach = 65536 * BYTES_SMPL_POSE / t / 1e9
        return {'bound': 'hbm', 'kernel': 'smpl_pose + smpl_skin + smpl_joints (whole hd_smpl_forward)', 'achieved': ach,
                'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': ach / peaks['hbm_gbs'], 'traffic': None,
                'algorithmic_bytes_per_launch': 65536 * BYTES_SMPL_POSE}
    eng, img_dev = env['eng'], env['img_dev']
    from human_dynamics_b200 import _lib
    import ctypes
    N = img_dev.shape[0] * img_dev.shape[1]
    cA = max(1, min(int(eng.config.frame_chunk), N))
    cB = max(1, min(int(eng.config.late_chunk), N))
    stp = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    tc_time, tc_flops, n_tc, conv_time = 0.0, 0.0, 0, 0.0
    # one chunk pass of each trunk stage with an event pair around every conv launch (plans are bound by the timed steps)
    for stage, c in (('A', cA), ('B', cB)):
        plan = eng._resnet_plan(c, 224, stage)
        reps = N // c
        evs = []
        torch.cuda.synchronize()
        for op in ([plan.conv1_op] if getattr(plan, 'conv1_op', None) is not None else []) + list(plan.ops):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); op.run(stp); b.record()
            evs.append((a, b, op))
        torch.cuda.synchronize()
        for a, b, op in evs:
            d = op.d
            if d is None:                 # not a conv (strided-shortcut subsample)
                continue
            kdim = 147 if (d.flags & 2) else d.KH * d.KW * d.Cin          # conv1 over padded planes: the 7x7x3 taps, not the padded K = 256
            fl = 2.0 * d.n_img * d.Ho * d.Wo * d.Cout * kdim
            t = a.elapsed_time(b) * 1e-3
            conv_time += t * reps
            if d.impl != _lib.HD_IMPL_SIMT or args.mode == 'simt':
                tc_time += t * reps; tc_flops += fl * reps; n_tc += reps
    kind = 'conv_gemm_tc_kernel (tcgen05 implicit GEMM, %s, persistent)' % args.mode if args.mode != 'simt' else 'conv_gemm_simt_kernel'
    ach = tc_flops / tc_time / 1e12
    peak = peaks['bf16_tflops_sustained']
    step_s = env['ms'] * 1e-3
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
    if os.path.exists(tpath) and args.mode in ('auto', 'tc3h'):
        with open(tpath) as f:
            tj = json.load(f)
        tb, mb = tj['tensor_bound_launch'], tj['memory_bound_launch']
        traffic = {'dram_bytes_per_launch': tb['dram_bytes'], 'algorithmic_bytes_per_launch': tb['algorithmic_bytes'], 'launch': tb['layer'],
                   'memory_bound_launch': {'dram_bytes_per_launch': mb['dram_bytes'], 'algorithmic_bytes_per_launch': mb['algorithmic_bytes'],
                                           'launch': mb['layer']},
                   'source': 'profiles/r02_traffic.json: ncu --set full captures of this round\'s kernels (tools/make_traffic_json.py); '
                             'bench.py cannot run ncu on itself, so the file is regenerated whenever the kernel changes'}
    return {'bound': 'tensor', 'kernel': kind, 'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s', 'frac': ach / peak, 'traffic': traffic,
            'launches_per_step': n_tc, 'avg_launch_us': tc_time / n_tc * 1e6, 'algorithmic_flops_per_launch_avg': tc_flops / n_tc,
            'share_of_step': tc_time / step_s,
            'note': 'algorithmic FLOPs (2*M*N*K, dense, as the reference computes them) of the %d conv launches of one step / their '
                    'CUDA-event durations (instrumented extra pass: one chunk of each trunk stage, scaled by its repeat count); '
                    'peak = bf16/fp16 dense sustained (%s). The parity modes issue 3 MMAs per product: ceiling = peak/3 (%.0f TFLOP/s) for the '
                    'fp16 split, peak/6 for 3xTF32.' % (n_tc, peaks['source'], peak / 3)}


if __name__ == '__main__':
    sys.exit(main())
