#!/usr/bin/env python
"""bench.py -- images/sec of the detector / segmenter forward hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                      (CPU arm: the reference's algorithm on the host cores)
  python bench.py --config {yolov5s,fcos,deeplab,yolox}     (default yolov5s = the headline, BASELINE.json configs[1]; the others are
                                                             configs[4], configs[2] and the inference half of configs[3])

One JSON line on rank 0.  `value`: inputs resident in HBM (device time, CUDA events, max over ranks).  `e2e`: the
same metric through the public pipeline API with pinned HOST buffers (H2D of every step's frames and D2H of every
step's results inside the timed region).  `roofline`: the conv stack (the dominant kernel family), algorithmic
FLOPs / measured duration against the measured cuBLAS bf16 peak.  `cpu_baseline`: the oracle port on the host cores.
"""
import argparse
import glob
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = 'images/sec YOLOv5-s 640x640 bs64 forward (backbone+neck+detect+decode+NMS)'
ALG_GFLOP_PER_IMG = 16.43359375  # 1051.75 GFLOP / 64 (SURVEY.md §8 d-1: 2*M*N*K over the 60 convs)

# secondary configurations (BASELINE.json configs[4], [2], inference half of [3]); per-GPU batch, input size, model builder
SECONDARY = {
    'fcos': dict(metric='images/sec FCOS ResNet50 800x800 bs32 forward (backbone+FPN+centerness head+decode+top-k+NMS)', batch=32, hw=(800, 800),
                 workload='FCOS R50 800x800 forward+decode+NMS, bs32 per GPU (conf/coco_fcos.yml; BASELINE.json configs[4])',
                 collective='one all_gather_into_tensor of [B,1000*6+1] f32 (scores, classes, boxes, count) per step'),
    'deeplab': dict(metric='images/sec DeepLabv3+ ResNet50 1024x2048 bs16 forward (backbone+ASPP+decoder+upsample+argmax)', batch=16, hw=(1024, 2048),
                    workload='DeepLabv3+ R50v1c 1024x2048 forward+argmax, bs16 per GPU (cityscapes_deeplabv3plus_r50.yml; BASELINE.json configs[2])',
                    collective='one all_gather_into_tensor of the uint8 label maps [B,1024,2048] per step'),
    'yolox': dict(metric='images/sec YOLOX-s 640x640 bs64 forward (backbone+neck+head+decode+batched_nms; inference half of configs[3])', batch=64,
                  hw=(640, 640), workload='YOLOX-s 640x640 forward+decode+batched_nms, bs64 per GPU (inference half of BASELINE.json configs[3])',
                  collective='one all_gather_into_tensor of [B,A,7] rows + counts per step'),
}


def csrc_sha1():
    """Hash of the CUDA sources: stamps profile-derived numbers (roofline.traffic) with the kernel version they were captured on."""
    h = hashlib.sha1()
    for f in sorted(glob.glob(os.path.join(ROOT, 'cvpytorch_b200', 'csrc', '*'))):
        if f.endswith(('.cu', '.cuh', '.h')) and not os.path.basename(f).startswith('train_'):  # (the training kernels are not on the measured inference path)
            h.update(open(f, 'rb').read())
    return h.hexdigest()[:12]


def measured_conv_traffic(batch):
    """DRAM bytes of the conv launches of one step from the newest committed ncu launch list (tools/launch_summary.py).  Returned only
    when it was captured on the CURRENT kernel sources (source_sha1 stamp) -- a stale capture reads as null, never as a number."""
    best = None
    for f in sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r*', 'conv_traffic.json'))):
        try:
            tj = json.load(open(f))
        except Exception:
            continue
        if int(tj.get('batch', 0)) == batch:
            best = (f, tj)
    if best is None:
        return None, 'no capture'
    f, tj = best
    rel = os.path.relpath(f, ROOT)
    if tj.get('source_sha1') != csrc_sha1():
        return None, f'{rel} was captured on kernel sources {tj.get("source_sha1", "unstamped")}, current {csrc_sha1()}: stale, not reported'
    return int(tj['conv_dram_bytes_per_step']), f'{rel} (ncu dram read+write of the conv launches of one step, kernel sources {tj["source_sha1"]})'


def env_int(k, d):
    return int(os.environ.get(k, d))


DUMP_LIMIT = 60 << 20  # data budget of --dump-outputs: with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes the arrays a caller of the timed path received from its last step as <out_dir>/<name>.npy, floating point as
    float32 (float64 stays float64), integers as float64 (exact).  An array larger than its share of DUMP_LIMIT is stored as every k-th
    element of the flattened array, k the smallest stride that fits, so that two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_LIMIT // len(arrays)
    for name, t in arrays.items():
        t = t.detach()
        a = (t.float() if t.is_floating_point() and t.dtype != torch.float64 else t.double()).cpu().numpy()
        if a.nbytes > share:
            a = a.reshape(-1)[::-(-a.nbytes // share)]
        np.save(os.path.join(out_dir, name + '.npy'), a)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.gpu}', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-lms', '25'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for l in self.lines:
            p = [x.strip() for x in l.split(',')]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for n, v in zip(names, p[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': float(max(mx)) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


# ------------------------------------------------------------------------------------------------ CPU arms
def synthetic_frames(batch, seed=1029):
    torch.manual_seed(seed)  # the trainer's own seed (trainer.py:55)
    return torch.randn(batch, 3, 640, 640)


def usable_cores():
    """Host threads this process may really use: affinity mask, capped by the cgroup CPU quota if one is set."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    for path in ('/sys/fs/cgroup/cpu.max', '/sys/fs/cgroup/cpu/cpu.cfs_quota_us'):
        try:
            txt = open(path).read().split()
            if path.endswith('cpu.max'):
                if txt[0] != 'max':
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    n = min(n, max(1, q // int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())))
        except Exception:
            pass
    return max(1, n)


def pick_cpu_threads(probe):
    """All the host threads the CPU arm can use *productively*: oversubscribed intra-op pools are slower than fewer
    threads, so time a small probe at n, n/2, n/4, ... and keep the fastest (reported as `cores`)."""
    n = usable_cores()
    cands = sorted({max(1, n >> k) for k in range(0, 4)} | {min(n, 32), min(n, 16)}, reverse=True)
    best, best_t = cands[0], float('inf')
    for c in cands:
        torch.set_num_threads(c)
        probe()
        t0 = time.perf_counter()
        probe()
        dt = time.perf_counter() - t0
        if dt < best_t * 0.95:
            best, best_t = c, dt
    return best


def cpu_reference_throughput(steps, warmup, batch=8):
    """The reference's algorithm (oracle port: torch CPU fp32 conv/BN/SiLU graph + numpy NMS) on all host cores."""
    from cvpytorch_b200 import synth
    from oracle import nms_oracle as NO
    from oracle import yolov5_oracle as YO
    sd = synth.yolov5s_state_dict(True)
    x = synthetic_frames(batch)
    cores = pick_cpu_threads(lambda: YO.forward(x[:2], sd))
    torch.set_num_threads(cores)

    def step():
        z, _ = YO.forward(x, sd)
        NO.non_max_suppression(z.numpy(), 0.001, 0.6, multi_label=True)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return batch * steps / dt, cores, dt / steps, f'{steps} steps x bs{batch} 640x640 forward+decode+NMS, torch {torch.__version__} fp32, {cores} threads'


def run_reference_arm(args):
    rank = env_int('RANK', 0)
    if rank != 0:
        return
    steps = max(1, args.steps)
    v, cores, spt, sample = cpu_reference_throughput(steps, max(1, min(args.warmup, 2)))
    line = {'impl': 'reference', 'metric': METRIC, 'value': round(v, 3), 'unit': 'images/sec', 'n_gpus': args.gpus, 'steps': steps,
            'warmup': max(1, min(args.warmup, 2)), 'ms_per_step': round(spt * 1e3, 3), 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'YOLOv5-s 640x640 forward+decode+NMS (conf/coco_yolov5_s.yml), CPU sample bs8 per step', 'parallelism': 'cpu'},
            'cpu_baseline': {'value': round(v, 3), 'unit': 'images/sec', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': round(v, 3), 'unit': 'images/sec', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ B200 arm
def _dist_setup():
    import torch.distributed as dist
    world = env_int('WORLD_SIZE', 1)
    rank = env_int('RANK', 0)
    local = env_int('LOCAL_RANK', 0)
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    from cvpytorch_b200.runtime import bind_to_gpu_numa_node
    numa = bind_to_gpu_numa_node(local)  # before any pinned allocation: host buffers land on the GPU's NUMA node
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t[0])
        return ms

    return dist, world, rank, local, dev, numa, barrier, max_over_ranks


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        return {}


def time_conv_stack(g, K2=10):
    """The conv launches of one step replayed back to back as their OWN CUDA graph (same launch conditions as the timed graph replays,
    no aux kernels in between), CUDA events around K2 replays -> ms per step of the conv stack for the roofline."""
    from cvpytorch_b200 import ops
    plans = [s[1] for s in g.steps if s[0] == 'conv']
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.run_plans(plans)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    cg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(cg):
        ops.run_plans(plans)
    for _ in range(2):
        cg.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K2):
        cg.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / K2


def per_layer_bound_ms(g, B, peak_tf, hbm):
    bound_ms = 0.0
    for (_n, cin, cout, k, s_, Ho, Wo) in g.layer_log:
        fl = 2.0 * B * Ho * Wo * cout * cin * k * k
        by = 4.0 * (B * (Ho * s_) * (Wo * s_) * cin + B * Ho * Wo * cout) + 4.0 * cout * cin * k * k
        bound_ms += max(3 * fl / (peak_tf * 1e12), by / (hbm * 1e9)) * 1e3
    return bound_ms


def run_b200_arm(args):
    from cvpytorch_b200 import _lib, synth
    from cvpytorch_b200 import dist as cdist
    from cvpytorch_b200 import ops
    from cvpytorch_b200.runtime import InferencePipeline
    dist, world, rank, local, dev, numa, barrier, max_over_ranks = _dist_setup()
    B = args.batch
    if args.scaling == 'strong':
        # fixed global batch (args.batch images in total), contiguous shards per rank (SURVEY.md 8e: global B=64 -> 8 img/GPU at W=8)
        if args.batch % world != 0:
            raise SystemExit('--scaling strong needs --batch divisible by the number of GPUs')
        B = args.batch // world
    model = synth.build_yolov5s(calibrated=True)
    K, W = args.steps, max(3, args.warmup)

    # ------------------------------------------------------------- device-resident arm ("value")
    G = model.build_graph(B, 640, 640, dev)
    g, ws = G['g'], G['ws']
    NBUF = 4  # distinct device-resident input batches, used round robin (every timed step reads a different 315 MB buffer)
    x_devs = [synthetic_frames(B, seed=1029 + rank + 97 * i).to(dev) for i in range(NBUF)]
    G['holder']['x'] = x_devs[0]
    gathered = torch.empty((world, cdist.packed_len(B, ws.max_det)), dtype=torch.float32, device=dev)

    def tail():  # the one collective of the path, from the buffer the NMS kernels wrote (no packing kernels)
        if world > 1:
            cdist.all_gather_packed(ws.packed, gathered)

    steps_list = g.steps

    def run_step(events=None):
        """One eager pass of the hot path.  events: list to append (start, end) CUDA event pairs around the conv segments."""
        i, n = 0, len(steps_list)
        while i < n:
            kind, obj = steps_list[i]
            if kind == 'conv':
                j = i
                while j < n and steps_list[j][0] == 'conv':
                    j += 1
                if events is not None:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                ops.run_plans([s[1] for s in steps_list[i:j]])
                if events is not None:
                    e1.record()
                    events.append((e0, e1))
                i = j
            else:
                obj()
                i += 1
        tail()

    graphs = []
    if args.graph:
        if world > 1:
            tail()  # NCCL communicator must exist before a capture can record the collective
            torch.cuda.synchronize()
        for i in range(NBUF):  # one captured step per input buffer (activation buffers are shared); the all-gather is part of the graph
            G['holder']['x'] = x_devs[i]
            g._graph = None
            graphs.append(g.capture(warmup=2 if i == 0 else 1, tail=tail if world > 1 else None))

    def do_step(i, events=None):
        if args.graph:
            graphs[i % NBUF].replay()
        else:
            G['holder']['x'] = x_devs[i % NBUF]
            run_step(events)

    for i in range(W):
        do_step(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = _lib.launch_count()
    ev = []
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_start.record()
    for i in range(K):
        do_step(i, ev if not args.graph else None)
    t_end.record()
    barrier()
    total_ms = max_over_ranks(t_start.elapsed_time(t_end))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # before the eager passes below overwrite the graph's output buffers
        dump_outputs(args.dump_outputs, {'det': ws.det, 'det_idx': ws.det_idx, 'det_count': ws.det_count})
    ms_per_step = total_ms / K
    value = world * B * K / (total_ms / 1e3)
    launches = _lib.launch_count() - n0
    conv_ms = None
    conv_graph_ms = None
    conv_how = 'CUDA events around the conv segments of the timed eager steps'
    if ev:
        conv_ms = sum(a.elapsed_time(b) for a, b in ev) / K
    if args.graph:
        # graph replays do not pass through the C ABI: one eager pass (outside the timed region) counts the kernels of a step; the conv
        # stack is timed as its own CUDA graph (all conv launches of a step back to back, same launch conditions as the timed replays)
        n1 = _lib.launch_count()
        G['holder']['x'] = x_devs[0]
        run_step()
        torch.cuda.synchronize()
        launches = (_lib.launch_count() - n1) * K
        ev2 = []
        K2 = min(max(K, 5), 20)
        for i in range(K2):
            G['holder']['x'] = x_devs[i % NBUF]
            run_step(ev2)
        torch.cuda.synchronize()
        conv_ms = sum(a.elapsed_time(b) for a, b in ev2) / K2
        conv_how = 'CUDA events around the conv segments of %d eager passes of the step (run right after the timed graph replays; same method as round 1)' % K2
        conv_graph_ms = time_conv_stack(g, K2=K2)
    overflow = int(ws.status[0].item())

    # ------------------------------------------------------------- end-to-end arm ("e2e"): pinned host in, host out
    def time_pipeline(pipe, hosts):
        for i in range(W):
            pipe.result(pipe.submit(hosts[i % len(hosts)]))
        barrier()
        smp = ClockSampler(local)
        if rank == 0:
            smp.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        slots = []
        for i in range(K):
            slots.append(pipe.submit(hosts[i % len(hosts)]))
            if i >= 1:
                pipe.result(slots[i - 1])  # host reads the previous step's detections while this one runs
        last = pipe.result(slots[-1])
        torch.cuda.current_stream().wait_event(pipe.ev_host[slots[-1]])  # chain the pipeline's last D2H into the timing stream
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1))
        return ms, last, (smp.stop() if rank == 0 else None)

    del graphs, x_devs
    pipe = InferencePipeline(model, B, 640, 640, dev, depth=2, use_cuda_graph=True)
    hosts = [synthetic_frames(B, seed=2000 + rank * 16 + i).pin_memory() for i in range(3)]
    e2e_ms, last, e2e_clk = time_pipeline(pipe, hosts)
    e2e_value = world * B * K / (e2e_ms / 1e3)
    kept_mean = float(last[2].float().mean())
    h2d_f32, d2h_f32 = pipe.h2d_bytes, pipe.d2h_bytes
    del pipe, hosts

    # same end-to-end loop fed with camera-side uint8 HWC frames (ToTensor + Normalize fused into the stem loader; SURVEY.md 8 f-1)
    pipe8 = InferencePipeline(model, B, 640, 640, dev, depth=2, use_cuda_graph=True, uint8_frames=True)

    def frames_u8(seed):
        # uint8 frames whose transformed values follow the same N(0,1) statistics as the fp32 arm (quantised to 1/255, clipped to [0,1]):
        # the NMS workload is data dependent, uniform byte noise would time a different candidate regime
        z = synthetic_frames(B, seed=seed)
        nm = model.input_norm
        m = torch.tensor(nm['mean'], dtype=torch.float32).view(1, 3, 1, 1)
        sd = torch.tensor(nm['std'], dtype=torch.float32).view(1, 3, 1, 1)
        u = ((z * sd + m) * 255.0).round_().clamp_(0, 255).to(torch.uint8)   # tensor (RGB, CHW) order
        return u.flip(1).permute(0, 2, 3, 1).contiguous().pin_memory()      # camera order: HWC, BGR

    hosts8 = [frames_u8(3000 + rank * 16 + i) for i in range(3)]
    e2e8_ms, _, e2e8_clk = time_pipeline(pipe8, hosts8)
    e2e8_value = world * B * K / (e2e8_ms / 1e3)
    h2d8, d2h8 = pipe8.h2d_bytes, pipe8.d2h_bytes

    if rank == 0:
        peaks = _peaks()
        peak_tf = float(peaks.get('bf16_tflops_sustained', 1400.0))
        peak_src = 'measured bf16_tflops_sustained (MEASURED_PEAKS.json)' if peaks else 'fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)'
        roof = None
        if conv_ms:
            ach = ALG_GFLOP_PER_IMG * B / conv_ms  # GFLOP / ms == TFLOP/s
            traffic, traffic_src = measured_conv_traffic(B)
            hbm = float(peaks.get('hbm_gbs', 6500.0))
            bound_ms = per_layer_bound_ms(g, B, peak_tf, hbm)
            roof = {'bound': 'tensor', 'achieved': round(ach, 2), 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': round(ach / peak_tf, 4),
                    'traffic': traffic, 'traffic_source': traffic_src,
                    'kernel': 'conv_tc_kernel<*> (all %d fused conv launches of one step)' % g.n_convs,
                    'conv_ms_per_step': round(conv_ms, 4), 'conv_ms_how': conv_how, 'peak_source': peak_src,
                    'conv_ms_as_own_graph': round(conv_graph_ms, 4) if conv_graph_ms else None,
                    'algorithmic_bytes_per_step': int(7.80e9 * B / 64), 'kernel_sources_sha1': csrc_sha1(),
                    'per_layer_roofline': {'bound_ms': round(bound_ms, 4), 'frac': round(bound_ms / conv_ms, 4),
                                           'definition': 'sum over the conv layers of max(3*flops/P_tensor, bytes/BW_hbm): three fp16 MMA products per '
                                                         'fp32 product, activations stored as fp16 hi+lo (4 B/element); P = %.1f TF/s, BW = %.1f GB/s' % (peak_tf, hbm)},
                    'note': 'algorithmic FLOPs 2*M*N*K of the fp32 reference graph (1051.75 GFLOP/bs64); the kernel issues 3 fp16 MMA products per fp32 '
                            'product (hi/lo split, fp32-equivalent accuracy), so frac <= 1/3 by construction; traffic = dram read+write of the conv '
                            'launches of one step (ncu), reported only when captured on the current kernel sources; per-layer numbers in profiles/'}
        cpu_v, cores, spt, sample = cpu_reference_throughput(args.cpu_steps, 1) if (args.cpu_steps > 0 and world == 1) else (
            None, 0, 0, 'skipped (timed at N=1 only)' if world > 1 else 'skipped')
        line = {'metric': METRIC, 'value': round(value, 2), 'unit': 'images/sec', 'n_gpus': world, 'steps': K, 'warmup': W,
                'ms_per_step': round(ms_per_step, 4), 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
                'dtype': 'fp16x3-split (fp32-equivalent, fp32 accumulate)', 'data': 'synthetic',
                'config': {'workload': 'YOLOv5-s 640x640 forward+decode+NMS, bs64 per GPU (conf/coco_yolov5_s.yml; BASELINE.json configs[1])',
                           'global_batch': world * B, 'per_gpu_batch': B, 'parallelism': f'dp{world}', 'conf_thres': 0.001, 'iou_thres': 0.6,
                           'weights': 'synthetic, BN-calibrated (tests/golden/yolov5s_calib.npz)', 'cuda_graph': bool(args.graph),
                           'l2': 'per-step inputs 315 MB (%d device buffers used round robin) and activations > 126 MB L2 (no explicit flush needed)' % NBUF,
                           'collective': ('one all_gather_into_tensor of the NMS result buffer [B*300*7+B] f32 per step, captured inside the CUDA graph'
                                          if args.graph else 'one eager all_gather_into_tensor per step') if world > 1 else 'none (N=1)',
                           'numa_node': numa, 'kept_per_image_mean': kept_mean, 'nms_capacity_overflow': overflow},
                'gpu_launches': int(launches),
                'e2e': {'value': round(e2e_value, 2), 'unit': 'images/sec', 'h2d_bytes_per_step': h2d_f32, 'd2h_bytes_per_step': d2h_f32,
                        'ms_per_step': round(e2e_ms / K, 4), 'sm_mhz': (e2e_clk or {}).get('sm_mhz'),
                        'api': 'cvpytorch_b200.runtime.InferencePipeline.submit/result (pinned host fp32 frames in, host detections out)'},
                'e2e_uint8_frames': {'value': round(e2e8_value, 2), 'unit': 'images/sec', 'h2d_bytes_per_step': h2d8, 'd2h_bytes_per_step': d2h8,
                                     'ms_per_step': round(e2e8_ms / K, 4), 'sm_mhz': (e2e8_clk or {}).get('sm_mhz'),
                                     'api': 'InferencePipeline(uint8_frames=True): pinned host uint8 HWC frames in (ToTensor + Normalize fused into the stem '
                                            'loader, cvb_stem_s2d_u8), host detections out; an extension beyond the reference input contract'},
                'clocks': clocks, 'roofline': roof,
                'cpu_baseline': {'value': round(cpu_v, 3) if cpu_v else None, 'unit': 'images/sec', 'cores': cores, 'kind': 'port', 'sample': sample,
                                 'note': 'oracle port with an early-exit numpy NMS: faster than the stock reference path (the reference\'s own '
                                         'non_max_suppression is ~10x slower per image on CPU), i.e. generous to the CPU'}}
        print(json.dumps(line), flush=True)
    if world > 1:
        # CUDA graphs that captured the NCCL all-gather are still alive here; tearing the process group down underneath them can hang
        # (seen at N=2).  Everything is measured and printed: synchronise, meet the other ranks once more and leave without the teardown.
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


# ------------------------------------------------------------------------------------------------ secondary configurations
def _secondary_model(name):
    from cvpytorch_b200 import synth
    return {'fcos': synth.build_fcos, 'deeplab': synth.build_deeplab, 'yolox': synth.build_yolox}[name](True)


def _secondary_cpu(name, steps, batch=1):
    """Oracle port of the configuration on the host cores, bounded sample (bs1 steps)."""
    from cvpytorch_b200 import synth
    cfg = SECONDARY[name]
    H, W = cfg['hw']
    torch.manual_seed(1029)
    x = torch.randn(batch, 3, H, W)
    if name == 'fcos':
        from oracle import fcos_oracle as O
        sd = synth.fcos_state_dict(True)

        def step():
            _, _, cls, cnt, reg = O.forward(x, sd)
            O.fcos_detect(cls, cnt, reg)
    elif name == 'deeplab':
        from oracle import deeplab_oracle as O
        sd = synth.deeplab_state_dict(True)

        def step():
            O.forward(x, sd)
    else:
        from oracle import yolox_oracle as O
        sd = synth.yolox_state_dict(True)

        def step():
            O.post_process(O.forward(x, sd))
    small = x[:, :, :H // 4, :W // 4].contiguous()
    probe_fn = {'fcos': lambda: __import__('oracle.fcos_oracle', fromlist=['x']).forward(small, sd),
                'deeplab': lambda: __import__('oracle.deeplab_oracle', fromlist=['x']).forward(small, sd),
                'yolox': lambda: __import__('oracle.yolox_oracle', fromlist=['x']).forward(small, sd)}[name]
    cores = pick_cpu_threads(probe_fn)
    torch.set_num_threads(cores)
    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return batch * steps / dt, cores, dt / steps, f'{steps} steps x bs{batch} {H}x{W} forward+post-process, torch {torch.__version__} fp32, {cores} threads'


def run_secondary_arm(args):
    from cvpytorch_b200 import _lib
    from cvpytorch_b200 import dist as cdist
    name = args.config
    cfg = SECONDARY[name]
    dist, world, rank, local, dev, numa, barrier, max_over_ranks = _dist_setup()
    B = args.batch or cfg['batch']
    H, Wd = cfg['hw']
    model = _secondary_model(name)
    K, W = args.steps, max(3, args.warmup)
    G = model.build_graph(B, H, Wd, dev)
    g = G['g']
    NBUF = 2
    x_devs = [torch.randn(B, 3, H, Wd, generator=torch.Generator().manual_seed(1029 + rank + 97 * i)).to(dev) for i in range(NBUF)]
    G['holder']['x'] = x_devs[0]

    # results of one step + the collective of the configuration (dist.py helpers; eager NCCL call after the replay)
    def results():
        if name == 'fcos':
            ws = G['ws']
            return ws.out_scores, ws.out_classes, ws.out_boxes, ws.out_count
        if name == 'deeplab':
            return (G['labels'],)
        return G['ws'].det, G['ws'].count

    def gather():
        if world == 1:
            return
        if name == 'fcos':
            sc, cl, bx, cnt = results()
            cdist.all_gather_fcos_detections(sc, cl, bx, cnt)
        elif name == 'deeplab':
            cdist.all_gather_label_maps(G['labels'], check=False)
        else:
            det, cnt = results()
            out = torch.empty((world,) + tuple(det.shape), dtype=det.dtype, device=dev)
            dist.all_gather_into_tensor(out, det.contiguous())
            outc = torch.empty((world,) + tuple(cnt.shape), dtype=cnt.dtype, device=dev)
            dist.all_gather_into_tensor(outc, cnt.contiguous())

    graphs = []
    for i in range(NBUF):
        G['holder']['x'] = x_devs[i]
        g._graph = None
        graphs.append(g.capture(warmup=2 if i == 0 else 1))

    def do_step(i):
        graphs[i % NBUF].replay()
        gather()

    for i in range(W):
        do_step(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0.record()
    for i in range(K):
        do_step(i)
    t1.record()
    barrier()
    total_ms = max_over_ranks(t0.elapsed_time(t1))
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * K / (total_ms / 1e3)
    if args.dump_outputs and rank == 0:  # before g.run() below overwrites the graph's output buffers
        names = {'fcos': ('scores', 'classes', 'boxes', 'count'), 'deeplab': ('labels',), 'yolox': ('det', 'count')}[name]
        dump_outputs(args.dump_outputs, dict(zip(names, results())))
    n1 = _lib.launch_count()
    g.run()
    torch.cuda.synchronize()
    launches = (_lib.launch_count() - n1) * K
    conv_ms = time_conv_stack(g, K2=min(max(K, 3), 10))
    status = int(G['ws'].status[0].item()) if name == 'fcos' else 0

    # ---- end to end: pinned host fp32 frames -> device -> graph -> (gather) -> results to pinned host, every step
    hosts = [torch.randn(B, 3, H, Wd, generator=torch.Generator().manual_seed(2000 + rank * 16 + i)).pin_memory() for i in range(2)]
    x_in = x_devs[0]
    G['holder']['x'] = x_in

    def result_tensors():
        r = results()
        if name == 'deeplab':  # class ids < 256: the label maps travel as uint8 (2 MB / image instead of 16 MB), widened on the host if needed
            return (r[0].to(torch.uint8),)
        return r
    outs_host = [torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in result_tensors()]
    h2d = x_in.numel() * 4
    d2h = sum(t.numel() * t.element_size() for t in outs_host)

    def e2e_step(i):
        x_in.copy_(hosts[i % 2], non_blocking=True)
        graphs[0].replay()
        gather()
        for h, t in zip(outs_host, result_tensors()):
            h.copy_(t, non_blocking=True)

    for i in range(W):
        e2e_step(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        e2e_step(i)
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = world * B * K / (e2e_ms / 1e3)

    if rank == 0:
        peaks = _peaks()
        peak_tf = float(peaks.get('bf16_tflops_sustained', 1400.0))
        hbm = float(peaks.get('hbm_gbs', 6500.0))
        ach = g.flops / conv_ms / 1e9  # FLOP / ms / 1e9 == TFLOP/s
        bound_ms = per_layer_bound_ms(g, B, peak_tf, hbm)
        roof = {'bound': 'tensor', 'achieved': round(ach, 2), 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': round(ach / peak_tf, 4), 'traffic': None,
                'kernel': 'conv_tc_kernel<*> (all %d tensor-core conv launches of one step)' % g.n_convs, 'conv_ms_per_step': round(conv_ms, 4),
                'algorithmic_gflop_per_image': round(g.flops / B / 1e9, 3), 'kernel_sources_sha1': csrc_sha1(),
                'per_layer_roofline': {'bound_ms': round(bound_ms, 4), 'frac': round(bound_ms / conv_ms, 4)},
                'note': 'algorithmic 2*M*N*K of the tensor-core convs (depthwise / GroupNorm / pooling / decode / NMS kernels excluded); three fp16 '
                        'MMA products per fp32 product, so frac <= 1/3 by construction'}
        cpu_v, cores, spt, sample = _secondary_cpu(name, args.cpu_steps) if (args.cpu_steps > 0 and world == 1) else (
            None, 0, 0, 'skipped (timed at N=1 only)' if world > 1 else 'skipped')
        line = {'metric': cfg['metric'], 'value': round(value, 2), 'unit': 'images/sec', 'n_gpus': world, 'steps': K, 'warmup': W,
                'ms_per_step': round(total_ms / K, 4), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'fp16x3-split (fp32-equivalent, fp32 accumulate)', 'data': 'synthetic',
                'config': {'workload': cfg['workload'], 'global_batch': world * B, 'per_gpu_batch': B, 'parallelism': f'dp{world}',
                           'weights': 'synthetic, calibrated (tests/golden/*_calib.npz)', 'cuda_graph': True,
                           'l2': 'inputs and activations of one step exceed the 126 MB L2 (no explicit flush needed)',
                           'collective': cfg['collective'] if world > 1 else 'none (N=1)', 'numa_node': numa, 'nms_capacity_overflow': status},
                'gpu_launches': int(launches),
                'e2e': {'value': round(e2e_value, 2), 'unit': 'images/sec', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                        'ms_per_step': round(e2e_ms / K, 4),
                        'api': 'pinned host fp32 frames -> model graph (== model.predict) -> results copied to pinned host memory, every step'},
                'clocks': clocks, 'roofline': roof,
                'cpu_baseline': {'value': round(cpu_v, 4) if cpu_v else None, 'unit': 'images/sec', 'cores': cores, 'kind': 'port', 'sample': sample}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


TRAIN_CFG = dict(cin=128, cout=128, n=3, hw=(80, 80), batch=16,
                 metric='images/sec YOLOX-s dark3 C3 block (CSPLayer 128->128, n=3, 80x80) training step fwd+bwd+SGD, bf16, bs16 per GPU',
                 workload='one C3 block of the YOLOX-s backbone (dark3: CSPLayer(128,128,n=3) on the 80x80 map of a 640x640 image), training step: forward + backward '
                          '+ gradient all-reduce + SGD(momentum) update, bf16 activations / gradients, fp32 master weights; bs16 per GPU = BASELINE.json configs[3] '
                          "(batch 128 over 8 GPUs); the block is the part of configs[3] built so far (SURVEY.md 8(f) rank 3)")


def _train_flops(B, H, W, cin, cout, n):
    hid = cout // 2
    npix = B * H * W
    convs = [(cin, hid, 1), (cin, hid, 1), (2 * hid, cout, 1)] + [(hid, hid, 1), (hid, hid, 3)] * n
    fwd = sum(2.0 * npix * ci * co * k * k for ci, co, k in convs)
    return 3.0 * fwd  # forward + backward-data + backward-weight


def _train_cpu(steps, B=2):
    """The oracle's training step (reference block restated, torch.autograd backward) on the host cores: bounded sample."""
    from oracle import c3_train_oracle as CO
    c = TRAIN_CFG
    H, W = c['hw']
    sd = CO.synthetic_state(c['cin'], c['cout'], c['n'])
    g = torch.Generator().manual_seed(5)
    x, G = torch.randn(B, c['cin'], H, W, generator=g), torch.randn(B, c['cout'], H, W, generator=g)
    cores = pick_cpu_threads(lambda: CO.train_step(x[:1, :, :20, :20], G[:1, :, :20, :20], sd, c['n']))
    torch.set_num_threads(cores)
    CO.train_step(x, G, sd, c['n'])
    t0 = time.perf_counter()
    for _ in range(steps):
        CO.train_step(x, G, sd, c['n'])
    dt = time.perf_counter() - t0
    return B * steps / dt, cores, dt / steps, f'{steps} steps x bs{B} 80x80 forward+backward of the block, torch {torch.__version__} fp32 autograd, {cores} threads'


def run_train_arm(args):
    """--config c3train: the training step of one YOLOX C3 block on the B200 kernels (cvpytorch_b200/train.py)."""
    from cvpytorch_b200 import _lib, train as T
    from oracle import c3_train_oracle as CO  # (parameters only: the seeded state the CPU leg also uses)
    c = TRAIN_CFG
    dist, world, rank, local, dev, numa, barrier, max_over_ranks = _dist_setup()
    B = args.batch or c['batch']
    H, Wd = c['hw']
    K, W = args.steps, max(3, args.warmup)
    m = T.CSPLayer(c['cin'], c['cout'], n=c['n'])
    m.load_state_dict({k: torch.as_tensor(v) for k, v in CO.synthetic_state(c['cin'], c['cout'], c['n']).items()})
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.eps, mod.momentum = 1e-3, 0.03
    m.to(dev).train()
    params = [p for p in m.parameters()]
    opt = torch.optim.SGD(params, lr=1e-3, momentum=0.9)
    NBUF = 4
    gen = torch.Generator().manual_seed(1029 + rank)
    xs = [torch.randn(B, H, Wd, c['cin'], generator=gen).to(dev).to(torch.bfloat16) for _ in range(NBUF)]   # NHWC bf16: the layout between blocks
    Gs = [torch.randn(B, H, Wd, c['cout'], generator=gen).to(dev).to(torch.bfloat16) for _ in range(NBUF)]  # stand-in for d(loss)/d(out) of the rest of the net

    def allreduce_grads():  # data-parallel gradient all-reduce (one flat fp32 bucket: 0.3 M parameters)
        if world == 1:
            return
        flat = torch.cat([p.grad.reshape(-1) for p in params])
        dist.all_reduce(flat)
        flat /= world
        off = 0
        for p in params:
            p.grad.copy_(flat[off:off + p.numel()].view_as(p.grad))
            off += p.numel()

    def step(i):
        x = xs[i % NBUF].requires_grad_(True)
        y = m.forward_nhwc(x)
        y.backward(Gs[i % NBUF])
        allreduce_grads()
        opt.step()
        opt.zero_grad(set_to_none=True)
        x.grad = None

    # the whole step (forward, backward, optimiser) as ONE CUDA graph: 100+ launches per step make the eager step CPU-launch bound.
    # (N > 1 keeps the eager step: the gradient all-reduce sits between backward and the update)
    graphed = None
    eager_step = step
    if args.graph and world == 1:
        try:
            sx = xs[0].clone().requires_grad_(True)
            sG = Gs[0].clone()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    m.forward_nhwc(sx).backward(sG)
                    opt.step()
                    opt.zero_grad(set_to_none=True)
                    sx.grad = None
            torch.cuda.current_stream().wait_stream(side)
            graphed = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graphed):
                m.forward_nhwc(sx).backward(sG)
                opt.step()
                opt.zero_grad(set_to_none=True)

            def step(i):  # noqa: F811
                sx.detach().copy_(xs[i % NBUF])
                sG.copy_(Gs[i % NBUF])
                graphed.replay()
            for i in range(W):
                step(i)
        except Exception as ex:  # noqa: BLE001
            print(f'[bench] CUDA graph capture of the training step failed ({ex}); timing the eager step', file=sys.stderr)
            graphed = None
            step = eager_step
    if graphed is None:
        for i in range(W):
            step(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0.record()
    for i in range(K):
        step(i)
    t1.record()
    barrier()
    total_ms = max_over_ranks(t0.elapsed_time(t1))
    if args.dump_outputs and rank == 0:  # the block's parameters and BatchNorm statistics after the last step, before eager_step(0) below
        dump_outputs(args.dump_outputs, m.state_dict())
    n0 = _lib.launch_count()
    eager_step(0)  # (counts the library launches of one step; graph replays do not pass through the C ABI)
    torch.cuda.synchronize()
    launches = (_lib.launch_count() - n0) * K
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * K / (total_ms / 1e3)

    # the tensor-core kernels alone (forward convs, backward-data, backward-weight of every layer), CUDA events around them
    def conv_only():
        x = xs[0]
        hid = c['cout'] // 2
        t = torch.randn(B, H, Wd, hid, generator=gen).to(dev).to(torch.bfloat16)  # (host RNG: the device generator is tied to the captured graph)
        w1 = (torch.randn(hid, c['cin'], 1, 1, generator=gen) * 0.05).to(dev)
        w3 = (torch.randn(hid, hid, 3, 3, generator=gen) * 0.05).to(dev)
        wo = (torch.randn(c['cout'], c['cin'], 1, 1, generator=gen) * 0.05).to(dev)
        wf1, wb1 = T.pack_weights(w1)
        wf3, wb3 = T.pack_weights(w3)
        wfo, wbo = T.pack_weights(wo)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(2):  # conv1, conv2: 128 -> 64, 1x1
            y = T.conv(x, wf1, hid, 1); T.conv(y, wb1, c['cin'], 1); T.conv_wgrad(x, y, 1)
        for _ in range(c['n']):
            wf11, wb11 = wf3[:, 4:5, :].contiguous(), wb3[:, 4:5, :].contiguous()
            y = T.conv(t, wf11, hid, 1); T.conv(y, wb11, hid, 1); T.conv_wgrad(t, y, 1)
            y = T.conv(t, wf3, hid, 3); T.conv(y, wb3, hid, 3); T.conv_wgrad(t, y, 3)
        y = T.conv(x, wfo, c['cout'], 1); T.conv(y, wbo, c['cin'], 1); T.conv_wgrad(x, y, 1)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)
    conv_only()
    conv_ms = min(conv_only() for _ in range(3))

    # library baseline on the same GPU (context, not the reference arm): the oracle's block through cuDNN / ATen under bf16 autocast
    lib_ms = None
    try:
        sdg = {k: torch.as_tensor(v).to(dev) for k, v in CO.synthetic_state(c['cin'], c['cout'], c['n']).items()}
        for k, v in sdg.items():
            if v.dtype.is_floating_point and 'running_' not in k:
                v.requires_grad_(True)
        xn = xs[0].float().permute(0, 3, 1, 2).contiguous().to(memory_format=torch.channels_last)
        Gn = Gs[0].float().permute(0, 3, 1, 2).contiguous().to(memory_format=torch.channels_last)

        def lib_step():
            xg = xn.detach().requires_grad_(True)
            with torch.autocast('cuda', dtype=torch.bfloat16):
                y = CO.csp_layer(xg, sdg, c['n'])
            y.backward(Gn.to(y.dtype))
            for v in sdg.values():
                v.grad = None
        for _ in range(3):
            lib_step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(10):
            lib_step()
        e1.record()
        torch.cuda.synchronize()
        lib_ms = e0.elapsed_time(e1) / 10
    except Exception as ex:  # noqa: BLE001  (context number only)
        lib_ms = None
        print(f'[bench] library baseline skipped: {ex}', file=sys.stderr)

    # end to end through the reference-facing module call: pinned host NCHW fp32 block input in, fp32 NCHW output + loss value back to the host
    hosts = [torch.randn(B, c['cin'], H, Wd, generator=gen).pin_memory() for _ in range(2)]
    Gn32 = Gs[0].float().permute(0, 3, 1, 2).contiguous()
    x_in = torch.empty(B, c['cin'], H, Wd, device=dev)
    loss_h = torch.empty((), dtype=torch.float32).pin_memory()

    def e2e_step(i):
        x_in.copy_(hosts[i % 2], non_blocking=True)
        xg = x_in.detach().requires_grad_(True)
        y = m(xg)
        loss = (y * Gn32).sum()
        loss.backward()
        allreduce_grads()
        opt.step()
        opt.zero_grad(set_to_none=True)
        loss_h.copy_(loss.detach(), non_blocking=True)
    for i in range(W):
        e2e_step(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        e2e_step(i)
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    if rank == 0:
        peaks = _peaks()
        peak_tf = float(peaks.get('bf16_tflops_sustained', 1400.0))
        hbm = float(peaks.get('hbm_gbs', 6500.0))
        flops = _train_flops(B, H, Wd, c['cin'], c['cout'], c['n'])
        ach = flops / conv_ms / 1e9
        # HBM bound of the conv kernels: every conv reads its input + writes its output once in each of the three passes (bf16)
        hid = c['cout'] // 2
        npix = B * H * Wd
        io = [(c['cin'], hid), (c['cin'], hid), (2 * hid, c['cout'])] + [(hid, hid), (hid, hid)] * c['n']
        conv_bytes = sum(3 * 2.0 * npix * (ci + co) for ci, co in io)
        cpu_v, cores, spt, sample = _train_cpu(args.cpu_steps) if (args.cpu_steps > 0 and world == 1) else (None, 0, 0, 'skipped (timed at N=1 only)' if world > 1 else 'skipped')
        line = {'metric': c['metric'], 'value': round(value, 2), 'unit': 'images/sec', 'n_gpus': world, 'steps': K, 'warmup': W, 'ms_per_step': round(total_ms / K, 4),
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16 (fp32 accumulate, fp32 master weights)', 'data': 'synthetic',
                'config': {'workload': c['workload'], 'global_batch': world * B, 'per_gpu_batch': B, 'parallelism': f'dp{world}', 'cuda_graph': graphed is not None,
                           'l2': '4 input / output-gradient buffer pairs used round robin (26 MB each: the block working set is L2 resident on B200, as it is inside the full net)',
                           'collective': 'one NCCL all-reduce of the flat fp32 gradient bucket per step' if world > 1 else 'none (N=1)', 'numa_node': numa},
                'gpu_launches': int(launches),
                'e2e': {'value': round(world * B * K / (e2e_ms / 1e3), 2), 'unit': 'images/sec', 'h2d_bytes_per_step': B * c['cin'] * H * Wd * 4, 'd2h_bytes_per_step': 4,
                        'ms_per_step': round(e2e_ms / K, 4), 'api': 'cvpytorch_b200.train.CSPLayer.__call__ (NCHW fp32 in / out like the reference block) + loss.backward() + optimizer.step(); pinned host input, loss value back'},
                'clocks': clocks,
                'roofline': {'bound': 'hbm', 'achieved': round(conv_bytes / conv_ms / 1e6, 1), 'peak': hbm, 'unit': 'GB/s', 'frac': round(conv_bytes / conv_ms / 1e6 / hbm, 4), 'traffic': None,
                             'kernel': 'tconv_kernel / twgrad_kernel (the 27 conv forward / backward-data / backward-weight launches of one step, timed back to back)',
                             'conv_ms_per_step': round(conv_ms, 4), 'tensor_tflops': round(ach, 1), 'tensor_frac_of_bf16_peak': round(ach / peak_tf, 4),
                             'algorithmic_bytes_per_step': conv_bytes, 'algorithmic_gflop_per_step': round(flops / 1e9, 2), 'kernel_sources_sha1': csrc_sha1(),
                             'note': 'bf16 128/64-channel convolutions at 80x80 are HBM / L2 bound (arithmetic intensity 32-64 flop/B per pass); the step also runs 42 '
                                     'element-wise BatchNorm / SiLU kernels and the torch optimiser'},
                'library_baseline': {'what': 'the same block through cuDNN / ATen (torch autocast bf16, channels_last) forward+backward on this GPU', 'ms_per_step': round(lib_ms, 4) if lib_ms else None},
                'cpu_baseline': {'value': round(cpu_v, 4) if cpu_v else None, 'unit': 'images/sec', 'cores': cores, 'kind': 'port', 'sample': sample}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_train_reference_arm(args):
    if env_int('RANK', 0) != 0:
        return
    steps = args.steps
    v, cores, spt, sample = _train_cpu(steps)
    line = {'impl': 'reference', 'metric': TRAIN_CFG['metric'], 'value': round(v, 4), 'unit': 'images/sec', 'n_gpus': args.gpus, 'steps': steps, 'warmup': 1,
            'ms_per_step': round(spt * 1e3, 3), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': TRAIN_CFG['workload'] + ', CPU sample bs2 per step', 'parallelism': 'cpu'},
            'cpu_baseline': {'value': round(v, 4), 'unit': 'images/sec', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': round(v, 4), 'unit': 'images/sec', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


def run_secondary_reference_arm(args):
    if env_int('RANK', 0) != 0:
        return
    name = args.config
    cfg = SECONDARY[name]
    steps = max(1, args.steps)
    v, cores, spt, sample = _secondary_cpu(name, steps)
    line = {'impl': 'reference', 'metric': cfg['metric'], 'value': round(v, 4), 'unit': 'images/sec', 'n_gpus': args.gpus, 'steps': steps, 'warmup': 1,
            'ms_per_step': round(spt * 1e3, 3), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': cfg['workload'] + ', CPU sample bs1 per step', 'parallelism': 'cpu'},
            'cpu_baseline': {'value': round(v, 4), 'unit': 'images/sec', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': round(v, 4), 'unit': 'images/sec', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None, help='timed steps (default: 100 for yolov5s and the --impl reference arms of the other '
                    'inference configurations, 10 for fcos / deeplab / yolox, 20 for c3train, 5 for the c3train --impl reference arm)')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='yolov5s', choices=['yolov5s', 'c3train'] + sorted(SECONDARY),
                    help='yolov5s (default) = the headline, BASELINE.json configs[1]; fcos / deeplab / yolox = the secondary configurations; '
                         'c3train = the training step of one YOLOX C3 block (the built part of configs[3])')
    ap.add_argument('--batch', type=int, default=0, help='images per GPU per step (default: the configuration\'s own, 64 for yolov5s)')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'], help='weak: --batch images per GPU (default); strong: --batch images in total')
    ap.add_argument('--graph', type=int, default=1, help='1 (default): the timed steps replay captured CUDA graphs (the conv-stack time for the roofline '
                    'comes from the conv launches replayed as their own graph); 0: eager launches with per-conv-segment events inside the timed region')
    ap.add_argument('--cpu-steps', type=int, default=3, help='CPU baseline steps timed on rank 0 (0 = skip)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write the outputs of the last timed step to DIR/<name>.npy '
                    '(rank 0; float32 / float64, at most 64 MB in all)')
    args = ap.parse_args()
    if args.steps is None:  # the secondary GPU steps are 10-50 ms each, the CPU training step takes seconds
        if args.config == 'c3train':
            args.steps = 5 if args.impl == 'reference' else 20
        else:
            args.steps = 100 if (args.config == 'yolov5s' or args.impl == 'reference') else 10
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of the B200 path (--impl b200)')
    if args.config == 'c3train':
        if args.impl == 'reference':
            return run_train_reference_arm(args)
        if not torch.cuda.is_available():
            raise SystemExit('bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)')
        args.cpu_steps = min(args.cpu_steps, 3)
        return run_train_arm(args)
    if args.config == 'yolov5s':
        args.batch = args.batch or 64
        if args.impl == 'reference':
            return run_reference_arm(args)
    else:
        if args.impl == 'reference':
            return run_secondary_reference_arm(args)
        args.cpu_steps = min(args.cpu_steps, 2)
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)')
    if args.config == 'yolov5s':
        run_b200_arm(args)
    else:
        run_secondary_arm(args)


if __name__ == '__main__':
    main()
