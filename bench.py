#!/usr/bin/env python
"""bench.py — frames/s of the full ThinkTwice forward (4 cams x 2 sweeps + LiDAR, K=5) on N B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl b200|reference]

One JSON line on rank 0 (contract in the task statement):
  value      : frames/s, whole job, inputs already resident in HBM (device-timed, max over ranks)
  e2e        : same metric through the public API with HOST (pinned) inputs, H2D + D2H inside the timed region
  roofline   : dominant kernel family (implicit-GEMM convolution), algorithmic FLOPs / CUDA-event time, vs the
               measured dense tensor peak of MEASURED_PEAKS.json
  cpu_baseline: the oracle (plain-PyTorch restatement of the reference forward, incl. its dead work) on the host cores
`--impl reference` times that CPU restatement alone (the reference itself cannot be imported here: mmcv/mmdet3d/
spconv are absent — DESIGN.md), rank 0 only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = json.load(open(os.path.join(ROOT, 'BASELINE.json')))['metric'] if os.path.exists(os.path.join(ROOT, 'BASELINE.json')) else \
    'frames/sec full encoder+decoder fwd (4-cam+LiDAR, 200\u00d7200 BEV) at 1/2/4/8 B200'
SHAPE = ('thinktwice.py config, 4 cams x 2 sweeps 448x896 + 40k-point LiDAR, K=5 decoder '
         '(the config file yields a 21x21 camera BEV / 84x84 LiDAR BEV, not 200x200: SURVEY.md fact 3)')


def workload(batch, world):
    """BASELINE.json configs[] entry this run measures."""
    if batch == 1:
        return f'configs[1]: {SHAPE}, batch 1 per GPU'
    if world == 1:
        return f'configs[2]: {SHAPE}, batch {batch} synthetic frames in one forward, 1 GPU (throughput mode)'
    return (f'configs[3]: {SHAPE}, batch {batch * world} synthetic frames sharded data-parallel over {world} GPUs '
            f'({batch} per GPU per forward), one NCCL gather of the waypoints')
# SURVEY.md §8d: dense MACs per frame (camera 1127.7 G + LiDAR dense 13.7 G + fusion 4.25 G + decoder 63.3 G)
ALGO_FLOPS_PER_FRAME = 2 * 1.209e12


def clocks_sampler(stop, out, idx):
    q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    while not stop.is_set():
        try:
            r = subprocess.run(['nvidia-smi', f'--id={idx}', f'--query-gpu={q}', '--format=csv,noheader,nounits'],
                               capture_output=True, text=True, timeout=5).stdout.strip().split(',')
            out.append([x.strip() for x in r])
        except Exception:
            pass
        stop.wait(0.2)


def summarize_clocks(samples):
    sm = sorted(float(s[0]) for s in samples if len(s) >= 7 and s[0].replace('.', '').isdigit())
    mx = [float(s[1]) for s in samples if len(s) >= 7 and s[1].replace('.', '').isdigit()]
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    reasons = sorted({names[i] for s in samples if len(s) >= 7 for i in range(4) if s[3 + i].lower().startswith('active')})
    return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
            'samples': len(sm)}


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        j = json.load(open(p))
        return j['bf16_tflops_sustained'], j['hbm_gbs'], 'measured (MEASURED_PEAKS.json, sustained bf16 cuBLAS)'
    return 1400.0, 6650.0, 'fallback (B200_PROFILING.md)'


def cpu_oracle_worker(max_frames):
    """child process: time the CPU restatement frame by frame, one line per frame (parent enforces the deadline)."""
    import torch
    from oracle.model import EncoderDecoder as Oracle, calibrate_bn, init_oracle_weights
    from thinktwice_b200.config import Config, DEFAULT_CONFIG
    from thinktwice_b200.synthetic import make_batch
    cfg = Config.fromfile(DEFAULT_CONFIG)
    torch.set_flush_denormal(True)
    try:                                                         # all physical cores (torchrun pins OMP_NUM_THREADS=1 for its children)
        import psutil
        ncores = psutil.cpu_count(logical=False) or os.cpu_count()
    except Exception:
        ncores = max(1, (os.cpu_count() or 2) // 2)
    torch.set_num_threads(ncores)
    print(f'THREADS {torch.get_num_threads()}', flush=True)
    oracle = Oracle(**{k: v for k, v in cfg.model.items() if k != 'type'}).eval()
    init_oracle_weights(oracle, 0)
    batch = make_batch(cfg, 1, seed=0)
    t0 = time.perf_counter()
    calibrate_bn(oracle, batch)                                  # BN statistics for well-conditioned activations; doubles as warm-up
    print(f'WARMUP {time.perf_counter() - t0:.3f}', flush=True)
    with torch.no_grad():
        for _ in range(max_frames):
            t0 = time.perf_counter()
            oracle.forward_inference(batch, dead_work=True)      # the reference executes its dead branches too
            print(f'FRAME {time.perf_counter() - t0:.3f}', flush=True)


def make_weights_worker(out):
    """child process (`--impl make-weights`): the synthetic checkpoint of SURVEY.md §8d — seeded random init of every layer, then
    BatchNorm running statistics set by ONE calibration pass of the CPU oracle over a synthetic frame and frozen, so that activations
    are O(1) like a trained network's (a raw random init drives this network's activations to ~1e6).  Written as an mmcv-style
    checkpoint file; the timed process only ever LOADS it (thinktwice_agent.py:170 path) and never imports oracle/."""
    import torch
    from oracle.model import EncoderDecoder as Oracle, calibrate_bn, init_oracle_weights
    from thinktwice_b200.config import Config, DEFAULT_CONFIG
    from thinktwice_b200.synthetic import make_batch
    cfg = Config.fromfile(DEFAULT_CONFIG)
    torch.set_num_threads(max(1, (os.cpu_count() or 2) // 2))
    oracle = Oracle(**{k: v for k, v in cfg.model.items() if k != 'type'}).eval()
    init_oracle_weights(oracle, 0)
    calibrate_bn(oracle, make_batch(cfg, 1, seed=0))
    tmp = out + f'.tmp{os.getpid()}'
    torch.save({'meta': {'recipe': 'SURVEY.md 8d: seeded init + one oracle BN-calibration pass'}, 'state_dict': oracle.state_dict()}, tmp)
    os.replace(tmp, out)


def synthetic_checkpoint(rank):
    """path of the synthetic calibrated checkpoint; rank 0 creates it (in a child process) when it is not there yet."""
    path = os.path.join(os.environ.get('TT_B200_CKPT_DIR', '/tmp'), 'tt_b200_synthetic_seed0.pth')
    if not os.path.exists(path):
        if rank == 0:
            env = {k: v for k, v in os.environ.items() if k not in ('OMP_NUM_THREADS', 'MKL_NUM_THREADS')}
            subprocess.run([sys.executable, os.path.abspath(__file__), '--impl', 'make-weights', '--out', path], check=True, env=env,
                           stdout=subprocess.DEVNULL)
        t0 = time.time()
        while not os.path.exists(path):
            if time.time() - t0 > 900:
                raise RuntimeError(f'{path} did not appear')
            time.sleep(1.0)
    return path


def cpu_oracle(max_frames, budget_s):
    """frames/s of the CPU restatement on a bounded sample (<= max_frames B=1 frames, <= budget_s seconds)."""
    env = {k: v for k, v in os.environ.items() if k not in ('OMP_NUM_THREADS', 'MKL_NUM_THREADS')}
    p = subprocess.Popen([sys.executable, os.path.abspath(__file__), '--impl', 'reference-worker', '--steps', str(max_frames)],
                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=env)
    frames, threads, warm = [], None, None
    deadline = time.time() + budget_s

    def reader():
        nonlocal threads, warm
        for line in p.stdout:
            k, _, v = line.strip().partition(' ')
            if k == 'THREADS':
                threads = int(v)
            elif k == 'WARMUP':
                warm = float(v)
            elif k == 'FRAME':
                frames.append(float(v))
    th = threading.Thread(target=reader, daemon=True)
    th.start()
    while p.poll() is None and time.time() < deadline:
        time.sleep(0.5)
    if p.poll() is None:
        p.kill()
    th.join(timeout=2)
    note = ''
    if frames:
        fps = len(frames) / sum(frames)
    elif warm:
        fps, note = 1.0 / warm, ' (timed frames did not finish in the budget; value from the calibration pass)'
    else:
        fps, note = 1.0 / budget_s, f' (no frame finished within {budget_s:.0f} s: value is an upper bound)'
    return fps, len(frames), threads or 0, note


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(arrays, out_dir, budget=DUMP_BUDGET_BYTES):
    """write {name: tensor} as out_dir/<name>.npy in float32 (float64 stays float64).  When the whole set exceeds `budget`
    bytes, every array larger than its even share is replaced by a fixed sample: the flat elements at indices drawn without
    replacement from a generator seeded by the array's size, in ascending order, so two runs sample the same elements."""
    import numpy as np
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in arrays.items()}
    total, share = sum(v.nbytes for v in arrays.values()), budget // max(1, len(arrays))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in sorted(arrays.items()):
        if total > budget and v.nbytes > share:
            v = v.reshape(-1)[np.sort(np.random.default_rng(v.size).choice(v.size, size=share // v.itemsize, replace=False))]
        np.save(os.path.join(out_dir, k + '.npy'), v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--batch', type=int, default=32, help='frames per GPU per step (32 = the throughput configs[2] / configs[3])')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference', 'reference-worker', 'make-weights'])
    ap.add_argument('--out', default=None, help='(make-weights) checkpoint file to write')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-latency', action='store_true', help='skip the extra B=1 latency measurement')
    ap.add_argument('--no-graph', action='store_true', help='launch every kernel from the host instead of replaying a CUDA graph')
    ap.add_argument('--dump-convs', default=None, help='write per-conv-launch (name, flops, ms) of one step to this JSON file')
    ap.add_argument('--conv', default='f16s', choices=['simt', '3xtf32', 'tf32', 'f16s'],
                    help='dense-conv engine: tcgen05 scaled-split fp16 (fp32-class, default), tcgen05 3xTF32, single-pass TF32, or SIMT fp32')
    ap.add_argument('--dbg', type=int, default=0, help='experiment: tt_debug_set knob bits (see csrc/gemm_conv_tc.cu)')
    ap.add_argument('--tc-reserve', type=int, default=0, help='experiment: SMs the persistent tcgen05 kernels leave free for the side branch')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='write the prediction dict of the last timed step (inputs resident) as DIR/<name>.npy (rank 0; <= 64 MB in '
                         'all, larger arrays replaced by a fixed seeded sample, see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))

    if args.impl == 'reference-worker':
        return cpu_oracle_worker(args.steps)
    if args.impl == 'make-weights':
        return make_weights_worker(args.out)
    import torch
    from thinktwice_b200.config import Config, DEFAULT_CONFIG
    cfg = Config.fromfile(DEFAULT_CONFIG)
    base = {'metric': METRIC, 'unit': 'frames/s', 'n_gpus': args.gpus, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'data': 'synthetic (seeded N(0,1) images, synthetic LiDAR; seeded random-init weights with BatchNorm statistics calibrated by one oracle pass, SURVEY 8d, loaded from a checkpoint file)',
            'config': {'workload': workload(args.batch, args.gpus), 'frames_per_gpu_per_step': args.batch, 'global_batch': args.batch * args.gpus,
                       'refine_num': 5, 'conv_engine': args.conv, 'cuda_graph': not args.no_graph,
                       'parallelism': f'dp{args.gpus} (frames sharded, one NCCL all_gather of pred_wp)',
                       'l2': 'per-step working set (0.5 GB weights + >1 GB activations per frame) exceeds the 126 MB L2; no explicit flush'}}

    if args.impl == 'reference':
        if rank != 0:
            return
        fps, n, cores, note = cpu_oracle(args.steps, budget_s=200.0)
        line = dict(base, impl='reference', value=fps, steps=n, warmup=1, ms_per_step=1000.0 / fps, dtype='f32',
                    n_gpus=args.gpus, gpu_launches=0,
                    cpu_baseline={'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                                  'sample': f'each step = ONE frame of the {args.batch}-frame batch run through the CPU oracle as a B=1 forward '
                                            f'(a full batch takes minutes per step); {n} frames timed, oracle incl. dead LiDAR-look / ffn work' + note},
                    e2e={'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0})
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), 'bench.py --impl b200 needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    from thinktwice_b200 import lib
    from thinktwice_b200.registry import build_model
    from thinktwice_b200.synthetic import make_batch

    model = build_model(cfg.model)
    ckpt = torch.load(synthetic_checkpoint(rank), map_location='cpu', weights_only=False)      # the agent's checkpoint path
    model.load_state_dict(ckpt['state_dict'])
    model.prepare(dev, impl={'simt': lib.IMPL_SIMT, '3xtf32': lib.IMPL_3XTF32, 'tf32': lib.IMPL_TF32, 'f16s': lib.IMPL_F16S}[args.conv])
    B = args.batch
    host = make_batch(cfg, B, seed=100 + rank)                    # every rank owns different frames (weak scaling)
    for k in ('img', 'points', 'speed', 'target_point', 'target_command'):
        host[k] = host[k].pin_memory()
    resident = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in host.items()}
    from thinktwice_b200.parallel import gather_waypoints
    gathered = torch.empty(world * B, 6, 4, 2, device=dev) if world > 1 else None
    last = {}

    def step(batch):
        pred = model.forward_inference(batch)
        last['pred'] = pred
        wp = pred['pred_wp']
        if world > 1:                                            # the path's single collective: gather of the waypoints
            return gather_waypoints(wp, world, out=gathered)
        return wp

    def timed(batch, steps, read_back):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            wp = step(batch)
            if read_back:
                wp.cpu()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(ms.item())

    if args.tc_reserve or args.dbg:
        lib.load().tt_debug_set((args.tc_reserve << 8) | (args.dbg & 0xFF) | ((args.dbg >> 8) << 16))
    n_eager = lib.launch_count()
    step(resident)                                               # eager step: allocates every buffer, counts launches
    torch.cuda.synchronize()
    launches_per_step = lib.launch_count() - n_eager
    if not args.no_graph:
        model.enable_cuda_graph()                                # the device half becomes one CUDA graph (captured on next call)
    for _ in range(max(args.warmup, 3)):
        step(resident)
    torch.cuda.synchronize()
    stop, samples = threading.Event(), []
    th = threading.Thread(target=clocks_sampler, args=(stop, samples, local_rank), daemon=True)
    th.start()
    ms = timed(resident, args.steps, read_back=False)
    if args.dump_outputs and rank == 0:                          # before the next forward: the bulky outputs are views of the arena
        pred = last['pred']
        dump_outputs({k: pred[k] for k in pred.keys()}, args.dump_outputs)
    launches = launches_per_step * args.steps                    # graph replays execute the same kernel nodes every step
    for _ in range(max(args.warmup, 3)):                         # the host-input path has its own graphs / buffers: warm them outside the timed region
        step(host).cpu()
    torch.cuda.synchronize()
    ms_e2e = timed(host, args.steps, read_back=True)
    stop.set(); th.join(timeout=2)
    # one traced e2e step: when each phase of the pipelined host-input forward finished, relative to its start (ms)
    model._pipe_trace = []
    t_call = time.perf_counter()
    step(host).cpu()
    t_ret = time.perf_counter()
    torch.cuda.synchronize()
    tr = model._pipe_trace
    model._pipe_trace = None
    e2e_trace = None
    if tr:                                                       # device: when each phase finished; host: when its launch was issued
        e2e_trace = {lab: round(tr[0][1].elapsed_time(ev), 2) for lab, ev, _ in tr[1:]}
        e2e_trace['host_issue_ms'] = {lab: round((t - t_call) * 1e3, 2) for lab, _, t in tr}
        e2e_trace['host_call_to_return_ms'] = round((t_ret - t_call) * 1e3, 2)

    # ---- the timed execution mode (graph replay + side stream) must reproduce the plain eager launch sequence
    wp_timed = step(resident).float().cpu().clone()
    wp_e2e = step(host).float().cpu().clone()                    # the e2e leg's mode: host inputs, uploads pipelined against the kernels
    model.use_graph = False
    wp_eager = step(resident).float().cpu()
    parity = float((wp_timed - wp_eager).abs().max() / wp_eager.abs().max().clamp_min(1e-12))
    assert parity < 1e-3 and bool(torch.isfinite(wp_timed).all()), f'graph replay differs from the eager forward: {parity}'
    parity_e2e = float((wp_e2e - wp_eager).abs().max() / wp_eager.abs().max().clamp_min(1e-12))
    assert parity_e2e < 1e-3 and bool(torch.isfinite(wp_e2e).all()), f'pipelined host-input forward differs from the eager forward: {parity_e2e}'
    saturated = model.f16s_saturations()
    assert saturated == 0, f'{saturated} tensor-core operands left the fp16 range (scaled-split engine)'

    # ---- roofline of the dominant kernel family (implicit-GEMM conv): per-launch CUDA events on the launching stream
    model.eng.prof, model.eng.marks = [], []                     # per-launch events need eager, serial launches
    step(resident)
    torch.cuda.synchronize()
    mk = model.eng.marks
    segments = {mk[i][0]: round(mk[i - 1][1].elapsed_time(mk[i][1]), 3) for i in range(1, len(mk))}
    eager_step_ms = mk[0][1].elapsed_time(mk[-1][1])             # the same serial eager step the per-launch events come from
    model.eng.marks = None
    conv_ms = sum(a.elapsed_time(b) for (_, _, a, b) in model.eng.prof)
    conv_flops = sum(f for (_, f, _, _) in model.eng.prof)
    n_conv = len(model.eng.prof)
    if args.dump_convs and rank == 0:
        json.dump([(n, f, a.elapsed_time(b)) for (n, f, a, b) in model.eng.prof], open(args.dump_convs, 'w'))
    model.eng.prof = None
    tensor_peak, hbm_peak, peak_src = load_peaks()
    traffic, traffic_note = None, None
    tpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', 'r2_kernels_b1.json')
    if os.path.exists(tpath):                                    # DRAM bytes per launch from the committed ncu --set full capture
        tj = json.load(open(tpath))
        dom = [l for l in tj['launches'] if 'conv_f16s_kernel' in l['kernel'] and ', 0, ' in l['kernel'] and l['dur_ns'] >= 100e3]
        if dom:
            traffic = sum(l['dram_bytes'] for l in dom) / len(dom)
            traffic_note = ('bytes per launch, dram__bytes_read.sum + dram__bytes_write.sum, mean over the %d dense conv_f16s launches of >= 100 us '
                            'in the committed capture (%s: one eager B=1 forward, tools/ncu_ops.py; per-launch rows in profiles/r2_kernels_b1.md)'
                            % (len(dom), tj['source']))
    achieved = conv_flops / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0

    # ---- closed-loop latency (configs[1]): one frame per forward through the same model, graph replay
    lat = None
    if B != 1 and not args.no_latency:
        host1 = make_batch(cfg, 1, seed=100 + rank)
        res1 = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in host1.items()}
        if not args.no_graph:
            model.use_graph = True
        for _ in range(4):
            model.forward_inference(res1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            model.forward_inference(res1)
        e1.record()
        torch.cuda.synchronize()
        lat = e0.elapsed_time(e1) / 20
        # the same with the streaming BEV cache (SURVEY 8f f2): the history sweep's BEV is the previous tick's key-frame BEV
        model.enable_streaming_bev_cache()
        for _ in range(4):
            model.forward_inference(res1)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(20):
            model.forward_inference(res1)
        e1.record()
        torch.cuda.synchronize()
        lat_stream = e0.elapsed_time(e1) / 20
        model.enable_streaming_bev_cache(False)
        # what the agent sees per tick: the batch in (pinned) host memory, uploads inside the call, waypoints read back (thinktwice_agent.py:452-461)
        lat_host = None
        try:                                                     # an extra key: never at the price of the bench line
            for k in ('img', 'points', 'speed', 'target_point', 'target_command'):
                host1[k] = host1[k].pin_memory()
            for _ in range(4):
                model.forward_inference(host1)['pred_wp'].cpu()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(20):
                model.forward_inference(host1)['pred_wp'].cpu()
            lat_host = (time.perf_counter() - t0) * 1e3 / 20
        except Exception as ex:                                  # noqa: BLE001
            print(f'[bench] closed-loop host-input latency skipped: {ex!r}', file=sys.stderr)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    frames = args.steps * B * world
    h2d = sum(v.numel() * v.element_size() for v in host.values() if torch.is_tensor(v))
    line = dict(base, value=frames / (ms * 1e-3), steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=ms / args.steps,
                dtype={'simt': 'f32', '3xtf32': 'f32 (3xTF32 tensor-core products, fp32 accumulate)', 'tf32': 'tf32',
                       'f16s': 'f32 (operands as scaled-split fp16 pairs hi + lo/2048 = 22 mantissa bits, 3 tensor-core products, fp32 accumulate)'}[args.conv], gpu_launches=launches, clocks=summarize_clocks(samples),
                e2e={'value': frames / (ms_e2e * 1e-3), 'unit': 'frames/s', 'h2d_bytes_per_step': h2d,
                     'd2h_bytes_per_step': B * 6 * 4 * 2 * 4, 'ms_per_step': ms_e2e / args.steps,
                     'mode': 'forward_inference(host batch): pinned-host inputs uploaded inside the call, ordered by first use and overlapped with the '
                             'kernels (LiDAR encoder under the image upload, key-frame images under the history sweeps), waypoints read back every step',
                     'phase_done_ms': e2e_trace},
                roofline={'bound': 'tensor', 'kernel': 'conv_f16s_kernel (implicit-GEMM conv / linear / sparse-conv family on tcgen05, scaled-split fp16 operands; + the few SIMT fallbacks)',
                          'achieved': achieved, 'peak': tensor_peak, 'unit': 'TFLOP/s', 'frac': achieved / tensor_peak,
                          'traffic': traffic, 'traffic_note': traffic_note, 'peak_source': peak_src, 'launches_per_step': n_conv,
                          'kernel_ms_per_step': conv_ms, 'kernel_share_of_step': conv_ms / eager_step_ms,
                          'share_note': 'per-launch CUDA events of one serial eager step (no graph, no stream overlap); share = '
                                        'family time / that step',
                          'algorithmic_flops_per_step': conv_flops,
                          'frac_lower_bound': conv_flops / (ms / args.steps * 1e-3) / 1e12 / tensor_peak,
                          'lower_bound_note': 'family FLOPs / the WHOLE timed (graph-replayed) step: what the family achieves at least'},
                segments_ms_serial_eager=segments, hbm_peak_allocated_gb=round(torch.cuda.max_memory_allocated(dev) / 1e9, 1),
                checks={'timed_mode_vs_eager_pred_wp_relerr': parity, 'e2e_mode_vs_eager_pred_wp_relerr': parity_e2e, 'f16s_saturated_operands': saturated})
    if lat is not None:
        line['latency_b1'] = {'ms_per_frame': lat, 'frames_per_s': 1000.0 / lat,
                              'note': 'configs[1]: one frame per forward (closed-loop mode), same model, CUDA-graph replay, inputs resident',
                              'e2e_host_inputs': None if lat_host is None else {'ms_per_frame': lat_host, 'frames_per_s': 1000.0 / lat_host,
                                                  'note': 'wall clock per call with the batch in pinned host memory (38.5 MB of images uploaded inside the call, '
                                                          'pipelined against the kernels) and the waypoints read back: what the closed-loop agent pays per tick'},
                              'streaming_bev_cache': {'ms_per_frame': lat_stream, 'frames_per_s': 1000.0 / lat_stream,
                                                      'note': 'closed-loop extension (SURVEY 8f f2), NOT the independent-frame metric: the history sweep reuses the previous '
                                                              'tick key-frame BEV (identical for a static rig); timing on a repeated frame'}}
    if not args.no_cpu_baseline and args.gpus == 1:
        fps, n, cores, note = cpu_oracle(2, budget_s=90.0)
        line['cpu_baseline'] = {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                                'sample': f'{n} full thinktwice.py frame(s), B=1, CPU oracle incl. the reference\'s dead work' + note}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
