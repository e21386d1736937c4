#!/usr/bin/env python
"""bench.py — stereo FPS of the online-adaptation hot path on N B200s (BASELINE.json configurations).

One "step" = one pass of the hot path over one batch of stereo pairs per GPU: what a single sess.run(fetches) does in
the reference inner loop (Stereo_Online_Adaptation.py:194-208): forward of the whole network, full-resolution
reprojection loss, the selected train op (MAD module / FULL) with its momentum update, loss read-back.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config C] [--batch B]   # this framework (CUDA, libmadstereo)
  python bench.py --impl reference ...                                          # the reference path on host cores
  python bench.py ... --dump-outputs DIR     # also write what the last timed step computed to DIR/*.npy (dump_outputs)

  --config 3 (default, the headline of BASELINE.json): MADNet + MAD (SEQUENTIAL sampler), 1280x384, 1 frame / GPU
           1: MADNet forward only, 640x384         2: MADNet FULL back-prop, 1280x384
           4: DispNet FULL back-prop, 1280x384     5: MADNet + MAD, 1920x1056, --batch frames / GPU (default 1)

Under torchrun (N>1) every rank processes its own frames (weak scaling); rank 0 prints ONE JSON line.
Before anything is timed rank 0 checks the engine's disparities on the first frame against the CPU oracle
(relative L-inf < 1e-3, the north-star bar) — a fast kernel with different results is not measured.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'real-time-self-adaptive-deep-stereo_b200')
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

L2_MB = 126
CONFIGS = {
    1: dict(net='MADNet', mode='NONE', H=384, W=640,
            metric='stereo FPS (forward only) @640x384',
            workload='MADNet forward only (block_config/MadNet_full.json layers), 640x384, %d frame(s) per GPU per step'),
    2: dict(net='MADNet', mode='FULL', H=384, W=1280,
            metric='stereo FPS (fwd+full backprop) @1280x384',
            workload='MADNet full back-propagation online adaptation, 1280x384, %d frame(s) per GPU per step'),
    3: dict(net='MADNet', mode='MAD', H=384, W=1280,
            metric='stereo FPS (fwd+MAD backprop) @1280x384',
            workload='MADNet MAD adaptation (block_config/MadNet_full.json, SEQUENTIAL sampler => uniform mix of the 5 modules), '
                     '1280x384, %d frame(s) per GPU per step'),
    4: dict(net='Dispnet', mode='FULL', H=384, W=1280,
            metric='stereo FPS (DispNet fwd+full backprop) @1280x384',
            workload='DispNet (block_config/dispnet_full.json layers) forward + full back-propagation online adaptation, 1280x384, '
                     '%d frame(s) per GPU per step'),
    5: dict(net='MADNet', mode='MAD', H=1056, W=1920,
            metric='stereo FPS (fwd+MAD backprop) @1920x1056',
            workload='MADNet MAD adaptation (SEQUENTIAL sampler), 1920x1056 (padded to 1920x1088), %d frame(s) per GPU per step'),
}


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        d = json.load(open(path))
        return {'hbm_gbs': d['hbm_gbs'], 'bf16_tflops': d['bf16_tflops'],
                'bf16_tflops_sustained': d.get('bf16_tflops_sustained', d['bf16_tflops']), 'src': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'src': 'fallback'}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([x.strip() for x in out.strip().split(',')])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace('.', '').isdigit())
        reasons = set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            if len(r) >= 7:
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(n)
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace('.', '').isdigit()]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx[0] if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def usable_cores():
    """Host threads the CPU arm can really use: affinity mask, clipped by the cgroup CPU quota and by 32 (the oracle's
    small convolutions stop scaling long before that)."""
    n = len(os.sched_getaffinity(0))
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return max(1, min(n, 32))


def make_inputs(cfg, batch, n_sets, rank):
    """uint8-valued frames (what the reference decodes from PNG/JPEG) as fp32 and uint8 arrays of identical content."""
    import numpy as np
    from madstereo.synthetic import make_pair
    sets = []
    for i in range(n_sets):
        l, r, _ = make_pair(cfg['H'], cfg['W'], seed=100 * rank + 10 * i, batch=batch)
        l8, r8 = np.clip(np.rint(l), 0, 255).astype(np.uint8), np.clip(np.rint(r), 0, 255).astype(np.uint8)
        sets.append((l8.astype(np.float32), r8.astype(np.float32), l8, r8))
    return sets


# ---------------------------------------------------------------------------------------------------
# large-shape correlation numbers (HBM roofline of the correlation kernel, SURVEY 8d)
# ---------------------------------------------------------------------------------------------------
def corr_large_shapes(dev):
    """The engine's own variant (fused concat: copy_left = 1, `u` channel kept) on HBM-sized shapes, outputs
    pre-allocated, L2 flushed between repetitions, CUDA events on the launching stream.
    Algorithmic bytes: forward B*h*w*(3C + nd + 1)*4 (reads L, R, u; writes the left copy and nd correlation channels),
    backward B*h*w*(4C + nd)*4."""
    import torch
    from ctypes import c_void_p
    from madstereo._lib import lib, check
    out = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    st = c_void_p(torch.cuda.current_stream().cuda_stream)
    P = lambda t: c_void_p(t.data_ptr() if t is not None else 0)

    def timeit(run):
        for _ in range(3):
            run()
        ts = []
        for _ in range(7):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); run(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        return ts[len(ts) // 2] * 1e3

    # MADNet level 2 at 1920x1088, 8 frames: fused-concat forward (what Engine::forward launches) and backward
    b, h, w, c, d = 8, 272, 480, 32, 2
    nd = 2 * d + 1
    ocs = (c + nd + 1 + 3) // 4 * 4
    x = torch.randn(b, h, w, c, device=dev); y = torch.randn(b, h, w, c, device=dev)
    cost = torch.zeros(b, h, w, ocs, device=dev)
    cost[..., c + nd] = torch.rand(b, h, w, device=dev) * 4 - 2          # the u channel lives inside the concat buffer
    u = cost[..., c + nd:]
    us = timeit(lambda: check(lib().ms_corr_fwd(P(x), c, P(y), c, P(u), ocs, P(cost), ocs, b, h, w, c, d, 1, 1, 1, st), 'corr_fwd'))
    byts = b * h * w * (3 * c + nd + 1) * 4
    out['madnet_L2_1920x1088_B8_fused_concat'] = {'us': us, 'bytes': byts, 'gbs': byts / us / 1e3}
    o = torch.empty(b, h, w, nd, device=dev); u1 = (torch.rand(b, h, w, 1, device=dev) * 4 - 2)
    us = timeit(lambda: check(lib().ms_corr_fwd(P(x), c, P(y), c, P(u1), 1, P(o), nd, b, h, w, c, d, 1, 0, 0, st), 'corr_fwd'))
    byts = b * h * w * (2 * c + nd + 1) * 4
    out['madnet_L2_1920x1088_B8_plain'] = {'us': us, 'bytes': byts, 'gbs': byts / us / 1e3}
    g = torch.randn(b, h, w, ocs, device=dev); dl = torch.empty_like(x); dr = torch.empty_like(x)
    us = timeit(lambda: check(lib().ms_corr_bwd(P(x), c, P(y), c, P(u), ocs, P(g), ocs, P(dl), c, P(dr), c, P(None), 1,
                                                b, h, w, c, d, 1, 1, st), 'corr_bwd'))
    byts = b * h * w * (4 * c + nd + 1 + c) * 4
    out['madnet_L2_1920x1088_B8_bwd'] = {'us': us, 'bytes': byts, 'gbs': byts / us / 1e3,
                                         'bytes_note': 'reads L, R, u, dcost (C + nd channels); writes dL, dR'}
    del x, y, cost, o, g, dl, dr
    # DispNet correlation (C=128, 81 displacements)
    b, h, w, c, d = 1, 96, 320, 128, 40
    nd = 2 * d + 1
    x = torch.randn(b, h, w, c, device=dev); y = torch.randn(b, h, w, c, device=dev); o = torch.empty(b, h, w, nd, device=dev)
    us_cc = timeit(lambda: check(lib().ms_corr_fwd(P(x), c, P(y), c, P(None), 1, P(o), nd, b, h, w, c, d, 1, 0, 0, st), 'corr_fwd'))
    us = timeit(lambda: check(lib().ms_corr_fwd_wide(P(x), c, P(y), c, P(o), nd, b, h, w, c, d, 64.0, st), 'corr_fwd_wide'))
    byts = b * h * w * (2 * c + nd) * 4
    out['dispnet_1280x384'] = {'us': us, 'bytes': byts, 'gbs': byts / us / 1e3, 'flops': 2.0 * b * h * w * c * nd,
                               'cuda_core_kernel_us': us_cc,
                               'note': 'what the DispNet engine launches: the band of L R^T on mma.sync tiles (fp16 hi/lo, 3 MMAs per '
                                       'product, csrc/corr_mma.cu); 15 FLOP/B, HBM-equivalent figure'}
    return out


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference path restated on host cores (oracle port)
# ---------------------------------------------------------------------------------------------------
def cpu_fps(cfg, steps, warmup):
    import torch
    cores = usable_cores()
    torch.set_num_threads(cores)
    (lf, rf, _, _), = make_inputs(cfg, 1, 1, 0)
    if cfg['net'] == 'Dispnet':
        from oracle.dispnet import DispNetAdapter, init_params
        ad = DispNetAdapter(init_params(seed=7), mode=cfg['mode'], lr=1e-4)
        run = lambda k: ad.step(lf, rf)
    else:
        from oracle.adaptation import OracleAdapter
        from oracle.madnet import MadNetOracle, init_params
        if cfg['mode'] == 'NONE':
            net = MadNetOracle(init_params(seed=42))
            def run(k):
                with torch.no_grad():
                    net.forward(lf, rf)
        else:
            ad = OracleAdapter(init_params(seed=42), mode=cfg['mode'], lr=1e-4)
            run = lambda k: ad.step(lf, rf, k % 5 if cfg['mode'] == 'MAD' else None)
    k = 0
    for _ in range(warmup):
        run(k); k += 1
    t0 = time.perf_counter()
    for _ in range(steps):
        run(k); k += 1
    dt = time.perf_counter() - t0
    return steps / dt, dt / steps * 1e3, cores


def run_reference(args, cfg):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    heavy = cfg['H'] * cfg['W'] > 1280 * 384 or cfg['net'] == 'Dispnet'
    steps, warmup = max(1, min(args.steps, 3 if heavy else 6)), max(1, min(args.warmup, 1 if heavy else 2))
    fps, ms, cores = cpu_fps(cfg, steps, warmup)
    sample = ('%d steps of the same workload (one %dx%d pair per step, modules in SEQUENTIAL order) after %d warm-up, torch-CPU '
              'fp32 oracle restatement of the TF1 graph (TF1 itself cannot run here)' % (steps, cfg['W'], cfg['H'], warmup))
    line = {'impl': 'reference', 'metric': cfg['metric'], 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus,
            'steps': steps, 'warmup': warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': cfg['workload'] % 1, 'arm': 'reference path on the host cores (oracle port; TF1 cannot run here), '
                                                              'one frame stream whatever N'},
            'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------
# this framework
# ---------------------------------------------------------------------------------------------------
DUMP_MAX_ELEMS = 4 << 20         # per array: at most 16 MB of float32, so a dump stays far below 64 MB


def dump_outputs(dirname, step, disp, weights):
    """What the last timed step handed its caller, one .npy per array, so that two builds can be compared output for
    output: loss.npy and train_loss.npy (float64 [1]), blocks.npy (the MAD modules it trained, float64), disparity.npy
    (the full-resolution disparity [B,H,W,1], float32) and weights.npy (the adapted weights, the engine's flat float32
    parameter arena).  An array above DUMP_MAX_ELEMS is replaced by a fixed seeded sample of that many elements
    (flattened, ascending index), the same for every run with the same arguments."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)

    def put(name, a):
        if a.size > DUMP_MAX_ELEMS:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        np.save(os.path.join(dirname, name + '.npy'), a)

    put('loss', np.array([step['loss']], dtype=np.float64))
    put('train_loss', np.array([step['train_loss']], dtype=np.float64))
    put('blocks', np.array(step['blocks'], dtype=np.float64))
    put('disparity', disp.detach().float().cpu().numpy())
    put('weights', weights.detach().float().cpu().numpy())


def parity_check(cfg, net, ad, eng, frame):
    """Engine forward on the first frame vs the CPU oracle with the SAME weights; returns the worst relative L-inf over
    the disparity outputs.  Checker only (outside every timed region)."""
    import numpy as np
    import torch
    lf, rf = frame[0][:1], frame[1][:1]
    params = eng.export_params()
    nd = len(net.get_disparities())
    eng.set_input(torch.from_numpy(frame[0]).to(eng.device), torch.from_numpy(frame[1]).to(eng.device))
    eng.run(0, 0, (1 << nd) - 1, 0)
    torch.cuda.synchronize()
    got = [d.numpy()[:1] for d in net.get_disparities()]
    torch.set_num_threads(usable_cores())
    with torch.no_grad():
        if cfg['net'] == 'Dispnet':
            from oracle.dispnet import DispNetOracle
            ref, _ = DispNetOracle(params).forward(lf, rf)
        else:
            from oracle.madnet import MadNetOracle
            ref, _ = MadNetOracle(params).forward(lf, rf)
    worst = 0.0
    for g, r in zip(got, ref):
        r = r.numpy()
        worst = max(worst, float(np.abs(g - r).max() / max(np.abs(r).max(), 1e-30)))
    return worst


def run_ours(args, cfg):
    import numpy as np
    import torch
    import torch.distributed as dist
    import Nets
    from madstereo.adaptation import OnlineAdaptation
    from madstereo.synthetic import init_params

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    # keep fd 1 clean for the single JSON line: NCCL / the banner of the reference-style constructors print to stdout
    sys.stdout.flush()
    saved_stdout_fd = os.dup(1)
    os.dup2(2, 1)
    if world != args.gpus and world > 1:
        raise SystemExit('--gpus %d but WORLD_SIZE=%d' % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    dev = torch.device('cuda', local)
    H, W, B = cfg['H'], cfg['W'], args.batch
    mode = cfg['mode']

    n_sets = 4 if B * H * W <= 4 * 384 * 1280 else 2
    sets = make_inputs(cfg, B, n_sets, rank)
    dev_pairs = [(torch.from_numpy(s[0]).to(dev), torch.from_numpy(s[1]).to(dev)) for s in sets]
    host_pairs = [(torch.from_numpy(s[2]).pin_memory(), torch.from_numpy(s[3]).pin_memory()) for s in sets]

    sys.stdout, real_stdout = sys.stderr, sys.stdout        # keep the reference-style banner off stdout
    if cfg['net'] == 'MADNet':
        net = Nets.get_stereo_net('MADNet', dict(left_img=dev_pairs[0][0], right_img=dev_pairs[0][1], split_layers=[None],
                                                 sequence=True, train_portion='BEGIN', bulkhead=(mode == 'MAD'), warping=True,
                                                 context_net=True, radius_d=2, stride=1, is_training=False))
        tcfg = json.load(open(os.path.join(PKG, 'block_config', 'MadNet_full.json')))
        ad = OnlineAdaptation(net, mode=mode, train_config=tcfg if mode == 'MAD' else None, lr=1e-4,
                              sample_mode='SEQUENTIAL', num_blocks=1)
    else:
        net = Nets.get_stereo_net('Dispnet', dict(left_img=dev_pairs[0][0], right_img=dev_pairs[0][1], split_layers=[None],
                                                  sequence=True, train_portion='BEGIN', bulkhead=False, correlation=True))
        ad = OnlineAdaptation(net, mode=mode, lr=1e-4)
    ad.load_weights(init_params(net.engine.layers, seed=42))
    sys.stdout = real_stdout
    eng = net.engine
    nd = len(net.get_disparities())

    parity = None
    if rank == 0 and not args.no_parity_check:
        err = parity_check(cfg, net, ad, eng, sets[0])
        parity = {'disp_rel_linf_vs_oracle': err, 'bar': 1e-3, 'frame': 'first synthetic pair, all %d disparity outputs' % nd}
        if not err < 1e-3:
            raise SystemExit('parity check failed before timing: disparity rel L-inf %.3e >= 1e-3' % err)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    disp_host = torch.empty(B, H, W, 1, dtype=torch.float32).pin_memory()
    full_disp = net.get_disparities()[-1]
    last = {}

    def timed(src, steps, warmup, pipelined=False, fetch_disp=False):
        # pipelined: the host->device copy of frame i+1 is issued (side stream) while frame i computes; every frame's
        # copy is still inside the timed region
        def one(i):
            last['step'] = ad.step(*src[i % n_sets], prefetch=src[(i + 1) % n_sets] if pipelined else None)
            if fetch_disp:
                disp_host.copy_(full_disp.tensor(), non_blocking=True)
        for i in range(warmup):
            one(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = eng.launch_count()
        e0.record()
        for i in range(steps):
            one(warmup + i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = eng.launch_count() - l0
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches

    clk = ClockSampler(local) if rank == 0 else None
    if clk:
        clk.start()
    ms_dev, launches = timed(dev_pairs, args.steps, args.warmup)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last['step'], full_disp.tensor(), eng.weights)
    ms_e2e_serial, _ = timed(host_pairs, args.steps, 3)
    ms_e2e, _ = timed(host_pairs, args.steps, 3, pipelined=True)
    ms_e2e_disp, _ = timed(host_pairs, args.steps, 3, pipelined=True, fetch_disp=True)
    if clk:
        clk.stop_flag = True
        clk.join(timeout=2)

    # ---- kernel-level profile: the SAME graph replays with event-record nodes around every kernel group inside the graph
    n_prof = 10
    eng.profile(2)                            # every rank takes part: the DP step contains the peer exchange
    for i in range(2):                        # graph capture of the instrumented variants (untimed)
        for k in range(5 if mode == 'MAD' else 1):
            ad.step(*dev_pairs[0])
    torch.cuda.synchronize()
    eng.profile(2)                            # reset the accumulators, keep the instrumented graphs
    t0 = time.perf_counter()
    for i in range(n_prof):
        ad.step(*dev_pairs[i % n_sets])
    torch.cuda.synchronize()
    prof_wall_ms = (time.perf_counter() - t0) * 1e3 / n_prof
    prof = eng.profile_read()
    layers = eng.profile_layers()
    eng.profile(0)
    barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    pk = peaks()
    frames = world * B * args.steps
    fps = frames / (ms_dev / 1e3)
    conv_ms = sum(prof[c]['ms'] for c in ('conv_fwd', 'conv_dgrad', 'conv_wgrad'))
    conv_macs = sum(prof[c]['macs'] for c in ('conv_fwd', 'conv_dgrad', 'conv_wgrad'))
    conv_calls = sum(prof[c]['calls'] for c in ('conv_fwd', 'conv_dgrad', 'conv_wgrad'))
    conv_tflops = 2.0 * conv_macs / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
    prof_total = sum(v['ms'] for v in prof.values())
    # the single layer shape that dominates the step (128 -> 128 3x3 at H/4 x W/4: estimator-2 disp2, context 2-3)
    dom = None
    dom_name = 'fgc-volume-filtering-2/disp2' if cfg['net'] == 'MADNet' else 'conv3/1'
    if dom_name in layers and 'fwd' in layers[dom_name]:
        li = eng.layer_by_name[dom_name]
        hh, ww = (H + 63) // 64 * 64 // (4 if cfg['net'] == 'MADNet' else 8), W // (4 if cfg['net'] == 'MADNet' else 8)
        macs = B * hh * ww * li.kh * li.kw * li.cin * li.cout
        dom = {'layer': dom_name, 'shape': '%d->%d %dx%d @%dx%d' % (li.cin, li.cout, li.kh, li.kw, hh, ww)}
        for d, v in layers[dom_name].items():
            us = v['ms'] / v['calls'] * 1e3
            dom[d] = {'us': us, 'useful_tflops': 2.0 * macs / us / 1e6, 'frac_of_bf16_peak': 2.0 * macs / us / 1e6 / pk['bf16_tflops'],
                      'tensor_flops_frac': 3.0 * 2.0 * macs / us / 1e6 / pk['bf16_tflops']}
        dom['note'] = ('in-graph CUDA-event time of that layer inside the replayed step graph; split-bf16 (3 kind::f16 MMAs per '
                       'product): tensor_flops_frac counts the 3 issued MMAs against the measured bf16 peak')
    if os.environ.get('MS_BENCH_LAYERS'):       # per-layer in-graph times (diagnosis; not part of the JSON line)
        try:
            os.makedirs(os.path.join(ROOT, 'gpurun_out'), exist_ok=True)
            with open(os.path.join(ROOT, 'gpurun_out', 'layers_cfg%d.json' % args.config), 'w') as f:
                json.dump({k: {d: {'us_per_call': v['ms'] / v['calls'] * 1e3, 'calls_per_step': v['calls'] / n_prof}
                               for d, v in dv.items()} for k, dv in layers.items()}, f, indent=1)
        except OSError:
            pass
    corr_large = corr_large_shapes(dev) if not args.no_corr_shapes else {}
    line = {
        'metric': cfg['metric'], 'value': fps, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': cfg['workload'] % B, 'baseline_config': args.config,
                   'parallelism': 'dp%d' % world, 'global_batch': world * B,
                   'l2': 'no flush: per-step activation+gradient working set ~0.7 GB >> %d MB L2; inputs rotate over '
                         '%d distinct frame sets' % (L2_MB, n_sets),
                   'step': 'set_input, forward, full-res loss, train-op loss+backward, gradient exchange over NVLink peer memory '
                           'fused with the momentum update (N>1), loss D2H (host reward policy needs it every frame)',
                   'arithmetic': 'fp32 storage; convolutions as split-bf16 (hi+lo) tcgen05 MMAs with fp32 accumulation '
                                 '(~2^-16 relative product error), everything else fp32'},
        'parity': parity,
        'e2e': {'value': frames / (ms_e2e / 1e3), 'unit': 'frames/s', 'h2d_bytes_per_step': 2 * B * H * W * 3, 'd2h_bytes_per_step': 16,
                'mode': 'uint8 frames in pinned host memory (what the reference decodes), H2D of frame i+1 on a side stream while '
                        'frame i computes (OnlineAdaptation.step(prefetch=...)), fp32 conversion on the device, loss scalars D2H',
                'serial_value': frames / (ms_e2e_serial / 1e3),
                'with_disparity_d2h': {'value': frames / (ms_e2e_disp / 1e3), 'd2h_bytes_per_step': 16 + B * H * W * 4,
                                       'note': 'also copies the full-resolution disparity map to pinned host memory every frame'}},
        'gpu_launches': int(launches),
        'roofline': {'bound': 'tensor',
                     'kernel': 'conv stack: conv_bf_kernel (split-bf16 tcgen05 implicit GEMM: forward + dgrad, stride 1/2, dilated) + '
                               'wgrad_bf_kernel (tcgen05 weight/bias gradients) + the direct kernels of the 3-channel / 1-channel layers; '
                               'useful FLOPs = 2*MACs (the 3 MMAs per product are not counted)',
                     'achieved': conv_tflops, 'peak': pk['bf16_tflops_sustained'], 'unit': 'TFLOP/s',
                     'frac': conv_tflops / pk['bf16_tflops_sustained'],
                     'frac_issued_mmas': 3.0 * conv_tflops / pk['bf16_tflops_sustained'],
                     'frac_note': 'frac counts useful FLOPs; the fp32-class arithmetic issues three 16-bit MMAs per product (frac_issued_mmas, an '
                                  'upper bound: the direct CUDA-core layers of the stack issue none)',
                     'peak_src': pk['src'] + ' bf16 sustained (kernels timed inside a long step)',
                     'timing': 'CUDA event-record nodes around every conv launch group INSIDE the replayed step graph '
                               '(ms_engine_profile(2)), %d steps' % n_prof,
                     'traffic': 16399616 if (args.config in (2, 3) and B == 1) else None,
                     'traffic_src': 'dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel (conv_bf_kernel, 128->128 3x3 '
                                    '@96x320 forward) from ncu --set full, profiles/r2_final_ncu_conv_bf_128x128_96x320.txt (16.394 MB read + 5.6 KB written); algorithmic: 15.7 MB of fp16 '
                                    'planes + 0.6 MB of weight tiles read, the 31 MB it writes stay in L2',
                     'avg_launch_us': 1e3 * conv_ms / max(conv_calls, 1),
                     'share_of_step': conv_ms / prof_total if prof_total else None,
                     'dominant_layer': dom},
        'profile_ms_per_step': dict({k: v['ms'] / n_prof for k, v in prof.items()},
                                    sum=prof_total / n_prof, instrumented_step_wall_ms=prof_wall_ms,
                                    event_node_overhead_us_subtracted_per_span=eng.profile_event_overhead_us()),
        'clocks': clk.summary() if clk else None,
    }
    if cfg['net'] == 'MADNet':
        cf, cb = prof['corr_fwd'], prof['corr_bwd']
        line['corr_kernel'] = {
            'bound': 'hbm', 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
            'in_step_fwd': {'achieved': cf['bytes'] / (cf['ms'] / 1e3) / 1e9 if cf['ms'] > 0 else 0.0,
                            'note': 'all 5 levels at this resolution (<= 8.5 MB each at 1280x384: L2-resident, launch-latency bound); '
                                    'fused-concat variant, bytes B*h*w*(3C+nd+1)*4'},
            'in_step_bwd': {'achieved': cb['bytes'] / (cb['ms'] / 1e3) / 1e9 if cb['ms'] > 0 else 0.0},
            'large': {k: dict(v, frac=v['gbs'] / pk['hbm_gbs']) for k, v in corr_large.items()}}
        big = corr_large.get('madnet_L2_1920x1088_B8_fused_concat')
        if big:
            line['corr_kernel'].update({'achieved': big['gbs'], 'frac': big['gbs'] / pk['hbm_gbs'],
                                        'shape': 'madnet_L2_1920x1088_B8_fused_concat (the variant the engine launches)'})
    if world == 1 and not args.no_cpu_baseline:
        heavy = H * W > 1280 * 384 or cfg['net'] == 'Dispnet'
        fps_cpu, ms_cpu, cores = cpu_fps(cfg, 2 if heavy else 3, 1)
        line['cpu_baseline'] = {'value': fps_cpu, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                                'sample': '%d steps of the same workload on one %dx%d pair after 1 warm-up; torch-CPU fp32 oracle '
                                          'restatement (TF1 cannot run here)' % (2 if heavy else 3, W, H)}
    sys.stdout.flush()
    os.dup2(saved_stdout_fd, 1)
    print(json.dumps(line), flush=True)
    os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument('--batch', type=int, default=1, help='frames per GPU per step (config 5: 8 = "batch 8" on one GPU)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-parity-check', action='store_true')
    ap.add_argument('--no-corr-shapes', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed as DIR/<name>.npy (rank 0; see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    cfg = CONFIGS[args.config]
    if args.impl == 'reference':
        return run_reference(args, cfg)
    return run_ours(args, cfg)


if __name__ == '__main__':
    sys.exit(main())
