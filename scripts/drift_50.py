"""VERDICT item 3: the arithmetic schemes end to end over 50 MAD adaptation steps at 1280x384 (SEQUENTIAL sampler, 4
alternating synthetic pairs): disparity error of the last frame and drift of the adapted weights against the fp64 oracle,
next to the fp32 oracle's own drift (the trajectory is chaotic at the kinks: the fp32 oracle is the yardstick).
  python scripts/drift_50.py [steps]   -> gpurun_out/drift_50.json
"""
import json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'real-time-self-adaptive-deep-stereo_b200')
sys.path.insert(0, ROOT); sys.path.insert(0, PKG)
import numpy as np, torch

STEPS = int(sys.argv[1]) if len(sys.argv) > 1 else 50
H, W = 384, 1280


def rel_l2(a, b):
    a = np.asarray(a, np.float64).ravel(); b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def rel_linf(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def main():
    from madstereo.synthetic import make_pair
    from oracle.adaptation import OracleAdapter
    from oracle.madnet import init_params
    frames = [make_pair(H, W, seed=40 + i)[:2] for i in range(4)]
    params = init_params(seed=42)
    torch.set_num_threads(min(32, len(os.sched_getaffinity(0))))
    out = {'steps': STEPS, 'resolution': [H, W]}
    runs = {}
    for name, dt in (('oracle_fp64', torch.float64), ('oracle_fp32', torch.float32)):
        t0 = time.time()
        ad = OracleAdapter(params, mode='MAD', lr=1e-4, dtype=dt)
        losses = []
        for t in range(STEPS):
            l, r = frames[t % 4]
            res = ad.step(l, r, t % 5)
            losses.append(res['full_loss'])
        runs[name] = {'w': {k: v.detach().numpy().astype(np.float64) for k, v in ad.net.p.items()}, 'loss': losses,
                      'disp': res['disparities'][-1]}
        print(name, 'done in %.1f s' % (time.time() - t0), flush=True)
    import Nets
    from madstereo.adaptation import OnlineAdaptation
    cfg = json.load(open(os.path.join(PKG, 'block_config', 'MadNet_full.json')))
    name = 'gpu_fp16x3_fwd_bf16x3_bwd (shipped)'
    l0 = torch.from_numpy(frames[0][0]).cuda(); r0 = torch.from_numpy(frames[0][1]).cuda()
    sys.stdout, real = sys.stderr, sys.stdout
    net = Nets.get_stereo_net('MADNet', dict(left_img=l0, right_img=r0, split_layers=[None], sequence=True, train_portion='BEGIN',
                                             bulkhead=True, warping=True, context_net=True, radius_d=2, stride=1, is_training=False))
    ad = OnlineAdaptation(net, mode='MAD', train_config=cfg, lr=1e-4, sample_mode='SEQUENTIAL', num_blocks=1, ssim_th=10.0)
    sys.stdout = real
    ad.load_weights(params)
    losses = []
    for t in range(STEPS):
        l, r = frames[t % 4]
        o = ad.step(torch.from_numpy(l).cuda(), torch.from_numpy(r).cuda(), want_disp_mask=0b100000)
        losses.append(o['loss'])
    runs[name] = {'w': {k: v.astype(np.float64) for k, v in net.engine.export_params().items()}, 'loss': losses,
                  'disp': net.get_disparities()[-1].numpy()}
    ref = runs['oracle_fp64']
    table = {}
    for name, r in runs.items():
        if name == 'oracle_fp64':
            continue
        dw = {k: rel_l2(r['w'][k] - params[k], ref['w'][k] - params[k]) for k in ref['w']}
        tot = rel_l2(np.concatenate([(r['w'][k] - params[k]).ravel() for k in ref['w']]), np.concatenate([(ref['w'][k] - params[k]).ravel() for k in ref['w']]))
        table[name] = {'disp_rel_linf_last_frame': rel_linf(r['disp'], ref['disp']),
                       'dw_rel_l2_all_weights': tot, 'dw_rel_l2_worst_tensor': max(dw.values()),
                       'loss_abs_diff_last_step': abs(r['loss'][-1] - ref['loss'][-1]),
                       'loss_abs_diff_max_over_steps': float(np.abs(np.array(r['loss']) - np.array(ref['loss'])).max())}
        print(name, json.dumps(table[name]), flush=True)
    out['vs_oracle_fp64'] = table
    os.makedirs(os.path.join(ROOT, 'gpurun_out'), exist_ok=True)
    json.dump(out, open(os.path.join(ROOT, 'gpurun_out', 'drift_50.json'), 'w'), indent=1)


if __name__ == '__main__':
    main()
