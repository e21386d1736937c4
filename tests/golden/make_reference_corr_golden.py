"""Golden vectors and timings of the REFERENCE's own CUDA correlation kernel (CorrelateData of Nets/Native/shift_corr.cu.cc,
compiled unmodified for sm_100a into oracle/_ref/libref_shift_corr.so by oracle/build_ref.sh).

Needs a GPU and oracle/_ref; writes tests/golden/reference_corr_native.npz (or the path given), which
tests/test_ops_gpu.py compares against, so the tests themselves never need the reference build:
  exact_x, exact_y, exact_out  the inputs and the full NHWC output of one small padded-input case
  <shape>_seed                 seed of the inputs of a timing shape (corr_inputs below; the test regenerates them)
  <shape>_x_probe              the first 16 values of x, to prove the regenerated inputs are the same
  <shape>_index, _sample       a seeded sample of the flattened NHWC reference output, and its values
  <shape>_absmax               max |output| over the whole output (denominator of the relative error)
  <shape>_reference_us         median kernel time over 7 launches, L2 flushed between launches
  device                       GPU name and power limit the timings were taken at

    python tests/golden/make_reference_corr_golden.py [out.npz]
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'reference_corr_native.npz')

EXACT = (2, 9, 33, 64, 2)             # b, h, w, c, max_disp
TIMED = {'madnet_L6_1280x384': (1, 6, 20, 192, 2), 'madnet_L5': (1, 12, 40, 128, 2), 'madnet_L4': (1, 24, 80, 96, 2),
         'madnet_L3': (1, 48, 160, 64, 2), 'madnet_L2': (1, 96, 320, 32, 2), 'madnet_L2_1920x1088_B8': (8, 272, 480, 32, 2),
         'dispnet_1280x384': (1, 96, 320, 128, 40)}
N_SAMPLE = 4096


def corr_inputs(b, h, w, c, seed):
    """Same generator as tests/test_ops_gpu.py: seeded on the host, so every GPU sees the same inputs."""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(b, h, w, c, generator=g), torch.randn(b, h, w, c, generator=g)


def sample_index(n, seed):
    return np.sort(np.random.default_rng(seed).choice(n, size=min(n, N_SAMPLE), replace=False))


def main(out_path):
    ref = ctypes.CDLL(os.path.join(ROOT, 'oracle', '_ref', 'libref_shift_corr.so'))
    ref.ref_shift_corr.argtypes = [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 5 + [ctypes.c_void_p]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')

    def run_ref(x, y, d):
        b, h, w, c = x.shape
        xp = torch.nn.functional.pad(x, (0, 0, d, d)).contiguous()
        yp = torch.nn.functional.pad(y, (0, 0, d, d)).contiguous()
        out_nchw = torch.zeros(b, 2 * d + 1, h, w, device='cuda')
        launch = lambda: ref.ref_shift_corr(xp.data_ptr(), yp.data_ptr(), d, b, h, w + 2 * d, c, out_nchw.data_ptr())
        torch.cuda.synchronize()
        assert launch() == 0
        torch.cuda.synchronize()
        return out_nchw, launch

    def timeit(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(7):
            flush.zero_()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        ts.sort()
        return ts[len(ts) // 2]

    out = {}
    b, h, w, c, d = EXACT
    rng = np.random.default_rng(5)
    x = rng.standard_normal((b, h, w, c)).astype(np.float32)
    y = rng.standard_normal((b, h, w, c)).astype(np.float32)
    o, _ = run_ref(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), d)
    out.update(exact_x=x, exact_y=y, exact_out=o.permute(0, 2, 3, 1).cpu().numpy())

    # the reference launches on the legacy default stream: make torch's stream the default one for its timing
    with torch.cuda.stream(torch.cuda.default_stream()):
        for seed, (name, (b, h, w, c, d)) in enumerate(TIMED.items()):
            x, y = corr_inputs(b, h, w, c, seed)
            o, launch = run_ref(x.cuda(), y.cuda(), d)
            flat = o.permute(0, 2, 3, 1).contiguous().view(-1)
            idx = sample_index(flat.numel(), seed)
            out[name + '_seed'] = np.int64(seed)
            out[name + '_x_probe'] = x.view(-1)[:16].numpy()
            out[name + '_index'] = idx
            out[name + '_sample'] = flat[torch.from_numpy(idx).cuda()].cpu().numpy()
            out[name + '_absmax'] = np.float64(flat.abs().max().item())
            out[name + '_reference_us'] = np.float64(timeit(launch))
            print('%-24s reference %9.2f us' % (name, out[name + '_reference_us']))
    smi = subprocess.run(['nvidia-smi', '-i', str(torch.cuda.current_device()), '--query-gpu=name,power.limit',
                          '--format=csv,noheader'], capture_output=True, text=True).stdout.strip()
    out['device'] = np.array(smi or torch.cuda.get_device_name())
    print(out['device'])
    np.savez_compressed(out_path, **out)
    print('wrote', out_path)


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else OUT)
