"""Golden digest of the reference's own voxel-pooling kernel, for tests/test_ops_gpu.py.  Needs a GPU and the reference
kernel built by oracle/build_ref.py (oracle/_ref/libvoxel_pooling_ref.so):

    python tests/golden/make_voxel_pool_golden.py [OUT_DIR]      -> OUT_DIR/ref_voxel_pooling_kernel.npz (default tests/golden)

For every shape of test_voxel_pooling_dropin_matches_oracle_and_reference_kernel the kernel runs on the test's seeded inputs
and the fixture keeps, under the key 'BxPxCxXxY.':
  index / sample : a seeded sample of the non-zero entries of its (B, Y, X, C) output (flat indices and values)
  channel_sum    : the output summed over Y and X, float64 (B, C)
  memo_sha256    : SHA-256 of its int32 (B, P, 3) last-position memo, which the product must reproduce bit for bit
"""
import ctypes as C
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(HERE))
SYMBOL = '_Z37voxel_pooling_forward_kernel_launcheriiiiiiPKiPKfPfPiP11CUstream_st'
SHAPES = [(1, 5000, 64, 21, 21), (2, 20000, 256, 21, 21), (1, 30000, 80, 200, 200), (1, 100, 7, 5, 4)]
SAMPLES = 2048


def key(shape):
    return 'x'.join(str(v) for v in shape) + '.'


def inputs(shape):
    """the seeded (geom, feats) the test builds for `shape`."""
    from test_ops_gpu import _rand_geom
    B, P, Cc, X, Y = shape
    gen = torch.Generator().manual_seed(P)
    geom = _rand_geom(gen, B, P, X, Y)
    return geom, torch.randn(B, P, Cc, generator=gen)


def memo_digest(memo):
    return hashlib.sha256(memo.cpu().contiguous().numpy().tobytes()).hexdigest()


def main(out_dir):
    fn = getattr(C.CDLL(os.path.join(ROOT, 'oracle', '_ref', 'libvoxel_pooling_ref.so')), SYMBOL)
    out = {}
    for shape in SHAPES:
        B, P, Cc, X, Y = shape
        geom, feats = inputs(shape)
        g, f = geom.cuda().contiguous(), feats.cuda().contiguous()
        o = torch.zeros(B, Y, X, Cc, device='cuda')
        memo = -torch.ones(B, P, 3, dtype=torch.int32, device='cuda')
        fn(B, P, Cc, X, Y, 1, C.c_void_p(g.data_ptr()), C.c_void_p(f.data_ptr()), C.c_void_p(o.data_ptr()),
           C.c_void_p(memo.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        o = o.cpu()
        nz = np.flatnonzero(o.numpy())
        idx = np.sort(np.random.default_rng(0).choice(nz, size=min(SAMPLES, nz.size), replace=False))
        k = key(shape)
        out[k + 'index'] = idx.astype(np.int32)
        out[k + 'sample'] = o.flatten()[torch.from_numpy(idx)].numpy()
        out[k + 'channel_sum'] = o.double().sum((1, 2)).numpy()
        out[k + 'memo_sha256'] = np.array(memo_digest(memo))
        print(k, f'{nz.size} non-zero of {o.numel()}', out[k + 'memo_sha256'])
    os.makedirs(out_dir, exist_ok=True)
    np.savez_compressed(os.path.join(out_dir, 'ref_voxel_pooling_kernel.npz'), **out)


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else HERE)
