"""Golden vectors of the reference's own code for checks in tests/test_reference_golden_cpu.py and tests/test_abi_cpu.py, which
compare with these files and never read the reference tree.  Run where that tree is available (see make_reference_golden.REF):

    python tests/golden/make_reference_checks_golden.py     -> tests/golden/ref_calibrated_plumbing_seed*.npz,
                                                               ref_full_thinktwice.npz, ref_camera_geometry_*.npz,
                                                               ref_config_model.json

What is stored is what the reference computed, from the same seeded weights and inputs the tests rebuild:

  * the reference EncoderDecoder.forward_inference with the oracle's calibrated weights, plumbing shape, seeds 0-2
  * the same at the full thinktwice.py shape (4 cams x 2 sweeps 448x896, 40k points, K = 5, B = 1)
  * the reference LSS geometry: frustum (as its three axes), voxel grid, get_geometry at a seeded sample of frustum positions, and the
    camera-awareness vector its DepthNet feeds to BatchNorm1d(22)
  * the model section of the reference's configs/thinktwice.py
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_reference_golden as mg  # noqa: E402  (puts the repository root on sys.path)

CALIBRATED_KEYS = ('pred_wp', 'mu_branches', 'sigma_branches', 'future_mu', 'future_sigma', 'pred_speed', 'pred_value_traj',
                   'refine_flattned_BEV_feature')
GEOMETRY_SAMPLES = 512                                             # frustum positions kept per camera
# CPU kernels split their reductions by thread count, which moves the full-shape forward by ~2e-6: the fixture and the test
# run it with this many threads, so that the test's 1e-6 bound compares the two implementations and not two thread splits
FULL_SHAPE_THREADS = 4


class fixed_threads:
    def __init__(self, n):
        self.n = n

    def __enter__(self):
        self.prev = torch.get_num_threads()
        torch.set_num_threads(self.n)

    def __exit__(self, *exc):
        torch.set_num_threads(self.prev)


def norm_config(x):
    """config values as JSON-comparable plain data (tuples and lists alike)."""
    if isinstance(x, dict):
        return {k: norm_config(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [norm_config(v) for v in x]
    return x


def pred_digest(pred):
    """what the fixture keeps of a forward_inference output: small tensors whole, refine_BEV_feature (B, K+1, 256, H, W)
    as its spatial means plus a strided sub-grid of every 4th channel."""
    out = {k: pred[k] for k in mg.PRED_KEYS if k != 'refine_BEV_feature'}
    f = pred['refine_BEV_feature']
    out['refine_BEV_feature.mean_hw'] = f.mean((-2, -1))
    out['refine_BEV_feature.sub'] = f[:, :, ::4, ::5, ::5]
    return out


def geometry_sample_index(frustum_shape):
    """seeded flat indices into the (D, fH, fW) frustum grid."""
    n = int(np.prod(frustum_shape[:3]))
    return np.sort(np.random.default_rng(0).choice(n, size=min(GEOMETRY_SAMPLES, n), replace=False)).astype(np.int64)


def frustum_from_axes(u, v, d):
    """(D, fH, fW, 4) grid of (u, v, d, 1) points."""
    D, H, W = len(d), len(v), len(u)
    return torch.stack([u.view(1, 1, W).expand(D, H, W), v.view(1, H, 1).expand(D, H, W), d.view(D, 1, 1).expand(D, H, W),
                        torch.ones(D, H, W, dtype=u.dtype)], -1)


def reference_encoder_decoder(fw, regs, mc):
    from oracle.lidar import LidarNet
    lss = sys.modules['olt_code.model_code.backbones.lss']
    regs['BACKBONES'].classes['LSS'], regs['BACKBONES'].classes['LidarNet'] = lss.LSS, LidarNet
    return fw.EncoderDecoder(img_encoder=dict(mc['img_encoder']), decoder=dict(mc['decoder']), lidar_encoder=dict(mc['lidar_encoder']),
                             train_cfg=mc['train_cfg'], test_cfg=mc.get('test_cfg')).eval()


def calibrated_forward(fw, regs, config, seed, num_points):
    """the reference's forward_inference with the oracle's seeded, BN-calibrated weights (B = 1)."""
    from oracle.model import EncoderDecoder as Oracle, calibrate_bn, init_oracle_weights
    from thinktwice_b200.config import Config
    from thinktwice_b200.synthetic import make_batch
    mc = Config.fromfile(config).model
    o = Oracle(**{k: v for k, v in mc.items() if k != 'type'})
    init_oracle_weights(o, seed)
    batch = make_batch(Config.fromfile(config), 1, seed=seed, num_points=num_points)
    calibrate_bn(o, batch)
    ref = reference_encoder_decoder(fw, regs, mc)
    ref.load_state_dict(o.state_dict())                                # strict: identical names and shapes
    batch['target_command_raw'] = batch['target_command'].argmax(-1)
    with torch.no_grad():
        return ref.forward_inference(batch)


def camera_geometry(which):
    """the reference LSS on the inputs test_product_host_camera_geometry_equals_the_reference_lss builds."""
    from thinktwice_b200.config import Config, DEFAULT_CONFIG, PLUMBING_CONFIG
    from thinktwice_b200.registry import BACKBONES
    from thinktwice_b200.synthetic import make_batch
    lss = sys.modules['olt_code.model_code.backbones.lss']
    cfg = Config.fromfile(PLUMBING_CONFIG if which == 'plumbing' else DEFAULT_CONFIG)
    kw = {k: v for k, v in dict(cfg.model['img_encoder']).items() if k != 'type'}
    ref = lss.LSS(**kw).eval()
    prod = BACKBONES.build(dict(cfg.model['img_encoder']))
    B = 2
    batch = make_batch(cfg, B, seed=3, num_points=10)
    metas = batch['img_metas']
    N, T = batch['img'].shape[2], len(metas[0])
    mats = prod.build_mats(metas, N)
    fr = ref.frustum                                                   # (D, fH, fW, 4) = (u, v, d, 1): kept as its three axes
    u, v, d = fr[0, 0, :, 0], fr[0, :, 0, 1], fr[:, 0, 0, 2]
    assert torch.equal(fr, frustum_from_axes(u, v, d))
    idx = geometry_sample_index(tuple(fr.shape))
    out = {'frustum.u': u, 'frustum.v': v, 'frustum.d': d, 'lower': ref.voxel_coord - ref.voxel_size / 2.0,
           'voxel_size': ref.voxel_size, 'voxel_num': torch.as_tensor(ref.voxel_num), 'sample_index': torch.from_numpy(idx)}
    for s in range(T):
        k = -1 if s == 0 else -s                                       # the sweep index LSS.forward passes (lss.py:689, 712)
        g = ref.get_geometry(mats['sensor2ego_mats'][:, k], mats['intrin_mats'][:, k], mats['ida_mats'][:, k], None)
        out[f'geom_mats{k}'] = g.reshape(B, N, -1, 3)[:, :, idx]
    seen = {}
    h = ref.depth_net.bn.register_forward_pre_hook(lambda m, inp: seen.setdefault('x', inp[0].detach().clone()))
    with torch.no_grad():
        ref.depth_net(torch.zeros(B * N, kw['depth_net_conf']['in_channels'], 2, 2), dict(mats))
    h.remove()
    out['depthnet_bn_input'] = seen['x'].reshape(B * N, 22)
    return out


def save(name, arrays):
    np.savez_compressed(os.path.join(HERE, name), **{k: v.detach().cpu().numpy() for k, v in arrays.items()})
    print(f'{name}: {os.path.getsize(os.path.join(HERE, name))} bytes')


def main():
    from thinktwice_b200.config import Config, DEFAULT_CONFIG, PLUMBING_CONFIG
    fw, regs = mg.load_reference()
    mg.load_reference_lss(regs)
    cfg_path = os.path.join(os.path.dirname(mg.REF), 'configs', 'thinktwice.py')
    with open(os.path.join(HERE, 'ref_config_model.json'), 'w') as f:
        json.dump(norm_config(Config.fromfile(cfg_path).model), f, indent=1, sort_keys=True)
    for which in ('plumbing', 'full'):
        save(f'ref_camera_geometry_{which}.npz', camera_geometry(which))
    for seed in (0, 1, 2):
        pred = calibrated_forward(fw, regs, PLUMBING_CONFIG, seed, 2000)
        save(f'ref_calibrated_plumbing_seed{seed}.npz', {k: pred[k] for k in CALIBRATED_KEYS})
    with fixed_threads(FULL_SHAPE_THREADS):
        save('ref_full_thinktwice.npz', pred_digest(calibrated_forward(fw, regs, DEFAULT_CONFIG, 0, 40000)))


if __name__ == '__main__':
    main()
