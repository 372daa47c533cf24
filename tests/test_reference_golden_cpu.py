"""The oracle (and the product's host-side action / PID code) against vectors produced by the REFERENCE'S OWN Python
(tests/golden/make_reference_golden.py: encoder_decoder_framework.py, thinktwice_decoder.py, multi_scale_deformable_attn_function.py,
dense_heads/utils.py, code/utils.py loaded unmodified behind import stubs).  Weights are regenerated from a name-keyed
generator, so the test also pins the state_dict names and shapes the reference exposes for fusion + decoder (607 tensors)."""
import os
import sys

import numpy as np
import pytest
import torch

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
sys.path.insert(0, G)


def rel(a, b):
    return float(np.abs(np.asarray(a) - b).max() / (np.abs(b).max() + 1e-12))


def _oracle_with_named_weights(cfg, seed):
    from make_reference_golden import named_init
    from oracle.model import EncoderDecoder as Oracle
    o = Oracle(**{k: v for k, v in cfg.model.items() if k != 'type'}).eval()
    sub = {k: v for k, v in o.state_dict().items() if not k.startswith(('img_encoder.', 'lidar_encoder.'))}

    class Shared:                                                      # the part of the model the fixture covers
        def state_dict(self):
            return sub

        def load_state_dict(self, d):
            o.load_state_dict(d, strict=False)
    named_init(Shared(), seed)
    return o, sub


@pytest.mark.parametrize('seed', [0, 1, 2])
def test_oracle_fusion_and_decoder_equal_the_reference_code(seed):
    from make_reference_golden import synthetic_inputs
    from thinktwice_b200.config import Config, DEFAULT_CONFIG
    cfg = Config.fromfile(DEFAULT_CONFIG)
    f = np.load(os.path.join(G, f'ref_fusion_decoder_seed{seed}.npz'))
    o, sub = _oracle_with_named_weights(cfg, seed)
    # structure: same parameter / buffer names and shapes as the reference modules
    assert sorted(sub) == list(f['names'])
    assert [str(tuple(sub[n].shape)) for n in f['names']] == list(f['shapes'])
    x = synthetic_inputs(cfg, seed, int(f['batch']))
    with torch.no_grad():
        state = torch.cat([x['speed'].float().view(-1, 1) / 12., x['target_point'].float(), x['target_command']], -1)
        meas = o.measurements_encoder(state)
        flat, bev32, mid, lidar_hi = o.get_fusion_feat(x['cam_bev'], x['lidar'])
        pred = o.decoder(flat, bev32, meas, o, [x['lidar2img'], x['ida_mat'], x['fpn'], lidar_hi], False, None)
    got = {'meas': meas, 'flat': flat, 'bev32': bev32, 'mid10': mid[3], 'mid4': mid[4], 'mid2': mid[5]}
    for k in ('pred_wp', 'mu_branches', 'sigma_branches', 'future_mu', 'future_sigma', 'pred_speed', 'pred_value_traj', 'pred_value_ctrl',
              'refine_flattned_BEV_feature', 'refine_BEV_feature'):
        got['pred.' + k] = pred[k]
    got['pred.refine_future_BEV_feature.mean_hw'] = pred['refine_future_BEV_feature'].mean((-2, -1))
    for k, v in got.items():
        assert rel(v.numpy(), f[k]) < 1e-6, k                          # same torch ops in the same order: expected exact


@pytest.mark.parametrize('seed', [0, 1, 2])
def test_product_host_action_and_pid_equal_the_reference_code(seed):
    """process_action / control_pid / PIDController of the product model (host numpy code, no GPU) on the reference's pred."""
    from make_reference_golden import synthetic_inputs
    from thinktwice_b200.config import Config, DEFAULT_CONFIG
    from thinktwice_b200.registry import build_model
    cfg = Config.fromfile(DEFAULT_CONFIG)
    f = np.load(os.path.join(G, f'ref_fusion_decoder_seed{seed}.npz'))
    x = synthetic_inputs(cfg, seed, int(f['batch']))
    m = build_model(cfg.model)
    pred = {k: torch.from_numpy(f['pred.' + k][:1]) for k in ('pred_wp', 'mu_branches', 'sigma_branches')}
    tp = x['target_point'][0].numpy()
    steer, throttle, brake, _ = m.process_action(pred, 3, x['speed'][:1], tp)
    assert np.allclose([steer, throttle, brake], f['action'], rtol=0, atol=1e-12)
    s2, t2, b2, meta = m.control_pid(pred['pred_wp'][:, -1], x['speed'][:1], tp)
    got = [float(s2), float(t2), float(b2)] + [meta[k] for k in ('desired_speed', 'angle', 'angle_last', 'angle_target', 'angle_final', 'delta')]
    assert np.allclose(got, f['pid'], rtol=0, atol=1e-12)


@pytest.mark.parametrize('seed', [0, 1])
def test_oracle_camera_encoder_equals_the_reference_lss(seed):
    """oracle.camera.LSS vs the reference's model_code/backbones/lss.py (DepthNet, ASPP, UNet, seg->feature, PAFPN forward,
    frustum / geometry with its quirks, lift, sweep handling) at the plumbing shape; B = 2 in seed 1."""
    from make_reference_golden import lss_digest, named_init
    from oracle.camera import LSS
    from thinktwice_b200.config import Config, PLUMBING_CONFIG
    from thinktwice_b200.synthetic import make_batch
    cfg = Config.fromfile(PLUMBING_CONFIG)
    f = np.load(os.path.join(G, f'ref_lss_plumbing_seed{seed}.npz'))
    o = LSS(**{k: v for k, v in dict(cfg.model['img_encoder']).items() if k != 'type'}).eval()
    sd = o.state_dict()
    assert sorted(sd) == list(f['names'])                              # same parameter / buffer names as the reference module
    assert [str(tuple(sd[n].shape)) for n in f['names']] == list(f['shapes'])
    named_init(o, seed, prefix='img_encoder.')
    batch = make_batch(cfg, int(f['batch']), seed=seed, num_points=10)
    with torch.no_grad():
        keep = {}
        out = o(batch['img'], batch['img_metas'], keep)
    out = dict(out)
    out.setdefault('depth', keep.get('depth'))
    got = lss_digest(out)
    for k, v in got.items():
        assert rel(v.numpy(), f[k]) < 2e-5, k                          # index_add order / conv algorithm choice: not bitwise


@pytest.mark.parametrize('seed', [0, 1])
def test_oracle_forward_inference_equals_the_reference_end_to_end(seed):
    """EncoderDecoder.forward_inference at the plumbing shape: reference framework + reference LSS + reference decoder (the LiDAR
    encoder, third-party glue, is oracle.lidar.LidarNet on both sides) vs the oracle, name-keyed weights; B = 2 in seed 1."""
    from make_reference_golden import PRED_KEYS, named_init
    from oracle.model import EncoderDecoder as Oracle
    from thinktwice_b200.config import Config, PLUMBING_CONFIG
    from thinktwice_b200.synthetic import make_batch
    cfg = Config.fromfile(PLUMBING_CONFIG)
    f = np.load(os.path.join(G, f'ref_e2e_plumbing_seed{seed}.npz'))
    o = Oracle(**{k: v for k, v in cfg.model.items() if k != 'type'}).eval()
    sd = o.state_dict()
    assert sorted(sd) == list(f['names'])                              # the full model: names and shapes as the reference builds them
    assert [str(tuple(sd[n].shape)) for n in f['names']] == list(f['shapes'])
    named_init(o, seed)
    batch = make_batch(cfg, int(f['batch']), seed=seed, num_points=1500)
    with torch.no_grad():
        pred = o.forward_inference(batch)
    for k in PRED_KEYS:
        assert rel(pred[k].numpy(), f[k]) < 1e-5, k


@pytest.mark.parametrize('seed', [0, 1, 2])
def test_committed_plumbing_golden_is_reproduced_by_the_reference_code(seed):
    """tests/golden/plumbing_seed*.npz (what the GPU suite holds the product to) were generated by the oracle; the reference's own
    EncoderDecoder.forward_inference (reference framework + LSS + decoder behind import stubs, state_dict names identical) with the
    SAME calibrated weights gave tests/golden/ref_calibrated_plumbing_seed*.npz (make_reference_checks_golden.py).  The committed
    golden and the oracle run now must both equal it — so the GPU golden test is, transitively, a test against the reference's code."""
    from make_reference_checks_golden import CALIBRATED_KEYS
    from oracle.model import EncoderDecoder as Oracle, calibrate_bn, init_oracle_weights
    from thinktwice_b200.config import Config, PLUMBING_CONFIG
    from thinktwice_b200.synthetic import make_batch
    cfg = Config.fromfile(PLUMBING_CONFIG)
    o = Oracle(**{k: v for k, v in cfg.model.items() if k != 'type'})
    init_oracle_weights(o, seed)
    batch = make_batch(cfg, 1, seed=seed, num_points=2000)
    calibrate_bn(o, batch)
    with torch.no_grad():
        pred = o.eval().forward_inference(batch)
    ref = np.load(os.path.join(G, f'ref_calibrated_plumbing_seed{seed}.npz'))
    g = np.load(os.path.join(G, f'plumbing_seed{seed}.npz'))
    for k in CALIBRATED_KEYS:
        assert rel(g[k], ref[k]) < 1e-5, k
        assert rel(pred[k].numpy(), ref[k]) < 1e-5, k


def test_full_thinktwice_config_oracle_equals_the_reference_code():
    """the bench workload itself (thinktwice.py: 4 cams x 2 sweeps 448x896, 40k LiDAR points, K = 5, B = 1): the reference's
    EncoderDecoder.forward_inference (its framework, LSS and decoder code; LiDAR encoder = oracle stand-in) with the same calibrated
    weights, as stored in tests/golden/ref_full_thinktwice.npz, against the oracle.  ~70 s of CPU."""
    from make_reference_checks_golden import FULL_SHAPE_THREADS, fixed_threads, pred_digest
    from oracle.model import EncoderDecoder as Oracle, calibrate_bn, init_oracle_weights
    from thinktwice_b200.config import Config, DEFAULT_CONFIG
    from thinktwice_b200.synthetic import make_batch
    cfg = Config.fromfile(DEFAULT_CONFIG)
    o = Oracle(**{k: v for k, v in cfg.model.items() if k != 'type'})
    init_oracle_weights(o, 0)
    batch = make_batch(cfg, 1, seed=0, num_points=40000)
    with fixed_threads(FULL_SHAPE_THREADS):
        calibrate_bn(o, batch)
        with torch.no_grad():
            po = pred_digest(o.eval().forward_inference(batch))
    ref = np.load(os.path.join(G, 'ref_full_thinktwice.npz'))
    assert sorted(po) == sorted(ref.files)
    for k, v in po.items():
        assert rel(v.numpy(), ref[k]) < 1e-6, k


@pytest.mark.parametrize('which', ['plumbing', 'full'])
def test_product_host_camera_geometry_equals_the_reference_lss(which):
    """what the PRODUCT computes on the host for the camera branch (thinktwice_b200/lss.py: frustum axes, build_mats, the
    [ida^-1 | sensor2ego . intrin^-1] pair the lift kernel consumes, DepthNet's 22 camera scalars, the voxel-grid lower bound)
    against the reference LSS, as stored in tests/golden/ref_camera_geometry_*.npz: create_frustum, get_geometry (incl.
    transpose-not-inverse and key-frame mats for the history sweep, at a seeded sample of frustum positions) and the tensor
    DepthNet feeds its BatchNorm1d(22)."""
    from make_reference_checks_golden import frustum_from_axes
    from thinktwice_b200.config import Config, DEFAULT_CONFIG, PLUMBING_CONFIG
    from thinktwice_b200.registry import BACKBONES
    from thinktwice_b200.synthetic import make_batch
    cfg = Config.fromfile(PLUMBING_CONFIG if which == 'plumbing' else DEFAULT_CONFIG)
    ref = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(G, f'ref_camera_geometry_{which}.npz')).items()}
    prod = BACKBONES.build(dict(cfg.model['img_encoder']))
    B = 2
    batch = make_batch(cfg, B, seed=3, num_points=10)
    metas = batch['img_metas']
    N = batch['img'].shape[2]
    # frustum and grid constants
    assert torch.equal(prod.frustum, frustum_from_axes(ref['frustum.u'], ref['frustum.v'], ref['frustum.d']))
    assert torch.equal(prod.voxel_coord - prod.voxel_size / 2.0, ref['lower'])
    assert [int(v) for v in prod.voxel_num] == [int(v) for v in ref['voxel_num']]
    # matrices as LSS.forward assembles them (lss.py:667-687)
    mats = prod.build_mats(metas, N)
    intr = torch.stack([torch.stack([torch.cat([torch.cat([m['cam_intrinsic'], torch.zeros(N, 3, 1)], 2),
                                                torch.tensor([0., 0., 0., 1.]).expand(N, 1, 4)], 1) for m in f]) for f in metas])
    assert torch.equal(mats['intrin_mats'], intr.float())
    # geometry: reference get_geometry vs the product's two matrices applied the way the lift kernel does
    T = len(metas[0])
    fr = prod.frustum.reshape(-1, 4)[ref['sample_index']]             # (S, 4) = (u, v, d, 1) at the stored positions
    for s in range(T):
        idx = -1 if s == 0 else -s                                     # the sweep index LSS.forward passes (lss.py:689, 712)
        geom_ref = ref[f'geom_mats{idx}']
        ida_inv = torch.inverse(mats['ida_mats'][:, idx])
        comb = mats['sensor2ego_mats'][:, idx].matmul(torch.inverse(mats['intrin_mats'][:, idx]))
        p = torch.einsum('bnij,sj->bnsi', ida_inv, fr)
        p = torch.cat([p[..., :2] * p[..., 2:3], p[..., 2:]], -1)
        geom = torch.einsum('bnij,bnsj->bnsi', comb, p)[..., :3]
        assert rel(geom.numpy(), geom_ref.numpy()) < 1e-6
        # and the integer voxel index, truncation toward zero (lss.py:630-631)
        lower = ref['lower']
        assert torch.equal(((geom - lower) / ref['voxel_size']).int(), ((geom_ref - lower) / ref['voxel_size']).int())
    # DepthNet's camera-awareness vector (lss.py:206-231): what reaches BatchNorm1d(22)
    assert torch.equal(prod.depthnet_mlp_input(mats)[:, :22], ref['depthnet_bn_input'])
