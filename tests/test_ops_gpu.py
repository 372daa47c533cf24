"""Per-op parity of the C-ABI library (libtt_b200.so) against plain PyTorch fp32 / the oracle, on the GPU.

Every test calls the product path through thinktwice_b200.lib (ctypes -> extern "C"), never a torch fallback.
Tolerances: fp32 SIMT kernels differ from torch only by summation order -> 1e-4 relative to the tensor's max
(the path-level bar of BASELINE.json is 1e-3); integer / index outputs are compared exactly.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


@pytest.fixture(scope='module')
def eng():
    from thinktwice_b200.engine import Engine
    return Engine('cuda:0')


def relerr(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-12))


def to_fmap(eng, x_nchw, ld=None, coff=0):
    from thinktwice_b200.engine import FMap
    N, Cc, H, W = x_nchw.shape
    ld = ld or Cc
    t = torch.zeros(N, H, W, ld, device='cuda')
    t[..., coff:coff + Cc] = x_nchw.permute(0, 2, 3, 1)
    return FMap(t, N, H, W, Cc, ld, coff)


def packer(sd):
    from thinktwice_b200.weights import Packer
    return Packer(sd, torch.device('cuda:0'))


CONV_CASES = [
    # N, H, W, Cin, Cout, k, stride, pad, dil, groups, bias, act
    (2, 14, 20, 16, 32, 3, 1, 1, 1, 1, True, 1),
    (1, 17, 13, 64, 128, 1, 1, 0, 1, 1, False, 0),
    (2, 32, 32, 3, 64, 7, 2, 3, 1, 1, False, 1),        # stem, scalar A path
    (1, 28, 56, 32, 48, 3, 1, 6, 6, 1, False, 1),       # dilated (ASPP)
    (2, 21, 21, 32, 64, 3, 2, 0, 1, 1, True, 1),        # conv21_10
    (1, 12, 12, 64, 64, 3, 1, 1, 1, 4, False, 0),       # grouped
    (1, 9, 9, 38, 32, 3, 1, 1, 1, 1, True, 3),          # GRU gate, scalar A path, sigmoid
    (3, 8, 8, 512, 18, 3, 1, 1, 1, 1, True, 0),         # DCN offset conv: Cout % 4 != 0
    (1, 40, 40, 256, 256, 3, 1, 1, 1, 1, True, 2),      # big tile path, gelu
    (4, 64, 64, 128, 64, 3, 2, 1, 1, 1, True, 1),       # 128x64 tile path
    (4, 2, 2, 256, 512, 3, 1, 1, 1, 1, True, 1),        # pyramid MLP2: M = 16, K = 2304 -> split-K
    (1, 21, 21, 2080, 128, 3, 1, 1, 1, 1, True, 1),     # decoder BEV update: M = 441, K = 18720 -> split-K
]


@pytest.mark.parametrize('case', CONV_CASES)
def test_conv2d_matches_torch(eng, case):
    N, H, W, Cin, Cout, k, s, p, dil, g, bias, act = case
    gen = torch.Generator().manual_seed(hash(case) % 1000)
    x = torch.randn(N, Cin, H, W, generator=gen).cuda()
    w = (torch.randn(Cout, Cin // g, k, k, generator=gen) * (Cin // g * k * k) ** -0.5)
    b = torch.randn(Cout, generator=gen) if bias else None
    sd = {'c.weight': w}
    if bias:
        sd['c.bias'] = b
    pw = packer(sd).conv('c', groups=g)
    y = eng.conv(to_fmap(eng, x), pw, name=f't.conv{case}', stride=s, pad=p, dil=dil, act=act)
    ref = F.conv2d(x, w.cuda(), b.cuda() if bias else None, stride=s, padding=p, dilation=dil, groups=g)
    ref = {0: ref, 1: F.relu(ref), 2: F.gelu(ref), 3: torch.sigmoid(ref)}[act]
    assert y.nchw().shape == ref.shape
    assert relerr(y.nchw(), ref) < 1e-4


def test_conv2d_concat_offsets_and_residuals(eng):
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(2, 24, 10, 12, generator=gen).cuda()
    w = torch.randn(16, 24, 3, 3, generator=gen) * 0.1
    r1 = torch.randn(2, 16, 10, 12, generator=gen).cuda()
    r2 = torch.randn(2, 16, 10, 12, generator=gen).cuda()
    pw = packer({'c.weight': w}).conv('c')
    xin = to_fmap(eng, x, ld=40, coff=8)                         # input lives inside a wider buffer
    out = eng.fmap('t.cat', 2, 10, 12, 48)
    eng.fill(out.t, 7.0)
    y = eng.conv(xin, pw, out=out.slice(20, 16), pad=1, act=1, res=to_fmap(eng, r1), res2=to_fmap(eng, r2, ld=32, coff=4))
    ref = F.relu(F.conv2d(x, w.cuda(), padding=1) + r1 + r2)
    assert relerr(y.nchw(), ref) < 1e-4
    assert float((out.t[..., :20] - 7).abs().max()) == 0 and float((out.t[..., 36:] - 7).abs().max()) == 0


def test_conv2d_upsampled_residual_pafpn(eng):
    from thinktwice_b200 import lib
    gen = torch.Generator().manual_seed(2)
    x = torch.randn(2, 32, 12, 16, generator=gen).cuda()
    top = torch.randn(2, 8, 6, 8, generator=gen).cuda()
    w = torch.randn(8, 32, 1, 1, generator=gen) * 0.2
    b = torch.randn(8, generator=gen)
    pw = packer({'c.weight': w, 'c.bias': b}).conv('c')
    y = eng.conv(to_fmap(eng, x), pw, name='t.lat', res=to_fmap(eng, top), res_mode=lib.RES_UP2)
    ref = F.conv2d(x, w.cuda(), b.cuda()) + F.interpolate(top, size=(12, 16), mode='nearest')
    assert relerr(y.nchw(), ref) < 1e-4


def test_conv_transpose_k2s2(eng):
    gen = torch.Generator().manual_seed(3)
    x = torch.randn(2, 32, 7, 9, generator=gen).cuda()
    w = torch.randn(32, 16, 2, 2, generator=gen) * 0.2
    b = torch.randn(16, generator=gen)
    ups = packer({'u.weight': w, 'u.bias': b}).convT('u')
    out = eng.fmap('t.up', 2, 14, 18, 16)
    for i in range(2):
        for j in range(2):
            eng.conv(to_fmap(eng, x), ups[i][j], out=out, scatter=(2, i, 2, j))
    ref = F.conv_transpose2d(x, w.cuda(), b.cuda(), stride=2)
    assert relerr(out.nchw(), ref) < 1e-4


def test_linear_small_and_padded(eng):
    gen = torch.Generator().manual_seed(4)
    for rows, cin, cout in [(1, 384, 512), (5, 1543, 512), (33, 514, 2), (480, 256, 1024), (1, 2304, 512), (4, 1024, 512)]:
        x = torch.randn(rows, cin, generator=gen).cuda()
        w = torch.randn(cout, cin, generator=gen) * cin ** -0.5
        b = torch.randn(cout, generator=gen)
        pw = packer({'l.weight': w, 'l.bias': b}).linear('l')
        y = eng.linear(eng.wrap(x.view(rows, 1, 1, cin).contiguous()), pw, name=f't.lin{rows}_{cin}_{cout}', act=2)
        ref = F.gelu(F.linear(x, w.cuda(), b.cuda()))
        assert relerr(y.t.view(rows, cout), ref) < 1e-4


def test_memory_bound_ops(eng):
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(2, 64, 15, 22, generator=gen).cuda()
    fx = to_fmap(eng, x)
    assert relerr(eng.maxpool3x3s2(fx, 't.mp').nchw(), F.max_pool2d(x, 3, 2, 1)) < 1e-6
    assert relerr(eng.upsample2x(fx, 't.up2').nchw(), F.interpolate(x, scale_factor=2, mode='bilinear', align_corners=True)) < 1e-5
    assert relerr(eng.global_avgpool(fx, 't.gap').t.view(2, 64), x.mean((2, 3))) < 1e-5
    assert relerr(eng.se_pool(fx, 't.sep').t.view(2, 64), 0.5 * x.mean((2, 3)) + 0.5 * x.amax((2, 3))) < 1e-5
    g = torch.randn(2, 64, generator=gen).cuda()
    fg = eng.wrap(g.view(2, 1, 1, 64).contiguous())
    assert relerr(eng.se_gate(fx, fg, 't.seg').nchw(), x * torch.sigmoid(g)[..., None, None]) < 1e-5
    sc = torch.randn(2, 64, 15, 22, generator=gen).cuda()
    assert relerr(eng.se_apply(fx, fg, to_fmap(eng, sc), name='t.sea').nchw(), F.relu(x * torch.sigmoid(g)[..., None, None] + sc)) < 1e-5
    sq = torch.randn(2, 8, 21, 21, generator=gen).cuda()
    assert relerr(eng.anti_transpose(to_fmap(eng, sq), 't.at').nchw(), torch.rot90(torch.flip(sq, dims=[2]), 1, dims=[2, 3])) == 0
    # NCHW <-> NHWC round trip incl. channel padding
    img = torch.randn(3, 3, 10, 14, generator=gen).cuda()
    f = eng.nchw_to_nhwc(img, 't.nhwc', cpad=4)
    assert torch.equal(f.t[..., :3], img.permute(0, 2, 3, 1)) and float(f.t[..., 3].abs().max()) == 0
    assert torch.equal(eng.nhwc_to_nchw(f.slice(0, 3), 't.nchw'), img)
    # layernorm
    r = torch.randn(37, 1543, generator=gen).cuda()
    gm, bt = torch.randn(1543, generator=gen).cuda(), torch.randn(1543, generator=gen).cuda()
    y = eng.layernorm(eng.wrap(r.view(37, 1, 1, 1543).contiguous()), gm, bt, name='t.ln', out_ld=1544)
    assert relerr(y.t.view(37, 1544)[:, :1543], F.layer_norm(r, (1543,), gm, bt)) < 1e-5
    assert float(y.t.view(37, 1544)[:, 1543].abs().max()) == 0
    # copy with row broadcast, eltwise
    src = torch.randn(3, 1, 1, 8, generator=gen).cuda()
    dst = eng.fmap('t.cp', 12, 1, 1, 20, zero=True)
    eng.copy_cols(eng.wrap(src), dst.slice(4, 8), rdiv=4)
    assert torch.equal(dst.t.view(12, 20)[:, 4:12], src.view(3, 8).repeat_interleave(4, 0))
    eng.copy_cols(eng.wrap(src), dst.slice(12, 8), rmod=3)
    assert torch.equal(dst.t.view(12, 20)[:, 12:20], src.view(3, 8).repeat(4, 1))
    a, b, c = (torch.rand(6, 1, 1, 10, generator=gen).cuda() for _ in range(3))
    assert relerr(eng.eltwise(2, eng.wrap(a), eng.wrap(b), eng.wrap(c), name='t.e2').t, (1 - a) * b + a * c) < 1e-6
    assert relerr(eng.eltwise(3, eng.wrap(a - 0.5), name='t.e3', act=5).t, torch.clamp(F.softplus(a - 0.5), min=1e-3)) < 1e-6


def _rand_geom(gen, B, P, X, Y):
    g = torch.stack([torch.randint(-2, X + 2, (B, P), generator=gen), torch.randint(-2, Y + 2, (B, P), generator=gen),
                     torch.randint(-1, 2, (B, P), generator=gen)], -1).int()
    return g


@pytest.mark.parametrize('shape', [(1, 5000, 64, 21, 21), (2, 20000, 256, 21, 21), (1, 30000, 80, 200, 200), (1, 100, 7, 5, 4)])
def test_voxel_pooling_dropin_matches_oracle_and_reference_kernel(shape):
    from oracle.voxel_pool import voxel_pooling_ref
    from thinktwice_b200.ops.voxel_pooling import voxel_pooling
    B, P, Cc, X, Y = shape
    gen = torch.Generator().manual_seed(P)
    geom = _rand_geom(gen, B, P, X, Y)
    feats = torch.randn(B, P, Cc, generator=gen)
    vn = torch.tensor([X, Y, 1])
    ref = voxel_pooling_ref(geom, feats, vn)
    out = voxel_pooling(geom.cuda().contiguous(), feats.cuda().contiguous(), vn.cuda())
    assert out.shape == (B, Cc, Y, X)
    assert relerr(out, ref) < 1e-5
    # the reference's own kernel on the same inputs, as stored by tests/golden/make_voxel_pool_golden.py: a sample of its
    # output, its per-channel sums and a digest of its last-position memo
    gdir = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
    sys.path.insert(0, gdir)
    from make_voxel_pool_golden import SYMBOL, key, memo_digest
    from thinktwice_b200.ops.voxel_pooling import last_pos_memo
    gold = np.load(os.path.join(gdir, 'ref_voxel_pooling_kernel.npz'))
    k = key(shape)

    def assert_matches_reference(o_byxc, memo):
        assert relerr(o_byxc.cpu().flatten()[torch.from_numpy(gold[k + 'index']).long()], torch.from_numpy(gold[k + 'sample'])) < 1e-5
        assert relerr(o_byxc.double().sum((1, 2)), torch.from_numpy(gold[k + 'channel_sum'])) < 1e-5
        assert memo_digest(memo) == str(gold[k + 'memo_sha256'])  # integer side: bit-exact
    assert_matches_reference(out.permute(0, 2, 3, 1), last_pos_memo())
    # the product's link-level drop-in: the SAME mangled symbol exported by libtt_b200.so (voxel_pooling_forward.cpp:21-22)
    from thinktwice_b200 import lib as ttlib
    fn3 = getattr(C.CDLL(ttlib.LIB_PATH), SYMBOL)
    g, f = geom.cuda().contiguous(), feats.cuda().contiguous()
    o3 = torch.zeros(B, Y, X, Cc, device='cuda')
    memo3 = -torch.ones(B, P, 3, dtype=torch.int32, device='cuda')
    fn3(B, P, Cc, X, Y, 1, C.c_void_p(g.data_ptr()), C.c_void_p(f.data_ptr()), C.c_void_p(o3.data_ptr()),
        C.c_void_p(memo3.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert_matches_reference(o3, memo3)


def test_voxel_pooling_empty_input():
    from thinktwice_b200.ops.voxel_pooling import voxel_pooling
    out = voxel_pooling(torch.zeros(1, 0, 3, dtype=torch.int32, device='cuda'), torch.zeros(1, 0, 8, device='cuda'),
                        torch.tensor([4, 4, 1]))
    assert out.shape == (1, 8, 4, 4) and float(out.abs().sum()) == 0


@pytest.mark.parametrize('B', [1, 2])
def test_lift_splat_matches_oracle_lift_and_pool(eng, B):
    """fused kernel == softmax (x) outer product (x) get_geometry (x) voxel pool of the oracle (lss.py:582-632)."""
    from oracle.camera import LSS as OLSS
    from oracle.voxel_pool import voxel_pooling_ref
    from thinktwice_b200.config import Config, PLUMBING_CONFIG
    from thinktwice_b200.lss import LSS
    from thinktwice_b200.synthetic import rig_metas
    cfg = Config.fromfile(PLUMBING_CONFIG).model.img_encoder
    kw = {k: v for k, v in cfg.items() if k != 'type'}
    kw['d_bound'] = [1.0, 41.0, 0.5]                             # full depth range: rays leave the 21x21 grid
    o = OLSS(**kw)
    m = LSS(**kw)
    N, D, fH, fW, Cc = 4, o.depth_channels, 16, 16, 256
    gen = torch.Generator().manual_seed(B)
    depth = torch.randn(B * N, D, fH, fW, generator=gen) * 2
    ctx = torch.randn(B * N, Cc, fH, fW, generator=gen)
    metas = [rig_metas((256, 256), 1) for _ in range(B)]
    mats = o.build_mats(metas, N)
    geom = o.get_geometry(mats['sensor2ego_mats'][:, -1], mats['intrin_mats'][:, -1], mats['ida_mats'][:, -1])
    lifted = (depth.softmax(1).unsqueeze(1) * ctx.unsqueeze(2)).reshape(B, N, Cc, D, fH, fW).permute(0, 1, 3, 4, 5, 2).contiguous()
    ref = voxel_pooling_ref(o.geom_index(geom).contiguous(), lifted, o.voxel_num)
    inside = ((o.geom_index(geom)[..., 0] >= 0) & (o.geom_index(geom)[..., 0] < 21)).float().mean()
    assert 0.05 < float(inside) < 0.95
    # product path
    from thinktwice_b200 import lib
    from thinktwice_b200.lib import LiftSplatDesc, _p
    fd, fc = to_fmap(eng, depth.cuda()), to_fmap(eng, ctx.cuda())
    ida_inv = torch.inverse(mats['ida_mats'][:, -1])
    comb = mats['sensor2ego_mats'][:, -1].matmul(torch.inverse(mats['intrin_mats'][:, -1]))
    mm = torch.stack([ida_inv, comb], 2).reshape(B * N, 32).contiguous().cuda()
    d = LiftSplatDesc()
    d.B, d.N, d.D, d.fH, d.fW, d.C = B, N, D, fH, fW, Cc
    d.ld_d, d.d_coff, d.ld_c, d.c_coff = D, 0, Cc, 0
    d.lower, d.size = lib.f3(m.voxel_coord - m.voxel_size / 2.0), lib.f3(m.voxel_size)
    d.X, d.Y, d.Z, d.bev_ld, d.bev_coff, d.anti_transpose = 21, 21, 1, Cc, 0, 0
    ws = torch.empty(lib.load().tt_lift_splat_workspace_bytes(C.byref(d)), dtype=torch.uint8, device='cuda')
    bev = torch.full((B, 21, 21, Cc), 3.0, device='cuda')
    fu, fv, fdd = m.frustum_u.cuda(), m.frustum_v.cuda(), m.frustum_d.cuda()      # keep alive across the call
    lib.call('tt_lift_splat', C.byref(d), _p(fd.t), _p(fc.t), _p(mm), _p(fu), _p(fv), _p(fdd), _p(bev), _p(ws))
    err = relerr(bev.permute(0, 3, 1, 2), ref)
    print('lift_splat err', err)
    assert err < 1e-3                                             # a few boundary points may switch cell (fp32 geometry)


def test_dcn_matches_torchvision(eng):
    from torchvision.ops import deform_conv2d
    from thinktwice_b200.lib import _p
    from thinktwice_b200 import lib
    gen = torch.Generator().manual_seed(9)
    N, Cc, H, W, G = 2, 64, 12, 17, 4
    x = torch.randn(N, Cc, H, W, generator=gen).cuda()
    off = (torch.randn(N, 18, H, W, generator=gen) * 1.5).cuda()
    w = (torch.randn(Cc, Cc // G, 3, 3, generator=gen) * 0.1)
    ref = deform_conv2d(x, off, w.cuda(), padding=1)
    fx, fo = to_fmap(eng, x), to_fmap(eng, off)
    col = eng.fmap('t.dcn.col', N, H, W, 9 * Cc)
    lib.call('tt_dcn_im2col', _p(fx.t), _p(fo.t), fo.ld, _p(col.t), N, H, W, Cc, G)
    pw = packer({'d.weight': w}).conv('d', groups=G)
    pw.Cin, pw.KH, pw.KW = 9 * Cc, 1, 1
    y = eng.conv(col, pw, name='t.dcn.out')
    assert relerr(y.nchw(), ref) < 1e-4


def test_voxelize_mean_matches_oracle(eng):
    from oracle.lidar import hard_voxelize
    from thinktwice_b200.lib import VoxelizeDesc, _p
    from thinktwice_b200 import lib
    gen = torch.Generator().manual_seed(11)
    B, P = 2, 3000
    pts = torch.rand(B, P, 5, generator=gen)
    pts[..., :3] = pts[..., :3] * torch.tensor([3.0, 3.0, 2.0]) - torch.tensor([0.3, 0.3, 0.2])
    pts[:, :500, :3] = pts[:, 500:1000, :3]                       # duplicates -> several points per voxel
    pts[:, 1000:1400, :3] = pts[:, 500:900, :3] + 1e-4
    vs, rng, mp = [0.1, 0.1, 0.2], [0.0, 0.0, 0.0, 2.4, 2.4, 1.6], 3
    d = VoxelizeDesc()
    d.B, d.P, d.F = B, P, 5
    d.lower, d.vsize, d.grid = lib.f3(rng[:3]), lib.f3(vs), lib.i3([24, 24, 8])
    d.zmax, d.max_points, d.max_voxels, d.cap = 6, mp, 100000, B * P
    ws = torch.empty(lib.load().tt_voxelize_workspace_bytes(C.byref(d)), dtype=torch.uint8, device='cuda')
    feats, coords = torch.zeros(B * P, 5, device='cuda'), torch.zeros(B * P, 4, dtype=torch.int32, device='cuda')
    count = torch.zeros(1, dtype=torch.int32, device='cuda')
    dpts = pts.cuda().contiguous()
    lib.call('tt_voxelize_mean', C.byref(d), _p(dpts), _p(feats), _p(coords), _p(count), _p(ws))
    n = int(count.item())
    got = {tuple(c.tolist()): f for c, f in zip(coords[:n].cpu(), feats[:n].cpu())}
    exp = {}
    for b in range(B):
        v, c, num = hard_voxelize(pts[b], vs, rng, mp, 100000)
        mean = v.sum(1) / num.float().view(-1, 1)
        for ci, mi in zip(c, mean):
            if int(ci[0]) < 6:
                exp[(b,) + tuple(ci.tolist())] = mi
    assert set(got) == set(exp)                                   # voxel set: exact
    err = max(float((got[k] - exp[k]).abs().max()) for k in exp)
    assert err < 1e-6


@pytest.mark.parametrize('Cin,Cout,density,impl', [(16, 32, 0.08, 1), (64, 128, 0.25, 3), (32, 32, 0.3, 3), (128, 64, 0.15, 3)])
def test_sparse_conv_layers_match_oracle(Cin, Cout, density, impl):
    """impl 1: fused SIMT gather GEMM; impl 3: tcgen05 3xTF32 gather GEMM (cp.async row gather, red.add epilogue)."""
    from oracle.lidar import SparseConvBase, SparseTensor
    from thinktwice_b200.lib import RulebookDesc, _p
    from thinktwice_b200 import lib
    from thinktwice_b200.engine import Engine
    from thinktwice_b200.weights import tf32_split
    eng = Engine('cuda:0', impl=impl)
    gen = torch.Generator().manual_seed(13)
    B, shape = 2, (9, 24, 20)
    mask = torch.rand(B, *shape, generator=gen) < density
    coords = mask.nonzero().int()
    coords = coords[torch.randperm(coords.shape[0], generator=gen)]
    n = coords.shape[0]
    feats = torch.randn(n, Cin, generator=gen)
    x = SparseTensor(feats, coords, shape, B)
    for (k, s, p, subm) in [((3, 3, 3), (1, 1, 1), (1, 1, 1), True), ((3, 3, 3), (2, 2, 2), (1, 1, 1), False),
                            ((3, 3, 3), (2, 2, 2), (0, 1, 1), False), ((3, 1, 1), (2, 1, 1), (0, 0, 0), False)]:
        conv = SparseConvBase(Cin, Cout, k, stride=s, padding=p, subm=subm)
        with torch.no_grad():
            ref = conv(x).dense()
        cap_in = n + 7
        out_shape = shape if subm else tuple((shape[i] + 2 * p[i] - k[i]) // s[i] + 1 for i in range(3))
        cap_out = cap_in if subm else min(cap_in * 8, B * out_shape[0] * out_shape[1] * out_shape[2])
        d = RulebookDesc()
        d.B, d.in_shape, d.out_shape, d.k, d.s, d.p = B, lib.i3(shape), lib.i3(out_shape), lib.i3(k), lib.i3(s), lib.i3(p)
        d.subm, d.cap_in, d.cap_out = int(subm), cap_in, cap_out
        t = 1024
        while t < 2 * max(cap_in, cap_out):
            t <<= 1
        d.table_size = t
        ws = torch.empty(lib.load().tt_rulebook_workspace_bytes(C.byref(d)), dtype=torch.uint8, device='cuda')
        ic = torch.zeros(cap_in, 4, dtype=torch.int32, device='cuda'); ic[:n] = coords.cuda()
        icount = torch.tensor([n], dtype=torch.int32, device='cuda')
        oc = torch.zeros(cap_out, 4, dtype=torch.int32, device='cuda'); ocount = torch.zeros(1, dtype=torch.int32, device='cuda')
        kvol = k[0] * k[1] * k[2]
        nbr = torch.zeros(cap_out, kvol, dtype=torch.int32, device='cuda')
        pin, pout = (torch.zeros(kvol, cap_out, dtype=torch.int32, device='cuda') for _ in range(2))
        pcount = torch.zeros(kvol, dtype=torch.int32, device='cuda')
        lib.call('tt_sparse_rulebook', C.byref(d), _p(ic), _p(icount), _p(oc), _p(ocount), _p(nbr), _p(pin), _p(pout), _p(pcount), _p(ws))
        assert int(pcount.sum()) == int((nbr[:int(ocount.item())] >= 0).sum())               # both rulebook forms agree
        w = conv.weight.detach()
        from thinktwice_b200.engine import PackedConv
        w_tc = torch.stack(tf32_split(w.reshape(Cout, kvol, Cin))).contiguous().cuda() if impl == 3 else None
        pw = PackedConv(w.reshape(Cout, kvol, Cin).permute(1, 2, 0).reshape(kvol * Cin, Cout).contiguous().cuda(), None, Cin, Cout,
                        w_tc=w_tc)
        n0 = lib.launch_count()
        fin = torch.zeros(cap_in, Cin, device='cuda'); fin[:n] = feats.cuda()
        out = torch.zeros(cap_out, Cout, device='cuda')
        rule = dict(kvol=kvol, cap=cap_out, pairs_in=pin, pairs_out=pout, pair_count=pcount, count=ocount)
        eng.sparse_conv(fin, pw, rule, out)
        assert lib.launch_count() - n0 == 3                        # init + ONE launch over all taps + finish
        m = int(ocount.item())
        D, H, W = out_shape
        dense = torch.zeros(B, H, W, Cout * D, device='cuda')
        lib.call('tt_sparse_to_bev', _p(out), _p(oc), _p(ocount), cap_out, Cout, D, H, W, 0, _p(dense))
        got = dense.view(B, H, W, Cout, D).permute(0, 3, 4, 1, 2)
        assert m == int((ref.abs().sum(1) != 0).sum()) or m >= int((ref.abs().sum(1) != 0).sum())
        assert relerr(got, ref) < 1e-4


def test_msda_matches_oracle(eng):
    from oracle.decoder import msda_pytorch
    from thinktwice_b200.lib import MsdaDesc, _p
    from thinktwice_b200 import lib
    gen = torch.Generator().manual_seed(17)
    BN, cap, heads, L, P, dh = 3, 20, 8, 4, 8, 32
    shapes = [(16, 20), (8, 10), (4, 5), (2, 3)]
    nk = sum(h * w for h, w in shapes)
    value = torch.randn(BN, nk, heads * dh, generator=gen)
    off = torch.randn(BN * cap, heads * L * P * 2, generator=gen) * 3
    logits = torch.randn(BN * cap, heads * L * P, generator=gen)
    ref_pts = torch.rand(BN * cap, 2, generator=gen) * 1.2 - 0.1
    norm = torch.tensor([[w, h] for h, w in shapes], dtype=torch.float32)
    loc = ref_pts.view(BN, cap, 1, 1, 1, 2) + off.view(BN, cap, heads, L, P, 2) / norm[None, None, None, :, None, :]
    aw = logits.view(BN, cap, heads, L * P).softmax(-1).view(BN, cap, heads, L, P)
    ref = msda_pytorch(value.view(BN, nk, heads, dh), torch.tensor(shapes), loc, aw)
    d = MsdaDesc()
    d.BN, d.rows_cap, d.heads, d.levels, d.points, d.dh = BN, cap, heads, L, P, dh
    d.lvl_h, d.lvl_w = lib.i4([s[0] for s in shapes]), lib.i4([s[1] for s in shapes])
    starts = np.cumsum([0] + [h * w for h, w in shapes])[:4]
    d.lvl_start, d.num_keys = lib.i4(starts), nk
    out = torch.zeros(BN * cap, heads * dh, device='cuda')
    ml = torch.tensor([cap], dtype=torch.int32, device='cuda')
    dv, do, dl, dr = value.cuda(), off.cuda(), logits.cuda(), ref_pts.cuda()      # keep alive across the call
    lib.call('tt_msda_forward', C.byref(d), _p(dv), _p(do), _p(dl), _p(dr), _p(ml), _p(out))
    assert relerr(out.view(BN, cap, heads * dh), ref) < 1e-4
