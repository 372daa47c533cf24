"""CPU: the C-ABI library loads and exports every symbol include/tt_b200.h declares (no compute calls without a GPU)."""
import ctypes as C
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, 'include', 'tt_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(tt_[a-z0-9_]+)\s*\(', src)))


def test_library_exports_every_declared_symbol():
    from thinktwice_b200 import lib
    if not os.path.exists(lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    L = C.CDLL(lib.LIB_PATH)
    syms = declared_symbols()
    assert len(syms) >= 30
    missing = [s for s in syms if not hasattr(L, s)]
    assert not missing, missing
    assert set(syms) <= set(lib.EXPORTS) | {'tt_debug_set'} or not (set(syms) - set(lib.EXPORTS) - {'tt_debug_set'})
    L.tt_version.restype = C.c_int
    assert L.tt_version() >= 100
    L.tt_last_error.restype = C.c_char_p
    assert isinstance(L.tt_last_error(), bytes)


def test_library_exports_the_reference_launcher_symbol():
    """the C++ symbol the reference's pybind wrapper calls (ops/voxel_pooling/src/voxel_pooling_forward.cpp:21-22,36):
    same mangled name as the definition in the reference's own .cu (oracle/_ref carries that one when it was built)."""
    from thinktwice_b200 import lib
    L = C.CDLL(lib.LIB_PATH)
    name = '_Z37voxel_pooling_forward_kernel_launcheriiiiiiPKiPKfPfPiP11CUstream_st'
    assert hasattr(L, name)
    ref = os.path.join(ROOT, 'oracle', '_ref', 'libvoxel_pooling_ref.so')
    if os.path.exists(ref):
        assert hasattr(C.CDLL(ref), name)                           # the reference build exports the very same symbol


def test_product_fails_loudly_without_cuda():
    import pytest
    import torch
    from thinktwice_b200 import lib
    from thinktwice_b200.config import Config, PLUMBING_CONFIG
    from thinktwice_b200.registry import build_model
    if torch.cuda.is_available():
        pytest.skip('CUDA present')
    m = build_model(Config.fromfile(PLUMBING_CONFIG).model)
    with pytest.raises(lib.TTError):
        m.prepare('cpu')
    from thinktwice_b200.ops.voxel_pooling import voxel_pooling
    with pytest.raises(lib.TTError):
        voxel_pooling(torch.zeros(1, 4, 3, dtype=torch.int32), torch.zeros(1, 4, 8), torch.tensor([2, 2, 1]))


def test_config_model_section_equals_reference_when_present():
    """the model section of configs/thinktwice.py carries the reference's values: compared with the reference's own model
    section, stored as tests/golden/ref_config_model.json (make_reference_checks_golden.py)."""
    import json
    import sys
    from thinktwice_b200.config import Config, DEFAULT_CONFIG
    sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))
    from make_reference_checks_golden import norm_config as norm
    ours = Config.fromfile(DEFAULT_CONFIG)
    assert ours.model.decoder.config.pred_len == 4 and ours.model.img_encoder.final_dim == (448, 896)
    with open(os.path.join(ROOT, 'tests', 'golden', 'ref_config_model.json')) as f:
        ref = json.load(f)

    def diff(a, b, path=''):
        out = []
        if isinstance(a, dict):
            for k in a:                                            # every key we carry must equal the reference's
                out += diff(a[k], b.get(k, '<missing>'), path + '/' + k) if isinstance(b, dict) else [path]
        elif a != b:
            out.append((path, a, b))
        return out
    assert not diff(norm(ours.model), ref)


def test_ctypes_structs_match_the_c_header(tmp_path):
    """sizeof / offsetof of every descriptor struct as gcc lays out include/tt_b200.h vs. the ctypes mirror in lib.py
    (the header is plain C99: it must compile without a C++ compiler)."""
    import ctypes as C
    import os
    import subprocess
    from thinktwice_b200 import lib
    pairs = {'tt_conv_desc': lib.ConvDesc, 'tt_lift_splat_desc': lib.LiftSplatDesc, 'tt_voxelize_desc': lib.VoxelizeDesc,
             'tt_rulebook_desc': lib.RulebookDesc, 'tt_sparse_conv_desc': lib.SparseConvDesc, 'tt_look_desc': lib.LookDesc,
             'tt_msda_desc': lib.MsdaDesc, 'tt_preproc_desc': lib.PreprocDesc}
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "tt_b200.h"', 'int main(void) {']
    for cname, cls in pairs.items():
        src.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            src.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    src += ['  return 0;', '}']
    cfile = tmp_path / 'abi.c'
    cfile.write_text('\n'.join(src))
    exe = tmp_path / 'abi'
    subprocess.run(['gcc', '-std=c99', '-Wall', '-Werror', '-I', os.path.join(root, 'include'), str(cfile), '-o', str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, cls in pairs.items():
        assert int(got[cname]) == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f'{cname}.{fname}']) == getattr(cls, fname).offset, f'{cname}.{fname}'


def test_new_entry_points_fail_loudly_without_cuda_too():
    """rows f1 / f4: the GPU pre-processor and the MSDA function refuse CPU devices / tensors instead of falling back."""
    import pytest
    import torch
    from thinktwice_b200 import lib
    from thinktwice_b200.ops.ms_deform_attn import MultiScaleDeformableAttnFunction_fp32
    from thinktwice_b200.preprocess import AgentPreprocessor
    if torch.cuda.is_available():
        pytest.skip('CUDA present')
    with pytest.raises(lib.TTError):
        AgentPreprocessor(dict(undistort=False, num_cams=1), {'final_dim': (4, 4), 'H': 8, 'W': 8, 'bot_pct_lim': (0.0, 0.0)}, 'cpu')
    v = torch.zeros(1, 4, 2, 8)
    loc, aw = torch.zeros(1, 3, 2, 1, 4, 2), torch.zeros(1, 3, 2, 1, 4)
    with pytest.raises(lib.TTError):
        MultiScaleDeformableAttnFunction_fp32.apply(v, torch.tensor([[2, 2]]), torch.tensor([0]), loc, aw, 64)
