"""CPU tests of the drop-in boundary: the C-ABI library loads, exports exactly what
include/gpt4roi_b200.h declares, the Python mirror refuses to run without a GPU (no
fallback), and the product never touches oracle/."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, 'include', 'gpt4roi_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(g4r_[a-z0-9_]+)\s*\(', src)))


@pytest.fixture(scope='module')
def built_lib():
    from gpt4roi_b200 import build, lib
    build.build()
    return lib


def test_header_symbols_are_exported(built_lib):
    decl = _declared_symbols()
    assert len(decl) >= 8
    so = ctypes.CDLL(built_lib.LIB_PATH)
    for name in decl:
        assert hasattr(so, name), '%s declared in include/gpt4roi_b200.h but not exported' % name


def test_python_signature_table_matches_header(built_lib):
    assert sorted(built_lib.SIGNATURES) == _declared_symbols()
    lib = built_lib.load()
    assert lib.g4r_version() >= 1000
    assert lib.g4r_built_arch() == 100


def test_library_is_sm100a_only(built_lib):
    out = subprocess.run(['cuobjdump', '--list-elf', built_lib.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip('cuobjdump unavailable')
    archs = set(re.findall(r'sm_(\d+a?)', out.stdout))
    assert archs == {'100a'}, archs


def test_no_cpu_fallback():
    import gpt4roi_b200 as g
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        g.roi_align(torch.zeros(1, 1, 4, 4), torch.zeros(1, 5), 2, 1.0, 2, 'avg', True)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        g.roi_align_mlvl([torch.zeros(1, 4, 4, 8)], torch.zeros(1, 5), 2, [1.0])


def test_operator_api_mirrors_reference_signatures():
    import inspect
    import gpt4roi_b200 as g
    m = g.RoIAlign(7, 0.25, 2)
    assert m.output_size == (7, 7) and m.spatial_scale == 0.25 and m.sampling_ratio == 2
    assert repr(m) == ('RoIAlign(output_size=(7, 7), spatial_scale=0.25, sampling_ratio=2, '
                       'pool_mode=avg, aligned=True, use_torchvision=False)')
    m = g.RoIAlign(out_size=3, sample_num=4)  # deprecated aliases, mmcv/ops/roi_align.py:171-177
    assert m.output_size == (3, 3) and m.sampling_ratio == 4
    names = ['input', 'rois', 'output', 'argmax_y', 'argmax_x', 'aligned_height', 'aligned_width',
             'spatial_scale', 'sampling_ratio', 'pool_mode', 'aligned']
    assert list(inspect.signature(g.roi_align_forward).parameters) == names
    names[0], names[2], names[4] = 'grad_output', 'argmax_y', 'grad_input'
    names[3] = 'argmax_x'
    assert list(inspect.signature(g.roi_align_backward).parameters) == names
    with pytest.raises(AssertionError):
        g.RoIAlignFunction.apply(torch.zeros(1, 1, 2, 2), torch.zeros(1, 4), 2)  # rois.size(1) != 5


def test_mmcv_ext_dropin_module():
    from gpt4roi_b200 import mmcv_ext
    m = mmcv_ext.make_module()
    assert hasattr(m, 'roi_align_forward') and hasattr(m, 'roi_align_backward')
    assert hasattr(m, 'nms') and hasattr(m, 'deform_conv_forward')  # ext_loader only asserts hasattr
    with pytest.raises(NotImplementedError):
        m.nms()


def test_reference_wrapper_runs_over_the_dropin_and_never_falls_back():
    """How the reference's UNMODIFIED `mmcv.ops.roi_align` / `RoIAlign` (mmcv-1.4.7/mmcv/ops/roi_align.py) uses
    `mmcv._ext`, recorded from the reference by make_golden.py --wrapper (tests/golden/mmcv_wrapper_calls.json), replayed
    against the drop-in `gpt4roi_b200.mmcv_ext`: every symbol `import mmcv.ops` asserts on exists (ext_loader only
    asserts hasattr), the wrapper's forward / backward calls land in OUR entry points and bind their signatures, and on
    CPU tensors those entries raise instead of computing on the CPU.  The same call pattern runs on the GPU in
    tests/test_roi_align_gpu.py::test_mmcv_ext_module_as_the_reference_wrapper_calls_it."""
    import importlib
    import inspect
    import json
    from gpt4roi_b200 import mmcv_ext
    ours = importlib.import_module('gpt4roi_b200.roi_align')
    with open(os.path.join(ROOT, 'tests', 'golden', 'mmcv_wrapper_calls.json')) as f:
        rec = json.load(f)
    m = mmcv_ext.make_module()
    assert len(rec['ext_names']) > 100 and not [n for n in rec['ext_names'] if not hasattr(m, n)]
    assert {'roi_align_forward', 'roi_align_backward'} <= set(rec['ext_names'])
    assert sorted({c['fn'] for c in rec['calls']}) == ['roi_align_backward', 'roi_align_forward']
    for call in rec['calls']:
        fn = getattr(m, call['fn'])
        assert fn is getattr(ours, call['fn'])

        def value(v):
            return torch.zeros(v['shape'], dtype=getattr(torch, v['dtype'])) if isinstance(v, dict) else v
        args = [value(a) for a in call['args']]
        kwargs = {k: value(v) for k, v in call['kwargs'].items()}
        inspect.signature(fn).bind(*args, **kwargs)
        with pytest.raises(RuntimeError, match='CUDA'):
            fn(*args, **kwargs)


def test_product_never_imports_oracle():
    bad = []
    for dp, _, fns in os.walk(os.path.join(ROOT, 'gpt4roi_b200')):
        for fn in fns:
            if fn.endswith(('.py', '.cu', '.cuh', '.h', '.cpp')):
                txt = open(os.path.join(dp, fn)).read()
                if re.search(r'^\s*(from|import)\s+oracle\b|oracle/|liboracle', txt, re.M):
                    bad.append(os.path.join(dp, fn))
    assert not bad, 'product code references oracle/: %s' % bad


def _env_switches_read(*dirs):
    found = set()
    for d in dirs:
        for dp, _, fns in os.walk(os.path.join(ROOT, d)):
            for fn in fns:
                if fn.endswith(('.py', '.cu', '.cuh')):
                    txt = open(os.path.join(dp, fn)).read()
                    found |= set(re.findall(r'''getenv\(\s*"(G4R_[A-Z0-9_]+)"''', txt))
                    found |= set(re.findall(r'''environ\.get\(\s*['"](G4R_[A-Z0-9_]+)['"]''', txt))
    return found


def test_every_environment_switch_is_documented():
    """Every G4R_* variable the package reads is a row of the README's environment table, and every row is read
    somewhere in the package or its tools: no undocumented knob, no documented knob that does nothing."""
    readme = open(os.path.join(ROOT, 'README.md')).read()
    table = readme.split('## Environment switches', 1)[1].split('\n## ', 1)[0]
    rows = set(re.findall(r'^\|\s*`(G4R_[A-Z0-9_]+)`\s*\|', table, re.M))
    assert rows
    read = _env_switches_read('gpt4roi_b200')
    assert read <= rows, 'read but not in the README table: %s' % sorted(read - rows)
    unread = rows - _env_switches_read('gpt4roi_b200', 'tools')
    assert not unread, 'in the README table but read nowhere: %s' % sorted(unread)


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    from gpt4roi_b200 import lib
    monkeypatch.setattr(lib, '_lib', None)
    monkeypatch.setattr(lib, 'LIB_PATH', str(tmp_path / 'nope.so'))
    with pytest.raises(ImportError, match='no CPU'):
        lib.load()


def test_training_ops_fail_loudly_without_cuda():
    """The training-step wrappers have no CPU path: CPU tensors raise (never a silent PyTorch fallback)."""
    import pytest
    import torch
    from gpt4roi_b200 import dense, train, train_ops
    x = torch.zeros(4, 8, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError):
        train_ops.cross_entropy(x, torch.zeros(4, dtype=torch.int64))
    with pytest.raises(RuntimeError):
        dense.matmul_t(x, x, b_mn=True)
    with pytest.raises(RuntimeError):
        train_ops.rmsnorm_bwd(x, torch.zeros(8, dtype=torch.bfloat16), x, 1e-6)
    # pure host logic: the label shift of llava/model/llava.py:241-242
    lab = torch.tensor([[5, 6, -100, 7]])
    assert train.Stage2Trainer.shift_labels(lab).tolist() == [[6, -100, 7, -100]]


def test_fuse_consumers_inverts_the_shuffle_wiring():
    """train_ops.fuse_consumers is the transpose of the forward wiring (level l reads top=min(l+1,n-1), down=max(l-1,0));
    every (reader, source) edge appears exactly once and no level has more than two readers per role (the kernel's limit)."""
    from gpt4roi_b200.train_ops import fuse_consumers
    for n in (1, 2, 3, 4, 5):
        edges_dn = {(l, max(l - 1, 0)) for l in range(n)}
        edges_tp = {(l, min(l + 1, n - 1)) for l in range(n)}
        got_dn, got_tp = set(), set()
        for m in range(n):
            dn, tp = fuse_consumers(n, m)
            assert len(dn) <= 2 and len(tp) <= 2
            got_dn |= {(l, m) for l in dn}
            got_tp |= {(l, m) for l in tp}
        assert got_dn == edges_dn and got_tp == edges_tp


def test_checkpoint_layout_round_trip(tmp_path):
    """fuse_llama_layer / unfuse_llama_layer are exact inverses, and save_checkpoint writes the sharded HF layout
    (pytorch_model-XXXXX-of-YYYYY.bin + pytorch_model.bin.index.json, reference parameter names) the reference's
    trainer produces (train.py:88-98) -- read back bit-identically by load_checkpoint."""
    import json
    import torch
    from gpt4roi_b200 import train
    g = torch.Generator().manual_seed(0)
    H, Fd = 16, 40
    sd = {}
    for i in range(2):
        q = 'model.layers.%d.' % i
        for n in 'qkvo':
            sd[q + 'self_attn.%s_proj.weight' % n] = torch.randn(H, H, generator=g)
        sd[q + 'mlp.gate_proj.weight'] = torch.randn(Fd, H, generator=g)
        sd[q + 'mlp.up_proj.weight'] = torch.randn(Fd, H, generator=g)
        sd[q + 'mlp.down_proj.weight'] = torch.randn(H, Fd, generator=g)
        sd[q + 'input_layernorm.weight'] = torch.randn(H, generator=g)
        sd[q + 'post_attention_layernorm.weight'] = torch.randn(H, generator=g)
    back = {}
    for i in range(2):
        fused = train.fuse_llama_layer(sd, i)
        assert fused['wqkv'].shape == (3 * H, H) and fused['wgu'].shape == (2 * Fd, H)
        assert torch.equal(fused['wgu'][0::2], sd['model.layers.%d.mlp.gate_proj.weight' % i])
        back.update(train.unfuse_llama_layer(fused, i))
    assert set(back) == set(sd) and all(torch.equal(back[k], sd[k]) for k in sd)
    sd['lm_head.weight'] = torch.randn(50, H, generator=g)
    names = train.save_checkpoint(sd, str(tmp_path), max_shard_bytes=6000)
    assert len(names) > 1 and all(n.startswith('pytorch_model-') and n.endswith('-of-%05d.bin' % len(names)) for n in names)
    index = json.load(open(tmp_path / 'pytorch_model.bin.index.json'))
    assert set(index['weight_map']) == set(sd) and index['metadata']['total_size'] == sum(v.numel() * 4 for v in sd.values())
    loaded = train.load_checkpoint(str(tmp_path))
    assert set(loaded) == set(sd) and all(torch.equal(loaded[k], sd[k]) for k in sd)


def test_llama_train_stack_state_dict_round_trip_on_cpu():
    """Construction and checkpoint export of the training stack are pure tensor plumbing (no kernel runs):
    state_dict() returns exactly the reference-named fp32 weights it was built from."""
    import torch
    from gpt4roi_b200.engine import EngineConfig
    from gpt4roi_b200.train import LlamaTrainStack
    cfg = EngineConfig(hidden=256, n_heads=2, n_layers=2, mlp=96, vocab=120)
    g = torch.Generator().manual_seed(1)
    sd = {'model.norm.weight': torch.randn(256, generator=g), 'lm_head.weight': torch.randn(120, 256, generator=g)}
    for i in range(2):
        q = 'model.layers.%d.' % i
        for n in 'qkvo':
            sd[q + 'self_attn.%s_proj.weight' % n] = torch.randn(256, 256, generator=g)
        sd[q + 'mlp.gate_proj.weight'] = torch.randn(96, 256, generator=g)
        sd[q + 'mlp.up_proj.weight'] = torch.randn(96, 256, generator=g)
        sd[q + 'mlp.down_proj.weight'] = torch.randn(256, 96, generator=g)
        sd[q + 'input_layernorm.weight'] = torch.randn(256, generator=g)
        sd[q + 'post_attention_layernorm.weight'] = torch.randn(256, generator=g)
    stack = LlamaTrainStack(cfg, sd, 'cpu')
    out = stack.state_dict()
    assert set(out) == set(sd) and all(torch.equal(out[k], sd[k]) for k in sd)
    assert stack.w[0]['wqkv'].dtype == torch.bfloat16 and stack.w[0]['wqkv'].shape == (768, 256)


def test_apply_delta_follows_the_reference_script():
    """scripts/apply_delta.py:21-40: equal shapes add, embed / lm_head add into the leading block, projector / SPI tensors
    pass through, anything else missing from the base raises NameError."""
    import pytest
    import torch
    from gpt4roi_b200.train import apply_delta
    base = {'model.layers.0.self_attn.q_proj.weight': torch.ones(4, 4), 'model.embed_tokens.weight': torch.ones(10, 4),
            'lm_head.weight': torch.full((10, 4), 2.0)}
    delta = {'model.layers.0.self_attn.q_proj.weight': torch.full((4, 4), 0.5), 'model.embed_tokens.weight': torch.zeros(16, 4),
             'lm_head.weight': torch.zeros(16, 4), 'model.mm_projector.weight': torch.full((4, 2), 3.0),
             'model.spi_module.roi_align.updims.bias': torch.full((4,), 7.0)}
    out = apply_delta(base, delta)
    assert torch.equal(out['model.layers.0.self_attn.q_proj.weight'], torch.full((4, 4), 1.5))
    assert torch.equal(out['model.embed_tokens.weight'][:10], torch.ones(10, 4)) and out['model.embed_tokens.weight'][10:].abs().sum() == 0
    assert torch.equal(out['lm_head.weight'][:10], torch.full((10, 4), 2.0))
    assert torch.equal(out['model.mm_projector.weight'], torch.full((4, 2), 3.0))
    assert torch.equal(out['model.spi_module.roi_align.updims.bias'], torch.full((4,), 7.0))
    with pytest.raises(NameError):
        apply_delta(base, {'model.layers.9.foo': torch.zeros(1)})


def test_save_checkpoint_writes_config_and_is_rank0_only(tmp_path):
    import json
    import torch
    from gpt4roi_b200 import train
    sd = {'a.weight': torch.arange(6.0).view(2, 3)}
    fused = torch.arange(12.0)
    sd['view'] = fused[:4]                                    # a view of a larger storage must not drag all of it along
    assert train.save_checkpoint(sd, str(tmp_path / 'r1'), rank=1) == []
    assert not (tmp_path / 'r1').exists()
    names = train.save_checkpoint(sd, str(tmp_path / 'r0'), config=dict(model_type='llava', hidden_size=4096), rank=0)
    assert json.load(open(tmp_path / 'r0' / 'config.json'))['model_type'] == 'llava'
    back = train.load_checkpoint(str(tmp_path / 'r0'))
    assert torch.equal(back['view'], fused[:4]) and back['view'].untyped_storage().nbytes() == 16
    assert (tmp_path / 'r0' / names[0]).stat().st_size < 4000


def test_stage1_to_stage2_bootstrap_follows_the_script(tmp_path):
    """train_stage2.sh:10-24: checkpoint-0 with links to the stage-1 files minus optimizer / scheduler / trainer state;
    a non-empty stage-2 dir resumes from its newest checkpoint instead."""
    import torch
    from gpt4roi_b200 import train
    s1, s2 = tmp_path / 'stage1', tmp_path / 'stage2'
    sd = {'a.weight': torch.arange(4.0)}
    train.save_checkpoint(sd, str(s1), config=dict(model_type='llava'), rank=0)
    for junk in ('optimizer.pt', 'scheduler.pt', 'trainer_state.json', 'training_args.bin'):
        (s1 / junk).write_bytes(b'x')
    s2.mkdir()
    ck = train.bootstrap_stage2(str(s1), str(s2))
    assert ck.endswith('checkpoint-0')
    names = sorted(p.name for p in (s2 / 'checkpoint-0').iterdir())
    assert 'config.json' in names and 'pytorch_model.bin.index.json' in names and not ({'optimizer.pt', 'scheduler.pt'} & set(names))
    assert all((s2 / 'checkpoint-0' / n).is_symlink() for n in names)
    assert torch.equal(train.load_checkpoint(ck)['a.weight'], sd['a.weight'])
    (s2 / 'checkpoint-3000').mkdir()
    assert train.bootstrap_stage2(str(s1), str(s2)).endswith('checkpoint-3000')
