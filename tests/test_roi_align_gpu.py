"""GPU parity tests for the RoIAlign kernels, through the C ABI (ctypes) only.

Bars (SURVEY.md 8(c)): indices/weights/fp32 outputs BIT-EXACT vs the oracle (= the
reference CPU kernel, no FMA); fp16/bf16 maps: fp32 accumulate, one rounding on store
(<= 1 ulp of the output dtype vs the fp32 oracle result); backward uses atomics (as the reference kernel
does: the summation order differs run to run), so rtol 1e-5 + atol 2e-5 (fp32; the atol covers elements whose
contributions cancel) + the mmcv gradient vectors at atol 1e-3.
"""
import numpy as np
import pytest
import torch

import gpt4roi_b200 as g
from oracle import roi_align_oracle as O
from tests.helpers import PYRAMID, SCALES, load_kat, load_ref_cases, make_rois

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _t(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


# ---- reference's own known-answer test, run through the drop-in operator ---------------
@pytest.mark.parametrize('dtype', [torch.float, torch.double, torch.half])
def test_mmcv_known_answers_forward_backward(dtype):
    """Same checks as mmcv-1.4.7/tests/test_ops/test_roi_align.py:67-104 (device='cuda')."""
    kat = load_kat()
    for case in kat['cases']:
        x = torch.tensor(case['input'], dtype=dtype, device=DEV, requires_grad=True)
        rois = torch.tensor(case['rois'], dtype=dtype, device=DEV)
        out = g.roi_align(x, rois, (kat['pool_h'], kat['pool_w']), kat['spatial_scale'],
                          kat['sampling_ratio'], 'avg', True)
        out.backward(torch.ones_like(out))
        assert np.allclose(out.data.float().cpu().numpy(), np.array(case['output']), atol=1e-3)
        assert np.allclose(x.grad.data.float().cpu().numpy(), np.array(case['grad_input']), atol=1e-3)
        if dtype in (torch.float, torch.double):  # exact for fp32/fp64
            assert np.array_equal(out.data.cpu().numpy(), np.array(case['output'], dtype=out.data.cpu().numpy().dtype))


def test_mmcv_gradcheck_double():
    """mmcv-1.4.7/tests/test_ops/test_roi_align.py:41-64."""
    kat = load_kat()
    for case in kat['cases']:
        x = torch.tensor(case['input'], dtype=torch.double, device=DEV, requires_grad=True)
        rois = torch.tensor(case['rois'], dtype=torch.double, device=DEV)
        layer = g.RoIAlign((kat['pool_h'], kat['pool_w']), kat['spatial_scale'], kat['sampling_ratio'])
        assert torch.autograd.gradcheck(layer, (x, rois), eps=1e-5, atol=1e-5)


def test_mmcv_ext_module_as_the_reference_wrapper_calls_it():
    """The `mmcv._ext` drop-in module (gpt4roi_b200.mmcv_ext, what `install()` registers), called exactly the way the
    reference's own wrapper calls it -- mmcv-1.4.7/mmcv/ops/roi_align.py:83-96 (forward: `new_zeros` output / argmax
    buffers, five positional tensors, six keyword scalars) and :113-123 (backward) -- on the mmcv known-answer cases and on
    a pyramid-sized fp32 case against the oracle (bit-exact forward).  tests/test_abi_cpu.py replays the calls recorded
    from the reference's actual wrapper (tests/golden/mmcv_wrapper_calls.json) against the same module."""
    from gpt4roi_b200 import mmcv_ext
    ext = mmcv_ext.make_module()
    kat = load_kat()
    for case in kat['cases']:
        x = torch.tensor(case['input'], dtype=torch.float, device=DEV)
        rois = torch.tensor(case['rois'], dtype=torch.float, device=DEV)
        out_h, out_w = kat['pool_h'], kat['pool_w']
        output = x.new_zeros((rois.size(0), x.size(1), out_h, out_w))
        argmax_y, argmax_x = x.new_zeros(0), x.new_zeros(0)                      # pool_mode 'avg': roi_align.py:88-90
        ext.roi_align_forward(x, rois, output, argmax_y, argmax_x, aligned_height=out_h, aligned_width=out_w,
                              spatial_scale=kat['spatial_scale'], sampling_ratio=kat['sampling_ratio'], pool_mode=1,
                              aligned=True)
        assert np.array_equal(output.cpu().numpy(), np.array(case['output'], dtype=np.float32))
        grad_output = torch.ones_like(output)
        grad_input = grad_output.new_zeros(x.shape)
        ext.roi_align_backward(grad_output, rois, argmax_y, argmax_x, grad_input, aligned_height=out_h,
                               aligned_width=out_w, spatial_scale=kat['spatial_scale'],
                               sampling_ratio=kat['sampling_ratio'], pool_mode=1, aligned=True)
        assert np.allclose(grad_input.cpu().numpy(), np.array(case['grad_input']), atol=1e-3)
    rng = np.random.default_rng(5)
    xin = rng.standard_normal((2, 64, 48, 48)).astype(np.float32)
    rois_np = make_rois(rng, 2, 6, 336.0)                                    # 2 images x 6 boxes
    want, _, _ = O.roi_align_forward(xin, rois_np, 14, SCALES[2], 2, 'avg', True)
    x, rois = _t(xin), _t(rois_np)
    output = x.new_zeros((12, 64, 14, 14))
    ext.roi_align_forward(x, rois, output, x.new_zeros(0), x.new_zeros(0), aligned_height=14, aligned_width=14,
                          spatial_scale=SCALES[2], sampling_ratio=2, pool_mode=1, aligned=True)
    assert np.array_equal(output.cpu().numpy(), want)
    with pytest.raises(NotImplementedError):
        ext.nms(x, rois)                                                       # not on the region-token path: loud


# ---- committed golden fixtures (outputs of the reference kernel itself) -----------------
def test_golden_reference_cases_nchw_bit_exact():
    z, meta = load_ref_cases()
    for m in meta:
        n = m['name']
        x, rois = _t(z[n + '.input']), _t(z[n + '.rois'])
        out = x.new_zeros(z[n + '.output'].shape)
        pm = 0 if m['pool_mode'] == 'max' else 1
        ay = x.new_zeros(out.shape) if pm == 0 else x.new_zeros(0)
        ax = x.new_zeros(out.shape) if pm == 0 else x.new_zeros(0)
        g.roi_align_forward(x, rois, out, ay, ax, aligned_height=m['PH'], aligned_width=m['PW'],
                            spatial_scale=m['spatial_scale'], sampling_ratio=m['sampling_ratio'],
                            pool_mode=pm, aligned=m['aligned'])
        assert np.array_equal(out.cpu().numpy(), z[n + '.output']), n
        if pm == 0:
            assert np.array_equal(ay.cpu().numpy(), z[n + '.argmax_y']), n
            assert np.array_equal(ax.cpu().numpy(), z[n + '.argmax_x']), n
        gi = x.new_zeros(x.shape)
        g.roi_align_backward(_t(z[n + '.grad_output']), rois, ay, ax, gi, aligned_height=m['PH'],
                             aligned_width=m['PW'], spatial_scale=m['spatial_scale'],
                             sampling_ratio=m['sampling_ratio'], pool_mode=pm, aligned=m['aligned'])
        np.testing.assert_allclose(gi.cpu().numpy(), z[n + ".grad_input"], rtol=1e-5, atol=2e-5, err_msg=n)


def test_golden_reference_cases_nhwc_bit_exact():
    z, meta = load_ref_cases()
    for m in meta:
        if m['pool_mode'] != 'avg' or m['C'] % 4:
            continue
        n = m['name']
        x = _t(z[n + '.input'].transpose(0, 2, 3, 1))
        out = g.roi_align_mlvl([x], _t(z[n + '.rois']), (m['PH'], m['PW']), [m['spatial_scale']],
                               sampling_ratio=m['sampling_ratio'], aligned=m['aligned'])
        got = out[0].permute(0, 3, 1, 2).cpu().numpy()
        assert np.array_equal(got, z[n + '.output']), n


# ---- seeded parity vs the oracle at hot-path shapes --------------------------------------
@pytest.mark.parametrize('size', [224, 336])
@pytest.mark.parametrize('ph', [14, 7])
def test_mlvl_forward_fp32_bit_exact_vs_oracle(size, ph):
    rng = np.random.default_rng(size + ph)
    N, C = 2, 64
    rois = make_rois(rng, N, 4, size, adversarial=True)
    maps = [rng.standard_normal((N, h, h, C)).astype(np.float32) for h in PYRAMID[size]]
    out = g.roi_align_mlvl([_t(m) for m in maps], _t(rois), ph, SCALES, sampling_ratio=2)
    out = out.cpu().numpy()
    for l, m in enumerate(maps):
        want, _, _ = O.roi_align_forward(m, rois, ph, SCALES[l], 2, 'avg', True, in_layout=O.NHWC,
                                         out_layout=O.NHWC)
        assert np.array_equal(out[l], want), 'level %d' % l


def test_mlvl_adaptive_sampling_bit_exact_vs_oracle():
    rng = np.random.default_rng(11)
    N, C = 2, 16
    rois = make_rois(rng, N, 5, 224, adversarial=True)
    maps = [rng.standard_normal((N, h, h, C)).astype(np.float32) for h in (32, 16)]
    out = g.roi_align_mlvl([_t(m) for m in maps], _t(rois), (5, 3), SCALES[2:], sampling_ratio=0).cpu().numpy()
    for l, m in enumerate(maps):
        want, _, _ = O.roi_align_forward(m, rois, (5, 3), SCALES[2 + l], 0, 'avg', True, O.NHWC, O.NHWC)
        assert np.array_equal(out[l], want)


@pytest.mark.parametrize('dtype', [torch.bfloat16, torch.float16])
def test_mlvl_forward_16bit_one_rounding(dtype):
    """16-bit maps: taps widened exactly, fp32 accumulate in reference order, ONE rounding."""
    rng = np.random.default_rng(5)
    N, C, size = 2, 64, 336
    rois = make_rois(rng, N, 4, size, adversarial=True)
    maps_t = [torch.from_numpy(rng.standard_normal((N, h, h, C)).astype(np.float32)).to(dtype) for h in PYRAMID[size]]
    out16 = g.roi_align_mlvl([m.to(DEV) for m in maps_t], _t(rois), 14, SCALES, sampling_ratio=2)
    out32 = g.roi_align_mlvl([m.to(DEV) for m in maps_t], _t(rois), 14, SCALES, sampling_ratio=2,
                             out_dtype=torch.float32)
    for l, m in enumerate(maps_t):
        want, _, _ = O.roi_align_forward(m.float().numpy(), rois, 14, SCALES[l], 2, 'avg', True, O.NHWC, O.NHWC)
        assert np.array_equal(out32[l].cpu().numpy(), want)                  # fp32 result exact
        assert torch.equal(out16[l].cpu(), torch.from_numpy(want).to(dtype))  # single RN rounding


def test_nchw_forward_max_and_double_vs_oracle():
    rng = np.random.default_rng(8)
    x = rng.standard_normal((2, 6, 24, 24))
    rois = make_rois(rng, 2, 6, 336, adversarial=True).astype(np.float64)
    for mode, sr in (('max', 2), ('avg', 0), ('max', 0)):
        want, way, wax = O.roi_align_forward(x, rois, 7, SCALES[3], sr, mode, True)
        xt, rt = _t(x), _t(rois)
        out = xt.new_zeros(want.shape)
        pm = 0 if mode == 'max' else 1
        ay = xt.new_zeros(want.shape) if pm == 0 else xt.new_zeros(0)
        ax = xt.new_zeros(want.shape) if pm == 0 else xt.new_zeros(0)
        g.roi_align_forward(xt, rt, out, ay, ax, 7, 7, SCALES[3], sr, pm, True)
        assert np.array_equal(out.cpu().numpy(), want)
        if pm == 0:
            assert np.array_equal(ay.cpu().numpy(), way) and np.array_equal(ax.cpu().numpy(), wax)


def test_mlvl_backward_vs_oracle():
    rng = np.random.default_rng(9)
    N, C, size = 2, 32, 224
    rois = make_rois(rng, N, 6, size, adversarial=True)
    shapes = [(N, h, h, C) for h in PYRAMID[size]]
    go = rng.standard_normal((4, len(rois), 14, 14, C)).astype(np.float32)
    grads = g.roi_align_mlvl_backward(_t(go), _t(rois), shapes, SCALES, 2)
    for l, s in enumerate(shapes):
        want = O.roi_align_backward(go[l], rois, s, SCALES[l], 2, 'avg', True, in_layout=O.NHWC,
                                    out_layout=O.NHWC)
        np.testing.assert_allclose(grads[l].cpu().numpy(), want, rtol=1e-4, atol=2e-5)


def test_mlvl_fused_groupnorm_relu_taps():
    """Optional per-tap affine+ReLU == applying it to the map first (floating point: 1e-6)."""
    rng = np.random.default_rng(10)
    N, C = 2, 32
    rois = make_rois(rng, N, 4, 224)
    maps = [torch.from_numpy(rng.standard_normal((N, h, h, C)).astype(np.float32)).to(DEV) for h in (32, 16)]
    sc = [torch.rand(N, C, device=DEV) + 0.5 for _ in maps]
    sh = [torch.randn(N, C, device=DEV) * 0.1 for _ in maps]
    fused = g.roi_align_mlvl(maps, _t(rois), 14, SCALES[2:], 2, gn_scale=sc, gn_shift=sh)
    pre = [torch.relu(m * a[:, None, None, :] + b[:, None, None, :]) for m, a, b in zip(maps, sc, sh)]
    plain = g.roi_align_mlvl(pre, _t(rois), 14, SCALES[2:], 2)
    torch.testing.assert_close(fused, plain, rtol=1e-6, atol=1e-6)


def test_empty_and_error_behaviour():
    x = torch.zeros(1, 8, 4, 4, device=DEV)
    out = g.roi_align(x, torch.zeros(0, 5, device=DEV), 2, 1.0, 2, 'avg', True)
    assert out.shape == (0, 8, 2, 2)
    with pytest.raises(RuntimeError):   # dtype mismatch rois vs input (roi_align_cuda.cu:22)
        g.roi_align(x, torch.zeros(1, 5, device=DEV, dtype=torch.half), 2, 1.0, 2, 'avg', True)
    with pytest.raises(RuntimeError):   # tensors on different devices
        g.roi_align(x, torch.zeros(1, 5), 2, 1.0, 2, 'avg', True)
    with pytest.raises(RuntimeError):   # C not a multiple of the 128-bit vector
        g.roi_align_mlvl([torch.zeros(1, 4, 4, 6, device=DEV)], torch.zeros(1, 5, device=DEV), 2, [1.0])


# ---- full-size, size-independent properties (BASELINE config-5 / config-2 shapes) ---------
def test_full_size_properties():
    torch.manual_seed(0)
    rng = np.random.default_rng(12)
    N, C, size, kpi = 8, 1024, 336, 8
    rois = _t(make_rois(rng, N, kpi, size))
    maps = [torch.randn(N, h, h, C, device=DEV) for h in PYRAMID[size]]
    a = g.roi_align_mlvl(maps, rois, 14, SCALES, 2)
    # determinism / idempotence
    assert torch.equal(a, g.roi_align_mlvl(maps, rois, 14, SCALES, 2))
    # linearity in the maps (fp32; averaging is linear): f(2x) == 2 f(x) exactly (power of two)
    assert torch.equal(g.roi_align_mlvl([m * 2 for m in maps], rois, 14, SCALES, 2), a * 2)
    # constant map -> every bin equals the constant wherever all samples are in range
    ones = [torch.full_like(m, 3.0) for m in maps]
    c = g.roi_align_mlvl(ones, rois, 14, SCALES, 2)
    assert torch.allclose(c, torch.full_like(c, 3.0), atol=1e-5)
    # permutation equivariance over RoIs
    perm = torch.randperm(rois.shape[0], device=DEV)
    assert torch.equal(g.roi_align_mlvl(maps, rois[perm].contiguous(), 14, SCALES, 2), a[:, perm])
    # spot-check a slice of the big result against the oracle
    sel = [0, 17, 40, 63]
    for l in (0, 3):
        want, _, _ = O.roi_align_forward(maps[l][..., :8].contiguous().cpu().numpy(), rois[sel].cpu().numpy(),
                                         14, SCALES[l], 2, 'avg', True, O.NHWC, O.NHWC)
        assert np.array_equal(a[l][sel][..., :8].cpu().numpy(), want)


# ---- NCHW drop-in, large-work fast path (transpose -> NHWC kernel -> transpose) ---------
@pytest.mark.parametrize('dtype', [torch.float32, torch.float16, torch.bfloat16])
def test_nchw_fast_path_is_bit_identical_to_the_direct_kernel(dtype):
    """Enough RoIs per map element for g4r_roi_align_forward_workspace() > 0: the operator then runs the three
    streaming passes; results must equal the direct NCHW kernel bit for bit (and the oracle for fp32), including
    adversarial boxes, adaptive sampling (sampling_ratio=0) and a non-square pooled size."""
    from gpt4roi_b200 import lib as L
    rng = np.random.default_rng(5)
    N, C, H, W = 3, 128, 24, 20
    x = torch.from_numpy(rng.standard_normal((N, C, H, W)).astype(np.float32)).to(DEV).to(dtype)
    rois_np = make_rois(rng, N, 60, 336, adversarial=True)
    rois_np[:, 1:] *= np.array([W / 336.0, H / 336.0, W / 336.0, H / 336.0], np.float32) * 14.0
    rois = torch.from_numpy(rois_np).to(DEV).to(dtype)
    K = rois.shape[0]
    e0 = x.new_zeros(0)
    for (ph, pw, sr) in ((7, 7, 2), (14, 14, 2), (5, 3, 0)):
        scale = float(np.float32(1 / 14.0))
        need = L.load().g4r_roi_align_forward_workspace(N, C, H, W, K, ph, pw, sr, 1, L.dtype_code(x), L.NCHW)
        assert need > 0, 'this configuration is meant to take the fast path'
        fast = x.new_zeros(K, C, ph, pw)
        g.roi_align_forward(x, rois, fast, e0, e0, ph, pw, scale, sr, 1, True)
        direct = x.new_zeros(K, C, ph, pw)
        with torch.cuda.device(DEV):
            L.check(L.load().g4r_roi_align_forward(L.ptr(x), L.ptr(rois), L.ptr(direct), None, None, N, C, H, W, K, ph, pw,
                                                   scale, sr, 1, 1, L.dtype_code(x), L.NCHW, L.stream_ptr(torch.device(DEV))))
        assert torch.equal(fast, direct), (dtype, ph, pw, sr)
        if dtype == torch.float32:
            want, _, _ = O.roi_align_forward(x.cpu().numpy(), rois_np, (ph, pw), scale, sr, 'avg', True)
            assert np.array_equal(fast.cpu().numpy(), want), (ph, pw, sr)
    # small problems keep the direct kernel (no workspace)
    assert L.load().g4r_roi_align_forward_workspace(1, 3, 4, 4, 1, 2, 2, 2, 1, 0, 0) == 0
    # max pooling is not on the fast path
    assert L.load().g4r_roi_align_forward_workspace(N, C, H, W, K, 7, 7, 2, 0, 0, 0) == 0
