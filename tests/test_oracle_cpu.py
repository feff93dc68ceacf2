"""CPU tests: pin the oracle (oracle/roi_align_oracle.c) against the reference's own
known-answer vectors and the committed golden fixtures (outputs of the reference kernel
compiled from its sources)."""
import json
import os

import numpy as np
import pytest

from oracle import roi_align_oracle as O
from tests.helpers import GOLDEN, load_kat, load_ref_cases, make_rois


@pytest.mark.parametrize('dtype', [np.float32, np.float64])
def test_oracle_reproduces_mmcv_known_answers(dtype):
    kat = load_kat()
    for case in kat['cases']:
        x = np.array(case['input'], dtype=dtype)
        rois = np.array(case['rois'], dtype=dtype)
        out, _, _ = O.roi_align_forward(x, rois, (kat['pool_h'], kat['pool_w']), kat['spatial_scale'],
                                        kat['sampling_ratio'], 'avg', True)
        # fp32/fp64 reproduce the literals exactly (they are dyadic rationals)
        assert np.array_equal(out, np.array(case['output'], dtype=dtype))
        gi = O.roi_align_backward(np.ones_like(out), rois, x.shape, kat['spatial_scale'],
                                  kat['sampling_ratio'], 'avg', True)
        assert np.array_equal(gi, np.array(case['grad_input'], dtype=dtype))


def test_oracle_matches_golden_reference_outputs_bit_exact():
    z, meta = load_ref_cases()
    assert len(meta) >= 10
    for m in meta:
        n = m['name']
        out, ay, ax = O.roi_align_forward(z[n + '.input'], z[n + '.rois'], (m['PH'], m['PW']),
                                          m['spatial_scale'], m['sampling_ratio'], m['pool_mode'],
                                          m['aligned'])
        assert np.array_equal(out, z[n + '.output']), n
        if m['pool_mode'] == 'max':
            assert np.array_equal(ay, z[n + '.argmax_y']), n
            assert np.array_equal(ax, z[n + '.argmax_x']), n
        gi = O.roi_align_backward(z[n + '.grad_output'], z[n + '.rois'], z[n + '.input'].shape,
                                  m['spatial_scale'], m['sampling_ratio'], m['pool_mode'], m['aligned'],
                                  ay, ax)
        assert np.array_equal(gi, z[n + '.grad_input']), n


def test_oracle_layouts_agree():
    rng = np.random.default_rng(1)
    x = rng.standard_normal((2, 6, 24, 24)).astype(np.float32)
    rois = make_rois(rng, 2, 5, 336, adversarial=True)
    a, _, _ = O.roi_align_forward(x, rois, 14, 1 / 14, 2, 'avg', True)
    b, _, _ = O.roi_align_forward(np.ascontiguousarray(x.transpose(0, 2, 3, 1)), rois, 14, 1 / 14, 2,
                                  'avg', True, in_layout=O.NHWC, out_layout=O.NHWC)
    assert np.array_equal(a, b.transpose(0, 3, 1, 2))
    g = rng.standard_normal(a.shape).astype(np.float32)
    ga = O.roi_align_backward(g, rois, x.shape, 1 / 14, 2, 'avg', True)
    gb = O.roi_align_backward(np.ascontiguousarray(g.transpose(0, 2, 3, 1)), rois, (2, 24, 24, 6), 1 / 14, 2,
                              'avg', True, in_layout=O.NHWC, out_layout=O.NHWC)
    assert np.array_equal(ga, gb.transpose(0, 3, 1, 2))


def test_oracle_rejects_negative_roi_like_reference():
    x = np.zeros((1, 1, 4, 4), np.float32)
    rois = np.array([[0, 3, 3, 1, 1]], np.float32)
    with pytest.raises(O.OracleError):
        O.roi_align_forward(x, rois, 2, 1.0, 2, 'avg', True)


def test_oracle_empty_rois():
    x = np.zeros((1, 2, 4, 4), np.float32)
    out, _, _ = O.roi_align_forward(x, np.zeros((0, 5), np.float32), 2, 1.0, 2, 'avg', True)
    assert out.shape == (0, 2, 2, 2)


def test_oracle_matches_live_reference_build():
    """The reference's cpu/roi_align.cpp compiled unmodified (oracle/_ref), run on seeded random + adversarial boxes
    (tests/golden/roi_align_adversarial_ref.npz, written by make_golden.py --adversarial): the oracle reproduces its
    outputs and argmax bit for bit."""
    z = np.load(os.path.join(GOLDEN, 'roi_align_adversarial_ref.npz'))
    meta = json.loads(bytes(z['meta']).decode())
    assert len(meta) == 3
    for m in meta:
        n = m['name']
        out, ay, ax = O.roi_align_forward(z[n + '.input'], z[n + '.rois'], m['PH'], m['spatial_scale'],
                                          m['sampling_ratio'], m['pool_mode'], True)
        assert np.array_equal(out, z[n + '.output']), n
        if m['pool_mode'] == 'max':
            assert np.array_equal(ay, z[n + '.argmax_y']) and np.array_equal(ax, z[n + '.argmax_x']), n


# ---------------------------------------------------------------------------------------
# splice oracle vs an independent torch restatement of the reference python loop
# ---------------------------------------------------------------------------------------
def _splice_torch(ids, emb, img, regions, P, tok):
    """Behavioural restatement of gpt4roi/models/spi_llava.py:99-196 (use_im_start_end branch)."""
    import torch
    outs = []
    for b in range(ids.shape[0]):
        cur_ids, cur = ids[b], emb[ids[b]]
        if (cur_ids == tok['patch']).sum() == 0:
            outs.append(cur)
            continue
        if (cur_ids == tok['start']).sum() != (cur_ids == tok['end']).sum():
            raise ValueError('The number of image start tokens and image end tokens should be the same.')
        new = None
        for s in torch.where(cur_ids == tok['start'])[0]:
            s = int(s)
            if cur_ids[s + P + 1] != tok['end']:
                raise ValueError('The image end token should follow the image start token.')
            new = torch.cat((cur[:s + 1], img[b], cur[s + P + 1:]), dim=0)
            spi = regions[b] if regions is not None else None
            if spi is not None:
                spi_embeds = torch.zeros_like(new)
                mask = cur_ids == tok['bbox']
                spi_embeds[mask] = spi.to(spi_embeds.dtype)
                new = new * (~mask).to(cur.dtype)[:, None] + spi_embeds
            else:
                assert (cur_ids == tok['bbox']).sum() == 0
        outs.append(new)
    return torch.stack(outs, 0)


def _mk_ids(rng, B, L, P, ks, tok, V):
    ids = rng.integers(3, V - 6, (B, L)).astype(np.int64)
    for b in range(B):
        ids[b, 1] = tok['start']
        ids[b, 2:2 + P] = tok['patch']
        ids[b, 2 + P] = tok['end']
        pos = rng.choice(np.arange(3 + P, L), size=ks[b], replace=False)
        ids[b, pos] = tok['bbox']
    return ids


def test_splice_oracle_matches_python_loop_semantics():
    import torch
    rng = np.random.default_rng(3)
    V, D, P, L, B = 64, 16, 9, 40, 4
    tok = dict(patch=V - 5, bbox=V - 4, start=V - 2, end=V - 1)
    ks = [3, 0, 1, 5]
    ids = _mk_ids(rng, B, L, P, ks, tok, V)
    ids[1, :] = rng.integers(3, V - 6, L)  # sample 1: text only (no image tokens)
    emb = torch.randn(V, D).to(torch.bfloat16)
    img = torch.randn(B, P, D).to(torch.bfloat16)
    regs = [torch.randn(k, D).to(torch.bfloat16) for k in ks]
    want = _splice_torch(torch.from_numpy(ids), emb, img, regs, P, tok)
    offs = np.concatenate([[0], np.cumsum(ks)]).astype(np.int32)
    u16 = lambda t: t.contiguous().view(torch.int16).numpy().view(np.uint16)
    got = O.splice(ids, u16(emb), u16(img), u16(torch.cat(regs, 0)), offs, P,
                   tok['patch'], tok['start'], tok['end'], tok['bbox'])
    got_t = torch.from_numpy(got.view(np.int16)).view(torch.bfloat16)
    assert torch.equal(got_t.float(), want.float())  # value equality (-0 == +0), see oracle header


def test_splice_oracle_error_codes():
    rng = np.random.default_rng(4)
    V, D, P, L, B = 64, 8, 4, 20, 1
    tok = dict(patch=V - 5, bbox=V - 4, start=V - 2, end=V - 1)
    emb = np.zeros((V, D), np.uint16)
    img = np.zeros((B, P, D), np.uint16)
    reg = np.zeros((2, D), np.uint16)
    offs = np.array([0, 2], np.int32)
    args = (P, tok['patch'], tok['start'], tok['end'], tok['bbox'])
    ids = _mk_ids(rng, B, L, P, [2], tok, V)
    O.splice(ids, emb, img, reg, offs, *args)
    bad = ids.copy(); bad[0, 2 + P] = 5
    with pytest.raises(ValueError, match='same'):
        O.splice(bad, emb, img, reg, offs, *args)
    bad = ids.copy(); bad[0, 2 + P] = 5; bad[0, L - 1] = tok['end']
    with pytest.raises(ValueError, match='follow'):
        O.splice(bad, emb, img, reg, offs, *args)
    with pytest.raises(ValueError, match='bbox'):
        O.splice(ids, emb, img, reg[:1], np.array([0, 1], np.int32), *args)
