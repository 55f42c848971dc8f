"""not gpu: the oracles of the caller-side networks (SURVEY.md section 8 rows f3 / f4) against the golden vectors written by the
UNMODIFIED reference (oracle/gen_golden.py); plus the host logic of the RealESRGANer front-end (tile plan, padding, colour
handling) against the reference's."""
import numpy as np
import pytest
import torch

import codeformer_b200 as cb
from codeformer_b200 import spec as S
from oracle import gen_golden as GG
from oracle import rrdbnet_oracle as RO
from tests.util import golden, maxabs

torch.set_grad_enabled(False)


@pytest.mark.parametrize('case', ['s2', 's4'])
def test_rrdbnet_oracle_matches_reference_golden(case):
    scale, sd, x = GG.rrdb_inputs(case)
    out = RO.rrdbnet_forward(sd, x, scale=scale, num_block=23)
    ref = golden('rrdbnet.npz')[case + '_out']
    assert out.shape == ref.shape
    assert maxabs(out, ref) < 2e-5, 'fp32 CPU restatement vs the reference module (thread-count noise only)'


def test_rrdbnet_state_dict_contract():
    """Same keys, shapes and order as the reference class: a reference checkpoint loads strictly."""
    ours = cb.ARCH_REGISTRY.get('RRDBNet')(3, 3, scale=2, num_feat=64, num_block=23, num_grow_ch=32)
    assert list(ours.state_dict().keys()) == list(S.rrdbnet_spec(3, 3, 2, 64, 23, 32).keys())
    ours.load_state_dict(S.random_state_dict(S.rrdbnet_spec(3, 3, 2, 64, 23, 32), 5), strict=True)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        ours(torch.zeros(1, 3, 8, 8))
    g = golden('reference_checks.npz')
    mine = ours.state_dict()
    assert list(g['rrdbnet_keys']) == list(mine.keys())
    assert list(g['rrdbnet_shapes']) == [','.join(map(str, v.shape)) for v in mine.values()]


_Toy = GG.ToyUpsampler


@pytest.mark.parametrize('tile,pre_pad,shape', GG.ESR_CASES)
def test_realesrganer_front_end_equals_the_reference(tile, pre_pad, shape):
    """enhance(): colour handling, reflect pre/mod padding, the tile loop and the crop-back, bit for bit against the
    reference's RealESRGANer around the same (CPU) model (realesrgan_utils.py:71-250; tests/golden/reference_checks.npz)."""
    model = _Toy().eval()
    ours = cb.RealESRGANer(scale=2, model_path=None, model=model, tile=tile, tile_pad=6, pre_pad=pre_pad, device='cpu')
    o1, m1 = ours.enhance(GG.esr_image(shape), outscale=2)
    g = golden('reference_checks.npz')
    o2, m2 = g[GG.esr_key(tile, pre_pad, shape)], str(g[GG.esr_key(tile, pre_pad, shape) + '_mode'])
    assert m1 == m2 and o1.dtype == o2.dtype and o1.shape == o2.shape
    assert np.array_equal(o1, o2)


def test_tile_plan_covers_the_image_once():
    er = cb.RealESRGANer(scale=2, model=_Toy(), tile=16, tile_pad=6, pre_pad=0, device='cpu')
    H, W = 37, 45
    cover = np.zeros((H * 2, W * 2), np.int32)
    for t in er.tile_plan(H, W):
        py0, py1, px0, px1 = t['in']
        oy0, oy1, ox0, ox1 = t['out']
        cy0, cy1, cx0, cx1 = t['crop']
        assert 0 <= py0 < py1 <= H and 0 <= px0 < px1 <= W
        assert (cy1 - cy0, cx1 - cx0) == (oy1 - oy0, ox1 - ox0) and cy1 <= (py1 - py0) * 2 and cx1 <= (px1 - px0) * 2
        cover[oy0:oy1, ox0:ox1] += 1
    assert (cover == 1).all()


def test_parsenet_oracle_matches_reference_golden():
    from codeformer_b200 import parsing as P
    from oracle import parsenet_oracle as PO
    sd, x = GG.parsenet_inputs()
    mask, img = PO.parsenet_forward(sd, x, P.parsenet_plan(512, 512)[0])
    g = golden('parsenet.npz')
    assert maxabs(mask[..., ::4, ::4], g['mask_s4']) < 2e-5 and maxabs(img[..., ::8, ::8], g['img_s8']) < 2e-5
    sure = torch.from_numpy(g['margin'].astype(np.float32)) > 1e-3
    assert torch.equal(mask.argmax(1)[sure], torch.from_numpy(g['classes']).long()[sure])


def test_parsenet_state_dict_contract():
    from codeformer_b200 import parsing as P
    net = cb.ParseNet(in_size=512, out_size=512, parsing_ch=19)
    spec = P.parsenet_spec(512, 512, 32, 64, 19, 10, (32, 256))
    sd = net.state_dict()
    assert list(sd.keys()) == list(spec.keys()) and len(sd) == 238
    assert all(tuple(sd[k].shape) == spec[k][0] and sd[k].dtype == spec[k][1] for k in sd)
    net.load_state_dict(P.random_parsenet_state_dict(spec, 2), strict=True)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        net.eval()(torch.zeros(1, 3, 64, 64))
    with pytest.raises(RuntimeError, match='inference-only'):
        net.train()
    g = golden('reference_checks.npz')
    assert list(g['parsenet_keys']) == list(sd.keys())
    assert list(g['parsenet_shapes']) == [','.join(map(str, v.shape)) for v in sd.values()]
    assert list(g['parsenet_dtypes']) == [str(v.dtype) for v in sd.values()]
