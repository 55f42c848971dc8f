"""The oracle (oracle/codeformer_oracle.py) against the golden vectors produced by the UNMODIFIED
reference (oracle/gen_golden.py)."""
import numpy as np
import pytest
import torch

from tests.util import faces_input, golden, maxabs, vq_micro_inputs
from oracle import codeformer_oracle as O
from oracle import gen_golden as GG
from codeformer_b200 import spec as S

torch.set_grad_enabled(False)


@pytest.fixture(scope='module')
def sd_main():
    return S.random_state_dict(S.codeformer_spec(), 1)


def test_main_config_matches_reference_golden(sd_main):
    g = golden('codeformer_main.npz')
    x = faces_input(slice(0, 1))
    out, logits, lq = O.codeformer_forward(sd_main, x, w=0.5, adain_on=True)
    # same torch build => only thread-order noise (reference: 3e-5 on out, 3e-6 on logits, SURVEY.md §4)
    assert maxabs(out, g['out']) < 2e-4
    assert maxabs(logits, g['logits']) < 2e-5
    assert maxabs(lq, g['lq_feat']) < 2e-5
    assert np.array_equal(logits.argmax(2).numpy(), g['top_idx'])


def test_variants_match_reference_golden(sd_main):
    g = golden('codeformer_variants.npz')
    x = faces_input(slice(1, 2))
    o, l, q = O.codeformer_forward(sd_main, x, w=0, adain_on=True)
    assert maxabs(o[..., ::4, ::4], g['w0_out']) < 2e-4 and np.array_equal(l.argmax(2).numpy(), g['w0_idx'])
    o, l, q = O.codeformer_forward(sd_main, x, w=1.0, adain_on=False)
    assert maxabs(o[..., ::4, ::4], g['w1_out']) < 2e-4 and np.array_equal(l.argmax(2).numpy(), g['w1_idx'])
    l, q = O.codeformer_forward(sd_main, x, w=0, code_only=True)
    assert maxabs(l[0, :4], g['code_only_logits_row0']) < 2e-5
    sd3 = S.random_state_dict(S.codeformer_spec(connect_list=('32', '64', '128')), 3)
    o, l, q = O.codeformer_forward(sd3, x, w=0.7, adain_on=True, connect_list=('32', '64', '128'))
    assert maxabs(o[..., ::4, ::4], g['c3_out']) < 2e-4 and np.array_equal(l.argmax(2).numpy(), g['c3_idx'])
    sd5 = S.random_state_dict(S.codeformer_spec(codebook_size=512, connect_list=('32', '64', '128')), 4)
    o, l, q = O.codeformer_forward(sd5, x, w=1, adain_on=False, connect_list=('32', '64', '128'))
    assert maxabs(o[..., ::4, ::4], g['k512_out']) < 2e-4 and np.array_equal(l.argmax(2).numpy(), g['k512_idx'])


def test_vqae_matches_reference_golden():
    g = golden('vqae.npz')
    sd = S.random_state_dict(S.vqae_spec(), 2)
    o, loss, st = O.vqae_forward(sd, faces_input(slice(0, 1)))
    assert maxabs(o[..., ::4, ::4], g['out']) < 2e-4
    assert np.array_equal(st['min_encoding_indices'].numpy(), g['idx'])
    assert abs(float(loss) - float(g['loss'])) < 1e-5
    assert abs(float(st['perplexity']) - float(g['perplexity'])) < 1e-3


@pytest.mark.parametrize('case', ['B', 'C'])
def test_vq_micro_matches_reference_golden(case):
    g = golden('vq_micro.npz')
    E, z = vq_micro_inputs(case)
    zq, loss, st = O.vq_forward({'quantize.embedding.weight': E}, z)
    assert np.array_equal(st['min_encoding_indices'].numpy(), g[f'{case}_idx'])
    assert maxabs(zq[0], g[f'{case}_zq_b0']) == 0.0
    assert abs(float(loss) - float(g[f'{case}_loss'])) < 1e-5 * max(1.0, float(g[f'{case}_loss']))


def test_oracle_equals_live_reference_small():
    """The restatement against the reference modules on a cheap case: VectorQuantizer on 4 latents + one TransformerSALayer
    (tests/golden/reference_checks.npz)."""
    g = golden('reference_checks.npz')
    E, z = vq_micro_inputs('B')
    zq, _, st = O.vq_forward({'quantize.embedding.weight': E}, z[:4])
    assert np.array_equal(st['min_encoding_indices'].numpy(), g['vq4_idx'])
    assert np.array_equal(zq.reshape(-1)[torch.from_numpy(g['vq4_sample_at'])].numpy(), g['vq4_zq_sample'])
    sd, t, pos = GG.transformer_layer_inputs()
    assert maxabs(O.transformer_layer(sd, 'L', t, pos, 8)[::16], g['sa_layer_out_s16']) < 5e-6


def test_plumbing_matches_reference_golden():
    """SURVEY section 8 f1: img2tensor+normalize and tensor2img of the reference, bit for bit (tests/golden/plumbing.npz)."""
    from oracle import plumbing_oracle as P
    g = golden('plumbing.npz')
    assert sorted(np.unique(g['face_bgr'])) == list(range(256))            # every byte value is exercised
    assert np.array_equal(P.face_to_input(g['face_bgr'][None])[0], g['x'])
    assert np.array_equal(P.output_to_face(g['out'])[0], g['restored_bgr'])
    # round trip of the fallback path (inference_codeformer.py:209-211): plumbing back and forth is the identity on u8
    assert np.array_equal(P.output_to_face(P.face_to_input(g['face_bgr'][None])), g['face_bgr'][None])


def test_plumbing_equals_live_reference():
    """img2tensor+normalize and tensor2img of the reference on a random 32x48 face (tests/golden/reference_checks.npz)."""
    from oracle import plumbing_oracle as P
    g = golden('reference_checks.npz')
    face, out = GG.plumbing_small_inputs()
    assert np.array_equal(g['plumbing_small_x'], P.face_to_input(face[None])[0])
    assert np.array_equal(g['plumbing_small_restored'], P.output_to_face(out)[0])
