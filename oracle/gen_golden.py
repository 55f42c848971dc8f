"""Generate tests/golden/*.npz from the UNMODIFIED reference (build container only).

TEST INFRASTRUCTURE.  Run:  PYTHONDONTWRITEBYTECODE=1 python oracle/gen_golden.py
Needs /root/reference (imported through oracle/ref_shim.py; never written to).  The
reference publishes no golden vectors (SURVEY.md §8c), so these files are what pins parity:
outputs of the reference's own nn.Modules on CPU fp32 (torch 2.11.0+cu128, 8 threads), with
the seeded parameters of codeformer_b200.spec.random_state_dict and committed input faces.

Files
  faces.npz                 4 of the reference's inputs/cropped_faces (RGB u8 [4,512,512,3]) -- data fixtures
  codeformer_main.npz       face 0, CodeFormer(w=0.5, adain=True): out, logits, lq_feat, top_idx   (config 1)
  codeformer_variants.npz   face 1: w=0 / w=1,adain=False / 3-connect colorization / codebook 512 inpainting;
                            `out` kept at stride 4 to stay small, logits argmax + lq_feat full
  vqae.npz                  face 0, VQAutoEncoder.forward: out (stride 4), indices, loss, perplexity, mean_distance
  vq_micro.npz              VectorQuantizer.forward on the config-3 inputs (seeded), indices + z_q samples + stats
  rrdbnet.npz               RRDBNet.forward (section 8 f4) of the reference, 23 blocks, scale 2 and scale 4, small seeded images
                            (`python oracle/gen_golden.py rrdbnet` regenerates only this file)
  parsenet.npz              ParseNet.forward (section 8 f3) of the reference, shipped 512 configuration, face 0
                            (`python oracle/gen_golden.py parsenet` regenerates only this file)
  plumbing.npz              the caller's image plumbing (section 8 f1): img2tensor(face/255.)+normalize and
                            tensor2img(min_max=(-1,1)).astype(uint8) of the reference on a u8 face that holds every byte
                            value in every channel and on an fp32 tensor that holds every rounding half-way point
                            (`python oracle/gen_golden.py plumbing` regenerates only this file)
  reference_checks.npz      small direct checks of the reference's own modules: state-dict keys and shapes of CodeFormer,
                            RRDBNet and ParseNet; VectorQuantizer on 4 config-3 latents; one TransformerSALayer (every 16th
                            token of its output); img2tensor/tensor2img on a 32x48 face; RealESRGANer.enhance around
                            ToyUpsampler for every ESR_CASES entry
                            (`python oracle/gen_golden.py reference_checks` regenerates only this file)
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim                      # noqa: E402
from codeformer_b200 import spec as S            # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')
FACES = ['0143.png', '0240.png', '0342.png', '0345.png']


def load_faces():
    import cv2
    imgs = []
    for f in FACES:
        img = cv2.imread(os.path.join(ref_shim.REF_ROOT, 'inputs', 'cropped_faces', f), cv2.IMREAD_COLOR)
        img = cv2.resize(img, (512, 512), interpolation=cv2.INTER_LINEAR)       # inference_codeformer.py:182
        imgs.append(cv2.cvtColor(img, cv2.COLOR_BGR2RGB))
    return np.stack(imgs).astype(np.uint8)


def to_input(faces_u8):
    """u8 RGB HWC -> f32 NCHW in [-1,1]; the arithmetic of inference_codeformer.py:199-200."""
    t = torch.from_numpy(faces_u8.astype(np.float32) / 255.).permute(0, 3, 1, 2).contiguous()
    return (t - 0.5) / 0.5


def vq_micro_inputs(case):
    g = torch.Generator().manual_seed(0)
    E = torch.randn(1024, 256, generator=g)
    if case == 'B':
        z = torch.randn(32, 256, 16, 16, generator=g)
    else:
        idx = torch.randint(0, 1024, (32 * 256,), generator=g)
        z = (E[idx] + 0.3 * torch.randn(32 * 256, 256, generator=g)).view(32, 16, 16, 256).permute(0, 3, 1, 2).contiguous()
    return E, z


def gen_plumbing():
    ref_shim.load()
    from basicsr.utils import img2tensor, tensor2img                      # basicsr/utils/img_util.py:9,38
    from torchvision.transforms.functional import normalize               # inference_codeformer.py:7
    rng = np.random.default_rng(7)
    face = rng.integers(0, 256, (64, 64, 3), dtype=np.uint8)              # BGR, as face_helper.cropped_faces
    ramp = np.arange(256, dtype=np.uint8).reshape(16, 16)
    face[:16, :16, 0], face[:16, :16, 1], face[:16, :16, 2] = ramp, ramp[::-1], ramp.T
    t = img2tensor(face / 255., bgr2rgb=True, float32=True)               # inference_codeformer.py:199
    normalize(t, (0.5, 0.5, 0.5), (0.5, 0.5, 0.5), inplace=True)          # :200
    out = (rng.standard_normal((1, 3, 64, 64)) * 0.7).astype(np.float32)  # some values beyond +-1: exercises the clamp
    k = np.arange(0, 255)
    half = ((k + 0.5) / 255 * 2 - 1).astype(np.float32)                   # (v+1)/2*255 = k + 0.5
    out.reshape(-1)[:255] = half
    out.reshape(-1)[255:510] = np.nextafter(half, np.float32(2))
    out.reshape(-1)[510:765] = np.nextafter(half, np.float32(-2))
    restored = tensor2img(torch.from_numpy(out.copy()), rgb2bgr=True, min_max=(-1, 1)).astype('uint8')   # :206,213
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, 'plumbing.npz'), face_bgr=face, x=t.numpy(), out=out, restored_bgr=restored)


RRDB_CASES = {            # name -> (scale, input shape, weight seed, input seed): the two RealESRGAN models of the reference
    's2': (2, (1, 3, 44, 36), 21, 31),      # set_realesrgan(): RRDBNet(3, 3, 64, 23, 32, scale=2)   inference_codeformer.py:41-48
    's4': (4, (2, 3, 20, 28), 22, 32),      # the x4 RealESRGAN model
}


def rrdb_inputs(case):
    scale, shape, wseed, xseed = RRDB_CASES[case]
    sd = S.random_state_dict(S.rrdbnet_spec(3, 3, scale, 64, 23, 32), wseed)
    x = torch.rand(shape, generator=torch.Generator().manual_seed(xseed))          # images in [0, 1] (realesrgan_utils.py:199)
    return scale, sd, x


def load_ref_rrdbnet():
    """The UNMODIFIED reference class (basicsr/archs/rrdbnet_arch.py) through the import shim."""
    ref_shim.load()
    from basicsr.archs.rrdbnet_arch import RRDBNet          # noqa: E402
    return RRDBNet


def gen_rrdbnet():
    """tests/golden/rrdbnet.npz: outputs of the reference RRDBNet (23 blocks) on small seeded inputs, both scales."""
    RRDBNet = load_ref_rrdbnet()
    out = {}
    torch.set_grad_enabled(False)
    for case in RRDB_CASES:
        scale, sd, x = rrdb_inputs(case)
        net = RRDBNet(3, 3, scale=scale, num_feat=64, num_block=23, num_grow_ch=32).eval()
        net.load_state_dict(sd, strict=True)
        out[case + '_out'] = net(x).numpy()
    np.savez_compressed(os.path.join(OUT, 'rrdbnet.npz'), **out)


def load_ref_parsenet():
    """The UNMODIFIED reference class (facelib/parsing/parsenet.py; imports only numpy / torch)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location('ref_parsenet', os.path.join(ref_shim.REF_ROOT, 'facelib', 'parsing', 'parsenet.py'))
    mod = importlib.util.module_from_spec(spec)
    sys.dont_write_bytecode = True
    spec.loader.exec_module(mod)
    return mod.ParseNet


def parsenet_inputs():
    """The shipped configuration (facelib/parsing/__init__.py:13) with seeded parameters, on committed face 0 in [-1,1]
    (face_restoration_helper.py:458-460)."""
    from codeformer_b200 import parsing as P
    sd = P.random_parsenet_state_dict(P.parsenet_spec(512, 512, 32, 64, 19, 10, (32, 256)), 41)
    faces = np.load(os.path.join(OUT, 'faces.npz'))['faces'][:1]
    return sd, to_input(faces)


def gen_parsenet():
    """tests/golden/parsenet.npz: ParseNet(512, 512, parsing_ch=19).eval() of the reference on face 0: logits at stride 4, the
    full-resolution argmax classes and the top-1/top-2 margin (index parity is asserted where the margin exceeds the noise)."""
    ParseNet = load_ref_parsenet()
    torch.set_grad_enabled(False)
    sd, x = parsenet_inputs()
    net = ParseNet(in_size=512, out_size=512, parsing_ch=19).eval()
    net.load_state_dict(sd, strict=True)
    mask, img = net(x)
    top2 = mask.topk(2, dim=1).values
    np.savez_compressed(os.path.join(OUT, 'parsenet.npz'), mask_s4=mask[..., ::4, ::4].numpy(), img_s8=img[..., ::8, ::8].numpy(),
                        classes=mask.argmax(1).numpy().astype(np.uint8), margin=(top2[:, 0] - top2[:, 1]).numpy().astype(np.float16))


class ToyUpsampler(torch.nn.Module):
    """A cheap x2 'upsampler' with a 5x5 receptive field: enough to make tiling / padding mistakes visible."""

    def __init__(self):
        super().__init__()
        g = torch.Generator().manual_seed(3)
        self.w = torch.nn.Parameter(torch.randn(3, 3, 5, 5, generator=g) * 0.1)

    def forward(self, x):
        y = torch.nn.functional.conv2d(x, self.w, padding=2)
        return torch.nn.functional.interpolate(y, scale_factor=2, mode='nearest')


ESR_CASES = [(0, 0, (37, 45, 3)), (16, 0, (37, 45, 3)), (16, 10, (50, 33, 3)), (20, 4, (41, 41)), (16, 0, (30, 34, 4))]   # tile, pre_pad, image shape


def esr_image(shape):
    return np.random.default_rng(7).integers(0, 256, shape, dtype=np.uint8)


def esr_key(tile, pre_pad, shape):
    return f'esr_t{tile}_p{pre_pad}_' + 'x'.join(map(str, shape))


def transformer_layer_inputs():
    """Seeded parameters of one TransformerSALayer(512, 8, 1024) (the ft_layers.0 entries of the CodeFormer spec, prefix 'L'),
    a [256, 2, 512] token sequence and its position embedding."""
    spec = S.codeformer_spec()
    sub = type(spec)((k, v) for k, v in spec.items() if k.startswith('ft_layers.0.'))
    sd = {'L.' + k[len('ft_layers.0.'):]: v for k, v in S.random_state_dict(sub, 3).items()}
    g = torch.Generator().manual_seed(3)
    t = torch.randn(256, 2, 512, generator=g)
    pos = torch.randn(256, 2, 512, generator=g) * 0.02
    return sd, t, pos


def plumbing_small_inputs():
    """A random 32x48 BGR face and a [1,3,32,48] network output (values beyond +-1 included)."""
    rng = np.random.default_rng(11)
    face = rng.integers(0, 256, (32, 48, 3), dtype=np.uint8)
    out = (rng.standard_normal((1, 3, 32, 48)) * 0.8).astype(np.float32)
    return face, out


def state_dict_table(sd):
    """-> (keys, shapes as 'd0,d1,...', dtypes) string arrays of a state dict."""
    return (np.array(list(sd.keys())), np.array([','.join(map(str, v.shape)) for v in sd.values()]),
            np.array([str(v.dtype) for v in sd.values()]))


def gen_reference_checks():
    """tests/golden/reference_checks.npz: what the tests used to compare against the reference modules imported live."""
    CodeFormer, _, VQ, _ = ref_shim.load()
    torch.set_grad_enabled(False)
    res = {}
    for name, net in (('codeformer', CodeFormer()),
                      ('rrdbnet', load_ref_rrdbnet()(3, 3, scale=2, num_feat=64, num_block=23, num_grow_ch=32)),
                      ('parsenet', load_ref_parsenet()(in_size=512, out_size=512, parsing_ch=19))):
        res[name + '_keys'], res[name + '_shapes'], res[name + '_dtypes'] = state_dict_table(net.state_dict())

    E, z = vq_micro_inputs('B')
    m = VQ(1024, 256, 0.25)
    m.embedding.weight.data.copy_(E)
    zq, _, st = m(z[:4])
    sample = np.sort(np.random.default_rng(0).choice(zq.numel(), 4096, replace=False))
    res.update(vq4_idx=st['min_encoding_indices'].numpy(), vq4_zq_sample=zq.reshape(-1)[torch.from_numpy(sample)].numpy(),
               vq4_sample_at=sample)

    from basicsr.archs.codeformer_arch import TransformerSALayer
    sd, t, pos = transformer_layer_inputs()
    layer = TransformerSALayer(512, 8, 1024).eval()
    layer.load_state_dict({k[2:]: v for k, v in sd.items()}, strict=True)
    res['sa_layer_out_s16'] = layer(t, query_pos=pos)[::16].numpy()

    from basicsr.utils import img2tensor, tensor2img
    from torchvision.transforms.functional import normalize
    face, out = plumbing_small_inputs()
    x = img2tensor(face / 255., bgr2rgb=True, float32=True)
    normalize(x, (0.5, 0.5, 0.5), (0.5, 0.5, 0.5), inplace=True)
    res.update(plumbing_small_x=x.numpy(),
               plumbing_small_restored=tensor2img(torch.from_numpy(out.copy()), rgb2bgr=True, min_max=(-1, 1)).astype('uint8'))

    from basicsr.utils.realesrgan_utils import RealESRGANer
    model = ToyUpsampler().eval()
    for tile, pre_pad, shape in ESR_CASES:
        er = RealESRGANer.__new__(RealESRGANer)              # the reference constructor insists on loading a checkpoint file
        er.scale, er.tile_size, er.tile_pad, er.pre_pad, er.mod_scale, er.half = 2, tile, 6, pre_pad, None, False
        er.device, er.model = torch.device('cpu'), model
        o, mode = er.enhance(esr_image(shape), outscale=2)
        res[esr_key(tile, pre_pad, shape)], res[esr_key(tile, pre_pad, shape) + '_mode'] = o, np.array(mode)
    np.savez_compressed(os.path.join(OUT, 'reference_checks.npz'), **res)


def main():
    if len(sys.argv) > 1 and sys.argv[1] == 'reference_checks':
        gen_reference_checks()
        return
    if len(sys.argv) > 1 and sys.argv[1] == 'parsenet':
        gen_parsenet()
        return
    if len(sys.argv) > 1 and sys.argv[1] == 'rrdbnet':
        gen_rrdbnet()
        return
    if len(sys.argv) > 1 and sys.argv[1] == 'plumbing':
        gen_plumbing()
        return
    torch.set_num_threads(os.cpu_count())
    CodeFormer, VQAE, VQ, _ = ref_shim.load()
    os.makedirs(OUT, exist_ok=True)
    faces = load_faces()
    np.savez_compressed(os.path.join(OUT, 'faces.npz'), faces=faces, names=np.array(FACES))
    x = to_input(faces)

    with torch.no_grad():
        net = CodeFormer(dim_embd=512, codebook_size=1024, n_head=8, n_layers=9,
                         connect_list=['32', '64', '128', '256']).eval()
        net.load_state_dict(S.random_state_dict(S.codeformer_spec(), 1), strict=True)
        out, logits, lq = net(x[0:1], w=0.5, adain=True)
        np.savez_compressed(os.path.join(OUT, 'codeformer_main.npz'), out=out.numpy(), logits=logits.numpy(),
                            lq_feat=lq.numpy(), top_idx=logits.argmax(2).numpy().astype(np.int64))
        var = {}
        o, l, q = net(x[1:2], w=0, adain=True)
        var.update(w0_out=o[..., ::4, ::4].numpy(), w0_idx=l.argmax(2).numpy(), w0_lq=q.numpy())
        o, l, q = net(x[1:2], w=1.0, adain=False)
        var.update(w1_out=o[..., ::4, ::4].numpy(), w1_idx=l.argmax(2).numpy())
        l, q = net(x[1:2], w=0, code_only=True)
        var.update(code_only_logits_row0=l[0, :4].numpy())
        net3 = CodeFormer(dim_embd=512, codebook_size=1024, n_head=8, n_layers=9,
                          connect_list=['32', '64', '128']).eval()                  # inference_colorization.py:45
        net3.load_state_dict(S.random_state_dict(S.codeformer_spec(connect_list=('32', '64', '128')), 3), strict=True)
        o, l, q = net3(x[1:2], w=0.7, adain=True)
        var.update(c3_out=o[..., ::4, ::4].numpy(), c3_idx=l.argmax(2).numpy())
        net5 = CodeFormer(dim_embd=512, codebook_size=512, n_head=8, n_layers=9,
                          connect_list=['32', '64', '128']).eval()                  # inference_inpainting.py:45
        net5.load_state_dict(S.random_state_dict(S.codeformer_spec(codebook_size=512, connect_list=('32', '64', '128')), 4),
                             strict=True)
        o, l, q = net5(x[1:2], w=1, adain=False)
        var.update(k512_out=o[..., ::4, ::4].numpy(), k512_idx=l.argmax(2).numpy())
        np.savez_compressed(os.path.join(OUT, 'codeformer_variants.npz'), **var)

        vq = VQAE(512, 64, [1, 2, 2, 4, 4, 8], 'nearest', 2, [16], 1024).eval()     # scripts/inference_vqgan.py:31
        vq.load_state_dict(S.random_state_dict(S.vqae_spec(), 2), strict=True)
        o, loss, st = vq(x[0:1])
        np.savez_compressed(os.path.join(OUT, 'vqae.npz'), out=o[..., ::4, ::4].numpy(), loss=loss.numpy(),
                            idx=st['min_encoding_indices'].numpy(), perplexity=st['perplexity'].numpy(),
                            mean_distance=st['mean_distance'].numpy())

        mic = {}
        for case in ('B', 'C'):
            E, z = vq_micro_inputs(case)
            m = VQ(1024, 256, 0.25)
            m.embedding.weight.data.copy_(E)
            zq, loss, st = m(z)
            mic.update({f'{case}_idx': st['min_encoding_indices'].numpy(), f'{case}_loss': loss.numpy(),
                        f'{case}_perplexity': st['perplexity'].numpy(), f'{case}_mean_distance': st['mean_distance'].numpy(),
                        f'{case}_zq_b0': zq[0].numpy()})
        np.savez_compressed(os.path.join(OUT, 'vq_micro.npz'), **mic)
    gen_plumbing()
    gen_rrdbnet()
    gen_parsenet()
    gen_reference_checks()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)) // 1024, 'KiB')


if __name__ == '__main__':
    main()
