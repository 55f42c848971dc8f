"""Drop-in boundary on the CPU: state-dict contract, registry, C-ABI symbols, host-side planning."""
import ctypes
import os
import re

import pytest
import torch

import codeformer_b200 as cb
from codeformer_b200 import _lib, spec as S
from tests.util import ROOT, golden


def test_state_dict_contract_codeformer():
    net = cb.CodeFormer()
    sp = S.codeformer_spec()
    sd = net.state_dict()
    assert list(sd.keys()) == list(sp.keys()) and len(sd) == 515
    assert all(tuple(sd[k].shape) == tuple(sp[k]) for k in sp)
    assert sum(v.numel() for v in sd.values()) * 4 == 376450828          # 376.45 MB, SURVEY.md §8b
    net.load_state_dict(S.random_state_dict(sp, 1), strict=True)
    # fix_modules=['quantize','generator'] only freezes parameters (codeformer_arch.py:172-175)
    assert not any(p.requires_grad for p in net.generator.parameters())
    assert all(p.requires_grad for p in net.encoder.parameters())
    # training-side attribute surface of codeformer_model.py:146-158,195-199
    assert net.generator.blocks[-1].weight.shape == (3, 64, 3, 3)
    assert net.fuse_convs_dict['256'].shift['2'].weight.shape == (128, 128, 3, 3)


@pytest.mark.parametrize('kw', [dict(connect_list=['32', '64', '128']),
                                dict(codebook_size=512, connect_list=['32', '64', '128'])])
def test_state_dict_contract_variants(kw):
    net = cb.CodeFormer(dim_embd=512, n_head=8, n_layers=9, **kw)
    sp = S.codeformer_spec(codebook_size=kw.get('codebook_size', 1024), connect_list=tuple(kw['connect_list']))
    assert list(net.state_dict().keys()) == list(sp.keys())


def test_state_dict_contract_vqae():
    v = cb.VQAutoEncoder(512, 64, [1, 2, 2, 4, 4, 8], 'nearest', 2, [16], 1024)
    assert list(v.state_dict().keys()) == list(S.vqae_spec().keys())
    with pytest.raises(NotImplementedError):
        cb.VQAutoEncoder(512, 64, [1, 2, 2, 4, 4, 8], 'gumbel')


def test_keys_equal_live_reference():
    """Keys, order and shapes of the reference's CodeFormer() state dict (tests/golden/reference_checks.npz)."""
    g = golden('reference_checks.npz')
    ours = cb.CodeFormer().state_dict()
    assert list(g['codeformer_keys']) == list(ours.keys())
    assert list(g['codeformer_shapes']) == [','.join(map(str, v.shape)) for v in ours.values()]


def test_registry_interface():
    assert cb.ARCH_REGISTRY.get('CodeFormer') is cb.CodeFormer
    assert cb.ARCH_REGISTRY.get('VQAutoEncoder') is cb.VQAutoEncoder
    assert 'CodeFormer' in cb.ARCH_REGISTRY
    with pytest.raises(KeyError):
        cb.ARCH_REGISTRY.get('nope')
    with pytest.raises(AssertionError):                      # duplicate names assert, registry.py:39
        cb.ARCH_REGISTRY.register(cb.CodeFormer)
    r = cb.registry.ArchTable('x')
    r.add(object, 'CodeFormer')

    @r.register()
    class Other:        # decorator form, as the reference's arch files use it (codeformer_arch.py:160)
        pass
    assert r.get('Other') is Other
    cb.install(r)                                            # existing entries are replaced, not added beside
    assert r.get('CodeFormer') is cb.CodeFormer and r.get('VQAutoEncoder') is cb.VQAutoEncoder

    class RefLike:      # an object shaped like the reference's registry (a private name -> class dict)
        def __init__(self):
            self._obj_map = {'CodeFormer': int}
    rl = cb.install(RefLike())
    assert rl._obj_map['CodeFormer'] is cb.CodeFormer


def test_c_abi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, 'include', 'cfb200.h')).read()
    hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
    declared = set(re.findall(r'\b(cfb_[a-z0-9_]+)\s*\(', hdr))
    assert len(declared) >= 25
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f'{name} declared in include/cfb200.h but not exported'
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert _lib.load().cfb_version() == 100


def test_host_planning_without_gpu():
    lib = _lib.load()
    net = cb.CodeFormer()
    h = ctypes.c_void_p(lib.cfb_net_create(ctypes.byref(net._cfb_config())))
    assert h
    # the fp32 engine: the plan cfb_net_create picks when no tcgen05 device is present, here on every machine (on a B200
    # the default engine plans the tensor-core path, whose arena is laid out differently)
    assert lib.cfb_net_set_engine(h, 1) == 0
    w1, w8 = lib.cfb_workspace_bytes(h, 1), lib.cfb_workspace_bytes(h, 8)
    assert 0 < w1 < w8 < 8 * w1 + (1 << 20)
    assert lib.cfb_workspace_bytes(h, 0) >= 0
    lib.cfb_net_destroy(h)
    bad = net._cfb_config()
    bad.nf = 48
    assert not lib.cfb_net_create(ctypes.byref(bad))
    assert b'nf=64' in lib.cfb_last_error()


def test_cpu_input_raises_no_fallback():
    net = cb.CodeFormer()
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        net(torch.zeros(1, 3, 512, 512), w=0.5)
    with pytest.raises(RuntimeError):
        net.quantize(torch.zeros(1, 256, 16, 16))
    with pytest.raises(RuntimeError, match='parameter holder'):
        net.encoder.blocks[0](torch.zeros(1, 3, 8, 8))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, 'codeformer_b200')
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dp, f)).read()
                assert 'oracle' not in src.replace('no CPU fallback', ''), f'{f} mentions the oracle'


class _BasicsrRegistry:
    """The behaviour of basicsr's Registry (basicsr/utils/registry.py) that install() relies on: the classes live in a private
    name -> class dict ``_obj_map``, ``register`` asserts when the name is already taken, ``get`` raises KeyError when absent."""

    def __init__(self):
        self._obj_map = {}

    def register(self, obj):
        assert obj.__name__ not in self._obj_map, f'{obj.__name__} is already registered'
        self._obj_map[obj.__name__] = obj

    def get(self, name):
        if self._obj_map.get(name) is None:
            raise KeyError(name)
        return self._obj_map[name]


def test_install_replaces_entries_of_the_reference_registry():
    """`install()` must swap the two entries of the reference's ARCH_REGISTRY in place (registry.py:39 would assert
    on a second registration), after which the reference's lookup returns the B200 classes."""
    REG = _BasicsrRegistry()
    for name in ('CodeFormer', 'VQAutoEncoder'):
        REG.register(type(name, (torch.nn.Module,), {}))         # the reference's own classes, registered at import
    with pytest.raises(AssertionError):
        REG.register(cb.CodeFormer)
    assert cb.install(REG) is REG
    assert REG.get('CodeFormer') is cb.CodeFormer and REG.get('VQAutoEncoder') is cb.VQAutoEncoder
    net = REG.get('CodeFormer')(dim_embd=512, codebook_size=1024, n_head=8, n_layers=9,
                                connect_list=['32', '64', '128', '256'])
    assert len(net.state_dict()) == 515
