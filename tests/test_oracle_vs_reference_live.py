"""CPU-only: randomised configurations - widths, depths, skip layers, SH degree, appearance / affine, cascade, background,
routing margin, 2-D / 3-D clustering, train / eval mode - rendered by the oracle with the same seeds as the UNMODIFIED
reference was, whose results and parameter gradients (tests/golden/reference_live_v1.pt, written by
tests/golden/make_reference_live.py) they must match bit for bit; and the reference's call surface (signatures, state-dict
layouts) that the product's drop-in symbols must reproduce."""
import dataclasses
import hashlib
import inspect
import os
import random

import pytest
import torch

import cases as C
from oracle import mn_oracle as O

GOLDEN_PATH = os.path.join(C.ROOT, 'tests', 'golden', 'reference_live_v1.pt')
SEEDS = list(range(16))
# (symbol of mega_nerf_b200, the reference symbol it replaces as 'module:qualname')
SURFACE = [('render_rays', 'mega_nerf.rendering:render_rays'), ('get_rays', 'mega_nerf.ray_utils:get_rays'),
           ('get_rays_batch', 'mega_nerf.ray_utils:get_rays_batch'),
           ('get_ray_directions', 'mega_nerf.ray_utils:get_ray_directions'),
           ('eval_sh', 'mega_nerf.spherical_harmonics:eval_sh'),
           ('NeRF.__init__', 'mega_nerf.models.nerf:NeRF.__init__'), ('NeRF.forward', 'mega_nerf.models.nerf:NeRF.forward'),
           ('MegaNeRF.__init__', 'mega_nerf.models.mega_nerf:MegaNeRF.__init__'),
           ('MegaNeRF.forward', 'mega_nerf.models.mega_nerf:MegaNeRF.forward'),
           ('Cascade.__init__', 'mega_nerf.models.cascade:Cascade.__init__'),
           ('Cascade.forward', 'mega_nerf.models.cascade:Cascade.forward'),
           ('Embedding.__init__', 'mega_nerf.models.nerf:Embedding.__init__'),
           ('ShiftedSoftplus.__init__', 'mega_nerf.models.nerf:ShiftedSoftplus.__init__')]
STATE_DICT_KINDS = ('nerf', 'cascade', 'mega')
STATE_DICT_SPEC = O.NerfSpec(layer_dim=32, appearance_count=5)


@pytest.fixture(scope='module')
def live():
    return torch.load(GOLDEN_PATH, map_location='cpu', weights_only=False)


def signature_of(fn):
    """[(name, repr(default), kind)] of every parameter."""
    return [(p.name, repr(p.default), str(p.kind)) for p in inspect.signature(fn).parameters.values()]


def state_dict_net(kind: str) -> O.Net:
    cents = O.grid_centroids(2, 2) if kind == 'mega' else None
    return O.make_net(kind, STATE_DICT_SPEC, seed=1, n_sub=4 if kind == 'mega' else 1, centroids=cents, cluster_2d=True)


def case_cotangent(seed: int, rays, opts):
    key = f'rgb_{"fine" if opts.fine_samples > 0 else "coarse"}'
    return key, torch.randn(rays.shape[0], 3, generator=torch.Generator().manual_seed(seed))


def random_case(seed: int):
    rnd = random.Random(seed)
    sh = rnd.random() < 0.25
    app = rnd.choice([0, 16, 48])
    affine = app > 0 and not sh and rnd.random() < 0.25
    layers = rnd.choice([2, 4, 8])
    spec = O.NerfSpec(pos_xyz_dim=rnd.choice([6, 12]), pos_dir_dim=0 if sh else rnd.choice([2, 4]), layers=layers,
                      skip_layers=(rnd.randrange(1, layers),) if rnd.random() < 0.8 else (), layer_dim=rnd.choice([32, 64, 96]),
                      appearance_dim=app, affine_appearance=affine, appearance_count=9, rgb_dim=27 if sh else 3,
                      shifted_softplus=rnd.random() < 0.8)
    kind = rnd.choice(['nerf', 'cascade', 'mega'])
    cascade = kind == 'cascade'
    grid = rnd.choice([(2, 2), (1, 3), (2, 4)])
    cents = O.grid_centroids(*grid) if kind == 'mega' else None
    c2d = rnd.random() < 0.6
    if cents is not None and not c2d:
        cents = cents.clone()
        cents[:, 0] = torch.rand(cents.shape[0], generator=torch.Generator().manual_seed(seed)) * 0.4 - 0.2
    margin = rnd.choice([1.0, 1.15, 1.4]) if kind == 'mega' else 1.0
    net = O.make_net(kind, spec, seed=seed, n_sub=0 if cents is None else cents.shape[0], centroids=cents,
                     boundary_margin=margin, cluster_2d=c2d)
    has_bg = rnd.random() < 0.3
    bg = None
    center = radius = None
    n_rays = rnd.choice([7, 33, 64])
    rays = O.synthetic_rays(n_rays, seed=seed, far=1e5 if has_bg else 0.6)
    if has_bg:
        bg = O.make_net('cascade' if cascade else 'nerf', dataclasses.replace(spec, xyz_dim=4), seed=seed + 1)
        center, radius = torch.tensor([0.05, -0.02, 0.03]), torch.tensor([0.8, 0.9, 1.0])
        rays[::2, 7] = 0.4
    idx = O.synthetic_indices(n_rays, 9, seed=seed) if app > 0 else None
    fine = rnd.choice([0, 8, 24]) if cascade else rnd.choice([8, 24])
    opts = O.RenderOpts(coarse_samples=rnd.choice([8, 16, 31]), fine_samples=fine, use_cascade=cascade, perturb=1.0,
                        pos_dir_dim=spec.pos_dir_dim, sh_deg=2 if sh else None, model_chunk_size=rnd.choice([64, 1000, 32768]))
    return net, bg, rays, idx, opts, center, radius, rnd.random() < 0.5


@pytest.mark.parametrize('seed', SEEDS)
def test_random_configuration_bit_exact(live, seed):
    net, bg, rays, idx, opts, c, r, training = random_case(seed)
    want = live['configurations'][seed]
    nt = dataclasses.replace(net, training=training)
    bt = dataclasses.replace(bg, training=training) if bg is not None else None
    key, cot = case_cotangent(seed, rays, opts)
    torch.manual_seed(seed)
    got, gn, gb = O.render_grads(nt, bt, rays, idx, opts, c, r, {key: cot})
    ref = want['results']
    assert set(got) == set(ref)
    for k in ref:
        assert torch.equal(ref[k], got[k]), (seed, k, float((ref[k] - got[k]).abs().max()))
    for tag, g_ in (('net', gn), ('bg', gb)):
        if want['grads'][tag] is None:
            assert g_ is None, (seed, tag)
            continue
        assert len(g_) == len(want['grads'][tag]), (seed, tag)
        for a, b in zip(want['grads'][tag], g_):
            assert set(a) == set(b), (seed, tag, set(a) ^ set(b))
            for k, e in a.items():
                flat = b[k].detach().reshape(-1)
                assert tuple(b[k].shape) == e['shape'], (seed, tag, k)
                sha = hashlib.sha256(b[k].detach().float().contiguous().numpy().tobytes()).hexdigest()
                assert sha == e['sha256'], (seed, tag, k, float((flat[e['idx']] - torch.tensor(e['val'])).abs().max()))


def test_call_surface_signatures_match_reference(live):
    """Drop-in boundary (SURVEY.md §8b): every replaced symbol takes the reference's parameters, in order, with the
    reference's defaults."""
    import mega_nerf_b200 as M
    surface = live['surface']
    for mine_path, ref_path in SURFACE:
        mine = M
        for a in mine_path.split('.'):
            mine = getattr(mine, a)
        pa, pb = signature_of(mine), surface['signatures'][ref_path]
        assert [x[0] for x in pa] == [x[0] for x in pb], (ref_path, pa, pb)
        assert [x[1:] for x in pa] == [x[1:] for x in pb], (ref_path, pa, pb)
    for name, params in surface['factories'].items():
        assert list(inspect.signature(getattr(M, name)).parameters) == params, name
    # state-dict layout of every model family
    spec = STATE_DICT_SPEC
    for kind in STATE_DICT_KINDS:
        cents = state_dict_net(kind).centroids
        from test_host_factories import M as _M  # noqa: F401
        if kind == 'nerf':
            mine = M.NeRF(spec.pos_xyz_dim, spec.pos_dir_dim, spec.layers, list(spec.skip_layers), spec.layer_dim, spec.appearance_dim,
                          spec.affine_appearance, spec.appearance_count, spec.rgb_dim, spec.xyz_dim, M.ShiftedSoftplus())
        elif kind == 'cascade':
            mk = lambda: M.NeRF(spec.pos_xyz_dim, spec.pos_dir_dim, spec.layers, list(spec.skip_layers), spec.layer_dim,  # noqa: E731
                                spec.appearance_dim, spec.affine_appearance, spec.appearance_count, spec.rgb_dim, spec.xyz_dim,
                                M.ShiftedSoftplus())
            mine = M.Cascade(mk(), mk())
        else:
            mk = lambda: M.NeRF(spec.pos_xyz_dim, spec.pos_dir_dim, spec.layers, list(spec.skip_layers), spec.layer_dim,  # noqa: E731
                                spec.appearance_dim, spec.affine_appearance, spec.appearance_count, spec.rgb_dim, spec.xyz_dim,
                                M.ShiftedSoftplus())
            mine = M.MegaNeRF([mk() for _ in range(4)], cents, 1.15, False, True)
        a, layout = mine.state_dict(), surface['state_dicts'][kind]
        assert list(a) == [k for k, _, _ in layout], (kind, set(a) ^ {k for k, _, _ in layout})
        assert all(tuple(a[k].shape) == s and str(a[k].dtype) == d for k, s, d in layout)
        # reference checkpoints load: a state dict in the reference's layout
        mine.load_state_dict({k: torch.zeros(s, dtype=getattr(torch, d.split('.')[-1])) for k, s, d in layout})
