"""Generate tests/golden/reference_live_v1.pt: what the UNMODIFIED reference computes on the randomised configurations of
tests/test_oracle_vs_reference_live.py, and the call surface (signatures, state-dict layouts) that test pins.

Needs a checkout of the reference (MEGA_NERF_REFERENCE=<path> python tests/golden/make_reference_live.py).

Per configuration the rendered results are stored whole; each parameter gradient is stored as the SHA-256 of its float32
bytes (the bit-exact check) plus a seeded sample of its elements (the numbers a failure reports), which keeps the file
small although the gradients of the larger networks run to megabytes.
"""
from __future__ import annotations

import hashlib
import inspect
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as MG  # noqa: E402  (sets sys.path for cases / oracle / reference)
import make_golden_backward as MB  # noqa: E402
import test_oracle_vs_reference_live as T  # noqa: E402

C, O = MG.C, MG.O
GRAD_SAMPLE = 8


def digest(t: torch.Tensor) -> str:
    return hashlib.sha256(t.detach().float().contiguous().numpy().tobytes()).hexdigest()


def grad_entry(g: torch.Tensor, seed: int) -> dict:
    flat = g.detach().reshape(-1)
    n = min(GRAD_SAMPLE, flat.numel())
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:n].sort().values
    return {'sha256': digest(g), 'shape': tuple(g.shape), 'idx': idx.tolist(), 'val': flat[idx].tolist()}


def random_configurations() -> dict:
    out = {}
    for seed in T.SEEDS:
        net, bg, rays, idx, opts, c, r, training = T.random_case(seed)
        rn = MG.ref_net(net)
        rb = MG.ref_net(bg) if bg is not None else None
        for mod in (rn, rb):
            if mod is not None:
                mod.train(training)
                for p in mod.parameters():
                    p.requires_grad_(True)
        key, cot = T.case_cotangent(seed, rays, opts)
        torch.manual_seed(seed)
        ref, _ = MG.R_render.render_rays(rn, rb, rays, idx, MG.hparams_of(opts), c, r, False, True, False)
        (ref[key] * cot).sum().backward()
        grads = {}
        for tag, mod, n_ in (('net', rn, net), ('bg', rb, bg)):
            grads[tag] = None if mod is None else [
                {k: grad_entry(g, seed * 1000 + j * 100 + i) for i, (k, g) in enumerate(sorted(sub.items()))}
                for j, sub in enumerate(MB.ref_grads(mod, n_))]
        out[seed] = {'results': {k: v.detach().clone() for k, v in ref.items()}, 'grads': grads}
    return out


def call_surface() -> dict:
    import importlib
    sig = {}
    for _, ref_path in T.SURFACE:
        mod, attr = ref_path.rsplit(':', 1)
        obj = importlib.import_module(mod)
        for a in attr.split('.'):
            obj = getattr(obj, a)
        sig[ref_path] = T.signature_of(obj)
    mu = importlib.import_module('mega_nerf.models.model_utils')
    factories = {name: list(inspect.signature(getattr(mu, name)).parameters) for name in ('get_nerf', 'get_bg_nerf')}
    layouts = {}
    for kind in T.STATE_DICT_KINDS:
        sd = MG.ref_net(T.state_dict_net(kind)).state_dict()
        layouts[kind] = [(k, tuple(v.shape), str(v.dtype)) for k, v in sd.items()]
    return {'signatures': sig, 'factories': factories, 'state_dicts': layouts}


def main():
    G = {'configurations': random_configurations(), 'surface': call_surface()}
    torch.save(G, T.GOLDEN_PATH)
    print(f'wrote {T.GOLDEN_PATH} ({os.path.getsize(T.GOLDEN_PATH)} bytes)')


if __name__ == '__main__':
    main()
