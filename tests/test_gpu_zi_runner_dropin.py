"""GPU: the reference's OWN Runner (mega_nerf/runner.py of the reference checkout that MEGA_NERF_REFERENCE names, unmodified;
skipped without one) on top of mega_nerf_b200.install():
`Runner.render_image` (runner.py:540-578, the eval path: get_ray_directions -> get_rays -> chunked render_rays with
get_depth / get_bg_fg_rgb) and one `Runner._training_step` (runner.py:347-378) + backward, compared with the same Runner
on the reference's unmodified hot path (torch-CUDA fp32, TF32 off) on the same synthetic dataset directory, same seed.
Each side runs in its own process (install() rebinds module attributes).  The dataset is 3 tiny posed images written to a
temp dir in the reference's on-disk layout (coordinates.pt, {train,val}/{metadata,rgbs})."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get('MEGA_NERF_REFERENCE', '')

CHILD = r'''
import os, sys, math
root, ref, ds, out, mode, variant = sys.argv[1:7]
sys.path.insert(0, root); sys.path.insert(0, os.path.join(root, 'tests')); sys.path.insert(0, ref)
import torch
torch.backends.cuda.matmul.allow_tf32 = False
torch.backends.cudnn.allow_tf32 = False
from ref_shims import install_shims
install_shims()
if mode == 'b200':
    import mega_nerf_b200
    mega_nerf_b200.install()
    mega_nerf_b200.set_precision('fp32')
from mega_nerf.opts import get_opts_base
from mega_nerf.runner import Runner
import mega_nerf.runner as RU
if mode == 'b200':
    assert RU.render_rays.__module__.startswith('mega_nerf_b200'), RU.render_rays.__module__
    assert RU.get_nerf.__module__.startswith('mega_nerf_b200')
else:
    assert RU.render_rays.__module__ == 'mega_nerf.rendering'
argv = ['--dataset_path', ds, '--exp_name', os.path.join(out, 'exp'), '--no_amp', '--coarse_samples', '16', '--fine_samples', '32',
        '--near', '0.05', '--far', '1.5', '--ray_altitude_range', '-0.6', '0.3', '--val_scale_factor', '1',
        '--image_pixel_batch_size', '96', '--model_chunk_size', '4096', '--appearance_dim', '8', '--layer_dim', '64', '--bg_layer_dim', '64']
if variant == 'nobg':
    argv += ['--no_bg_nerf']
parser = get_opts_base()
parser.add_argument('--exp_name', type=str, required=True)
parser.add_argument('--dataset_path', type=str, required=True)
hp = parser.parse_args(argv)
runner = Runner(hp, set_experiment_path=False)
assert runner.device.type == 'cuda' or os.environ.get('MN_RUNNER_TEST_ALLOW_CPU') == '1'
res = {}
with torch.no_grad():
    runner.nerf.eval()
    if runner.bg_nerf is not None:
        runner.bg_nerf.eval()
    results, rays = runner.render_image(runner.val_items[0])
res['eval'] = {k: v.float().cpu() for k, v in results.items()}
res['eval_rays'] = rays.cpu()
# one training step on a fixed batch of pixels of the first train image (eval-like determinism: no jitter)
runner.nerf.train()
if runner.bg_nerf is not None:
    runner.bg_nerf.train()
hp.perturb = 0.0
md = runner.train_items[0]
from mega_nerf.ray_utils import get_rays, get_ray_directions
d = get_ray_directions(md.W, md.H, md.intrinsics[0], md.intrinsics[1], md.intrinsics[2], md.intrinsics[3], hp.center_pixels, runner.device)
r = get_rays(d, md.c2w.to(runner.device), runner.near, runner.far, runner.ray_altitude_range).view(-1, 8)[:64].contiguous()
rgbs = (md.load_image().float() / 255.0).view(-1, 3)[:64].to(runner.device)
idx = torch.full((64,), md.image_index, dtype=torch.int32, device=runner.device)
torch.manual_seed(7)
metrics, present = runner._training_step(rgbs, r, idx)
metrics['loss'].backward()
res['train'] = {'loss': float(metrics['loss']), 'psnr': float(metrics['psnr']), 'present': bool(present),
                'grads': {k: p.grad.detach().float().cpu() for k, p in runner.nerf.named_parameters() if p.grad is not None}}
torch.save(res, os.path.join(out, mode + '.pt'))
print('RUNNER_OK', mode, sorted(res['eval']))
'''


def make_dataset(ds):
    """3 posed 12x8 images in the reference's dataset layout (runner.py:595-660, image_metadata.py:11-29)."""
    import numpy as np
    from PIL import Image
    g = torch.Generator().manual_seed(3)
    for sub in ('train', 'val'):
        os.makedirs(os.path.join(ds, sub, 'metadata'))
        os.makedirs(os.path.join(ds, sub, 'rgbs'))
    torch.save({'origin_drb': torch.zeros(3), 'pose_scale_factor': 1.0}, os.path.join(ds, 'coordinates.pt'))
    W, H = 12, 8
    for i in range(3):
        sub = 'val' if i == 2 else 'train'
        # camera above the ground (x is "down" in the reference's drb frame), looking mostly down (+x)
        rot = torch.tensor([[0.0, 0.0, -1.0], [1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])
        c2w = torch.cat([rot, torch.tensor([[-0.3], [0.1 * i - 0.1], [0.05 * i]])], 1)
        torch.save({'c2w': c2w, 'intrinsics': torch.tensor([10.0, 10.0, W / 2, H / 2]), 'W': W, 'H': H, 'distortion': torch.zeros(4)},
                   os.path.join(ds, sub, 'metadata', f'{i:06d}.pt'))
        img = (torch.rand(H, W, 3, generator=g) * 255).byte().numpy()
        Image.fromarray(np.ascontiguousarray(img)).save(os.path.join(ds, sub, 'rgbs', f'{i:06d}.png'))


def run_side(mode, variant, ds, out):
    r = subprocess.run([sys.executable, '-c', CHILD, ROOT, REF, ds, out, mode, variant], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and 'RUNNER_OK' in r.stdout, f'{mode}/{variant}: rc={r.returncode}\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}'
    return torch.load(os.path.join(out, mode + '.pt'), map_location='cpu', weights_only=False)


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, 'mega_nerf')), reason='needs a reference checkout named by MEGA_NERF_REFERENCE')
@pytest.mark.parametrize('variant', ['bg', 'nobg'])
def test_reference_runner_on_top_of_install(tmp_path, variant):
    ds, out = str(tmp_path / 'dataset'), str(tmp_path / 'out')
    os.makedirs(out)
    make_dataset(ds)
    ref = run_side('reference', variant, ds, out)
    got = run_side('b200', variant, ds, out)
    assert float((got['eval_rays'] - ref['eval_rays']).abs().max()) <= 1e-5          # get_ray_directions + get_rays through install()
    assert set(got['eval']) == set(ref['eval']), (sorted(got['eval']), sorted(ref['eval']))
    for k, v in ref['eval'].items():
        scale = float(v.abs().max()) + 1e-12
        err = float((got['eval'][k] - v).abs().max()) / scale
        assert err <= 2e-4, (variant, k, err)             # fp32 kernels vs the reference under torch-CUDA fp32 (different sum orders)
    assert got['train']['present'] == ref['train']['present']
    assert abs(got['train']['loss'] - ref['train']['loss']) <= 2e-3 * abs(ref['train']['loss'])
    assert set(got['train']['grads']) == set(ref['train']['grads'])
    num = sum(float(((got['train']['grads'][k] - g) ** 2).sum()) for k, g in ref['train']['grads'].items())
    den = sum(float((g ** 2).sum()) for g in ref['train']['grads'].values())
    assert (num / max(den, 1e-30)) ** 0.5 <= 2e-2, (variant, (num / den) ** 0.5)
