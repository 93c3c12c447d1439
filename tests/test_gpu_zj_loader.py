"""GPU: loader-side ray generation (SURVEY.md §8f-6).  `get_rays_pairs` against the oracle's get_rays_batch product gathered at
the same (image, pixel) pairs, and `mega_nerf_b200.loader._load_chunk_inner` against what the reference's own
`FilesystemDataset._load_chunk_inner` returned for the same stand-in dataset object and the same parquet chunk in the
reference's column layout (filesystem_dataset.py:95-131,222-260), stored in tests/golden/loader_chunk_v1.pt by
tests/golden/make_loader_chunk.py."""
import hashlib
import os
import types
from itertools import cycle
from pathlib import Path

import pytest
import torch

import cases  # noqa: F401
from oracle import mn_oracle as O
from test_gpu_parity import DEV, M

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK_GOLDEN_PATH = os.path.join(ROOT, 'tests', 'golden', 'loader_chunk_v1.pt')
RAY_CHUNK_SIZE = 64 * 1024                                               # the reference loader's rays per get_rays_batch call
NEAR, FAR, ALT = 0.1, 3.0, [-0.35, 0.05]


def scene(n_img=7, W=13, H=9):
    g = torch.Generator().manual_seed(11)
    dirs = O.ray_directions(W, H, 9.5, 9.1, 6.2, 3.4, True).view(-1, 3)
    q, _ = torch.linalg.qr(torch.randn(n_img, 3, 3, generator=g))
    c2w = torch.cat([q, torch.cat([-0.3 - 0.2 * torch.rand(n_img, 1, generator=g), torch.rand(n_img, 2, generator=g) - 0.5], 1).unsqueeze(-1)], -1)
    return dirs, c2w, g


@pytest.mark.parametrize('alt', [None, [-0.35, 0.05]])
def test_rays_pairs_match_batch_product(alt):
    dirs, c2w, g = scene()
    Mp = 5000
    ii = torch.randint(0, c2w.shape[0], (Mp,), generator=g, dtype=torch.int32)
    pi = torch.randint(0, dirs.shape[0], (Mp,), generator=g, dtype=torch.int32)
    want = O.rays_from_pose_batch(dirs.view(1, -1, 3).expand(c2w.shape[0], -1, -1).contiguous(), c2w, 0.1, 3.0, alt)[ii.long(), pi.long()]
    got = M().raygen.get_rays_pairs(dirs.to(DEV), c2w.to(DEV), ii.to(DEV), pi.to(DEV), 0.1, 3.0, alt)
    assert got.shape == (Mp, 8)
    assert float((got.cpu() - want).abs().max()) <= 5e-7
    # and the product entry itself at those pairs (the patched get_rays_batch with the loader's [P,3] call shape)
    prod = M().get_rays_batch(dirs.to(DEV), c2w.to(DEV), 0.1, 3.0, alt)[ii.long().to(DEV), pi.long().to(DEV)]
    assert torch.equal(prod, got)


def test_rays_pairs_bad_index_raises():
    dirs, c2w, g = scene()
    m = M()
    ii = torch.tensor([0, c2w.shape[0]], dtype=torch.int32)          # second image index is out of range
    pi = torch.tensor([0, 1], dtype=torch.int32)
    out = m.raygen.get_rays_pairs(dirs.to(DEV), c2w.to(DEV), ii.to(DEV), pi.to(DEV), 0.1, 3.0, None)
    assert torch.isnan(out[1]).all() and torch.isfinite(out[0]).all()
    from mega_nerf_b200 import _cabi as K
    with pytest.raises(RuntimeError, match='index out of range'):
        K.check(K.lib().mn_check_status(K.ctx(DEV), K.stream_of(DEV)), K.ctx(DEV))


def chunk_case():
    """-> (directions, c2ws, img_indices, pixel_indices, rgbs as uint8) of one seeded parquet chunk"""
    dirs, c2w, g = scene(n_img=5, W=16, H=10)
    rows = 70000                                                          # > RAY_CHUNK_SIZE: the reference loops twice
    img = torch.randint(0, c2w.shape[0], (rows,), generator=g, dtype=torch.int32)
    pix = torch.randint(0, dirs.shape[0], (rows,), generator=g, dtype=torch.int32)
    rgb = torch.randint(0, 256, (rows, 3), generator=g, dtype=torch.uint8)
    return dirs, c2w, img, pix, rgb


def write_chunk(path, img, pix, rgb):
    import pyarrow as pa
    import pyarrow.parquet as pq
    cols = {'img_indices': pa.array(img.numpy()), 'pixel_indices': pa.array(pix.numpy())}
    for c in range(3):
        cols[f'rgbs_{c}'] = pa.array(rgb[:, c].numpy())
    pq.write_table(pa.table(cols), path)


def chunk_dataset(path, dirs, c2w, device):
    """the attributes of a FilesystemDataset that _load_chunk_inner reads"""
    return types.SimpleNamespace(_chunk_index=cycle(range(1)), _parquet_paths=[Path(path)], _directions=dirs.to(device), _c2ws=c2w,
                                 _device=device, _near=NEAR, _far=FAR, _ray_altitude_range=ALT)


def digest(t: torch.Tensor) -> str:
    return hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()


def test_chunk_loader_matches_reference_method(tmp_path):
    dirs, c2w, img, pix, rgb = chunk_case()
    path = tmp_path / 'chunk0.parquet'
    write_chunk(path, img, pix, rgb)
    want = torch.load(CHUNK_GOLDEN_PATH, map_location='cpu', weights_only=False)
    from mega_nerf_b200 import loader
    got = loader._load_chunk_inner(chunk_dataset(path, dirs, c2w, DEV))
    assert got[0] == str(path)
    assert digest(got[1]) == want['rgbs_sha256'] and digest(got[3]) == want['img_indices_sha256']
    assert got[2].shape == (img.shape[0], 8) and got[2].device.type == 'cpu'
    # the reference's ray of every row: its (get_rays_batch call, image, pixel) entry of the stored table
    rows = torch.arange(img.shape[0])
    ref_rays = want['rays_by_pair'][rows // RAY_CHUNK_SIZE, img.long(), pix.long()]
    assert float((got[2] - ref_rays).abs().max()) <= 2e-6                 # torch matmul vs the FMA chain of mn_rays
