"""Generate tests/golden/loader_chunk_v1.pt: what the UNMODIFIED reference's `FilesystemDataset._load_chunk_inner`
returns for the seeded parquet chunk of tests/test_gpu_zj_loader.py (on the host: the method computes its rays with
torch matmuls on whichever device the dataset names).

Needs a checkout of the reference (MEGA_NERF_REFERENCE=<path> python tests/golden/make_loader_chunk.py).

The chunk's 70 000 rows draw from 5 images x 160 pixels, so its rays are stored as the reference's ray of every
(get_rays_batch call, image, pixel) triple - every row is one entry of that table - and the colours and image indices,
exact functions of the chunk, as the SHA-256 of their bytes.
"""
from __future__ import annotations

import os
import sys
import tempfile

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as MG  # noqa: E402,F401  (sets sys.path for cases / oracle / reference)
import test_gpu_zj_loader as T  # noqa: E402
from ref_shims import install_shims  # noqa: E402


def main():
    install_shims()
    from mega_nerf.datasets.filesystem_dataset import FilesystemDataset, RAY_CHUNK_SIZE
    assert RAY_CHUNK_SIZE == T.RAY_CHUNK_SIZE
    dirs, c2w, img, pix, rgb = T.chunk_case()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, 'chunk0.parquet')
        T.write_chunk(path, img, pix, rgb)
        _, rgbs, rays, img_indices = FilesystemDataset._load_chunk_inner(T.chunk_dataset(path, dirs, c2w, torch.device('cpu')))
    rows = torch.arange(img.shape[0])
    table = torch.full((int(rows[-1]) // RAY_CHUNK_SIZE + 1, c2w.shape[0], dirs.shape[0], 8), float('nan'))
    table[rows // RAY_CHUNK_SIZE, img.long(), pix.long()] = rays
    assert torch.equal(table[rows // RAY_CHUNK_SIZE, img.long(), pix.long()], rays)
    G = {'rays_by_pair': table, 'rgbs_sha256': T.digest(rgbs), 'img_indices_sha256': T.digest(img_indices)}
    torch.save(G, T.CHUNK_GOLDEN_PATH)
    print(f'wrote {T.CHUNK_GOLDEN_PATH} ({os.path.getsize(T.CHUNK_GOLDEN_PATH)} bytes)')


if __name__ == '__main__':
    main()
