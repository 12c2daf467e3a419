"""world_size-2 (and 3) gloo tests of the multi-GPU host logic on CPU: partitioning, ragged
all-gathers, re-assembly of features / chain states / frame tiles (boostmvsnerfs_b200/dist.py).
The compute hooks are replaced by deterministic CPU stand-ins; the assembled frame must be
identical on every rank and equal to the single-process result."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from boostmvsnerfs_b200 import dist as bdist
from boostmvsnerfs_b200.config import RenderConfig


def test_chain_blocks_and_slabs():
    import numpy as np
    for K in (1, 3, 4, 8, 9):
        for g in (1, 2, 3, 4, 8):
            blocks = [bdist.chain_block(K, g, r) for r in range(g)]
            assert blocks[0][0] == 0 and max(b for _, b in blocks) == K
            assert sorted(k for a, b in blocks for k in range(a, b)) == list(range(K))
            assert all(blocks[i][1] == blocks[i + 1][0] or blocks[i + 1] == (K, K) for i in range(g - 1))
    # every row a ray reads through the fp32 align_corners mapping lies inside its rank's slab
    for H, hv in ((544, 272), (1088, 544), (96, 48), (64, 8), (33, 17), (66, 33)):
        scale = np.float32(hv - 1) / np.float32(H - 1)
        for g in (1, 2, 3, 4, 8):
            for r in range(g):
                t0, t1 = bdist.row_tile(H, g, r)
                y0, y1 = bdist.slab_rows(t0, t1, H, hv)
                assert 0 <= y0 < y1 <= hv
                rows = np.arange(t0, t1, dtype=np.float32)
                i0 = (scale * rows).astype(np.int64)
                i1 = np.minimum(i0 + 1, hv - 1)
                if len(rows):
                    assert i0.min() >= y0 and i1.max() < y1, (H, hv, g, r)
                # the trilinear volume fetch (lean_gather.cuh) reaches its rows through grid_sample's normalisation
                # instead, each op rounded to fp32: iy = ((y / (H-1) * 2 - 1 + 1) * 0.5) * (hv-1), rows floor(iy) and +1
                gy = rows / np.float32(H - 1) * np.float32(2) - np.float32(1)
                iy = (gy + np.float32(1)) * np.float32(0.5) * np.float32(hv - 1)
                f0 = np.floor(iy).astype(np.int64)
                f1 = np.minimum(f0 + 1, hv - 1)
                if len(rows):
                    assert f0.min() >= y0 and f1.max() < y1, (H, hv, g, r)
            assert sum(b - a for a, b in (bdist.slab_rows(*bdist.row_tile(H, g, q), H, hv) for q in range(g))) <= hv + 4 * g


def test_partitions_cover_everything_exactly_once():
    for n in (1, 4, 6, 8, 544, 545):
        for g in (1, 2, 3, 4, 8):
            owned = [bdist.owned_round_robin(n, g, r) for r in range(g)]
            assert sorted(sum(owned, [])) == list(range(n))
            tiles = [bdist.row_tile(n, g, r) for r in range(g)]
            assert tiles[0][0] == 0 and tiles[-1][1] == n
            assert all(tiles[i][1] == tiles[i + 1][0] for i in range(g - 1))
            assert max(b - a for a, b in tiles) - min(b - a for a, b in tiles) <= 1
            parts = [[f"i{i}" for i in o] for o in owned]
            assert bdist.interleave_round_robin(parts, n) == [f"i{i}" for i in range(n)]


class _Ctx:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


class FakeNet:
    """Stands in for BoostEnerfNetwork: config + bookkeeping only."""
    generate_rays = False

    def __init__(self, rc, k_best):
        self.rc = rc
        self.view_selection_outputs = {"synth_0": k_best}

    def _check_mode(self, batch):
        pass

    def _stage(self, name):
        return _Ctx()

    def _camera_stage(self, exts, ixts, tar_ext, tar_ixt, image_hw=None):
        return None, None, None

    def parameters(self):
        return iter([torch.zeros(1)])


class FakeRenderer(bdist.ShardedFrameRenderer):
    """Deterministic stand-ins: features depend on the view id, a chain's volume / maps on its triple, the features and the
    ROW (so a wrong slab offset changes the result), the tile on the slab rows each ray reads and on the ray ids."""

    def compute_features(self, inps, views):
        if not len(views):
            return None
        shapes = self.feature_shapes(inps)
        return {n: torch.stack([inps[v].mean() + torch.arange(C * h * w, dtype=torch.float32).view(C, h, w) * (v + 1)
                                for v in views]) for n, (C, h, w) in shapes.items()}

    def compute_chains(self, feats, projs, near_far, triples, H, W, views_dev=None):
        rc = self.net.rc
        out = {}
        for i in range(rc.num):
            if not rc.render_if[i] or not triples:
                continue
            D, h, w = rc.volume_planes[i], int(H * rc.volume_scale[i]), int(W * rc.volume_scale[i])
            sig = [sum(float(feats['level_0'][v].sum()) for v in t) * 1e-6 + sum(t) for t in triples]
            row = torch.arange(h, dtype=torch.float32).view(1, 1, h, 1)
            vol = torch.stack([torch.full((8, D, h, w), s) + torch.arange(8.).view(8, 1, 1, 1) + 10 * row for s in sig])
            vol = vol.contiguous(memory_format=torch.channels_last_3d)
            out[i] = {'feat_vol': vol,
                      'depth_all': torch.stack([torch.full((h, w), s + 1) + row[0, 0] for s in sig]),
                      'std_all': torch.stack([torch.full((h, w), s + 2) + 2 * row[0, 0] for s in sig]),
                      'nf_all': torch.stack([torch.stack([torch.full((h, w), s + 3) + 3 * row[0, 0],
                                                          torch.full((h, w), s + 4) + 4 * row[0, 0]]) for s in sig])}
        return out

    def render_tile(self, level, feats, inps, vols, maps, y0, rays, cams, triples, H, W, ray_begin, n_rays, views_dev=None):
        rc = self.net.rc
        S = rc.num_samples[level]
        hv = int(H * rc.volume_scale[level])
        Hr = int(H * rc.render_scale[level])
        r = rays[ray_begin:ray_begin + n_rays]
        ids = r[:, 6] + 1000 * r[:, 7]
        # the two map / volume rows a ray of image row py reads (align_corners upsample), relative to the slab
        src = r[:, 7] * ((hv - 1) / max(Hr - 1, 1))
        i0 = src.floor().long().clamp(0, hv - 1)
        i1 = (i0 + 1).clamp(max=hv - 1)
        assert int(i0.min()) >= y0 and int(i1.max()) < y0 + vols.shape[3], "slab does not cover the rays' rows"
        val = torch.zeros(n_rays)
        for k in range(vols.shape[0]):
            per_row = vols[k].sum(dim=(0, 1, 3)) * 1e-4 + maps[k].sum(dim=(0, 2)) * 1e-2          # (rows,)
            val = val + (k + 1) * (per_row[i0 - y0] + 0.5 * per_row[i1 - y0])
        return torch.stack([ids + val * 1e-3 + c for c in range(4 + S)], dim=1)


def _scene(N=5, H=32, W=64):
    from boostmvsnerfs_b200.synth import make_scene
    return make_scene(H=H, W=W, n_views=N, seed=3)


def _worker(rank, world, port, K, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        # ragged gather with an empty contributor
        counts = [2, 0, 1][:world] if world == 3 else [2, 1]
        local = torch.full((counts[rank], 3), float(rank)) + torch.arange(3.)
        parts = bdist.all_gather_ragged(local, counts)
        for r in range(world):
            assert parts[r].shape == (counts[r], 3) and (counts[r] == 0 or parts[r][0, 0] == r)
        rc = RenderConfig.enerf_pretrain(K)
        kb = list(range(K))
        out = FakeRenderer(FakeNet(rc, kb)).forward(_scene())
        ret[rank] = {k: v.clone() for k, v in out.items()}
    finally:
        dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _single_process(K):
    """world_size 1 through the same code path (gloo group of one)."""
    port = _free_port()
    ret = mp.Manager().dict()
    mp.spawn(_worker_single, args=(port, K, ret), nprocs=1, join=True)
    return ret[0]


def _worker_single(rank, port, K, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        rc = RenderConfig.enerf_pretrain(K)
        out = FakeRenderer(FakeNet(rc, list(range(K)))).forward(_scene())
        ret[0] = {k: v.clone() for k, v in out.items()}
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,K", [(2, 4), (2, 3), (3, 2)])
def test_sharded_frame_assembly_matches_single_process(world, K):
    ref = _single_process(K)
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), K, ret), nprocs=world, join=True)
    assert sorted(ret.keys()) == list(range(world))
    for r in range(world):
        assert sorted(ret[r].keys()) == sorted(ref.keys())
        for k in ref:
            assert torch.equal(ret[r][k], ref[k]), f"rank {r} {k} differs from the single-process frame"
    assert ref["rgb_level1"].shape == (1, 32 * 64, 3) and ref["rgb_level0"].shape == (1, 8 * 16, 3)
