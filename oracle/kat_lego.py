"""Known-answer test: render the reference's SHIPPED, TRAINED Lego deployment model through the oracle.

The only real fixture the reference ships is its mobile-demo model
(deployment/InstantNGP/taichi_ngp/compiled/*.bin: hash grid L=4 F=4 32->128 T=2^21, 16-wide MLPs,
occupancy bitfield, pose, pixel directions).  Rendering it end to end with the oracle's
ray/AABB -> march -> dense hash indexing -> SH -> MLP weight layout -> compositing
(restating deployment/InstantNGP/taichi_ngp/kernels.py:262-571 and new_kernels.py:4-18) must produce
the yellow Lego bulldozer; any indexing / layout mistake produces noise.

The 44 MB hash table is too large to keep in the repository, so the tests use a part of the model: the occupied
cells inside one box of the 128^3 occupancy grid, with the hash-table entries that any point of those cells reads
(every other entry is zero and is never read, because marching only samples occupied cells).  That part renders
exactly as the full model does wherever the full model's rays only meet kept cells.  tests/golden/make_golden.py
cuts it from the shipped files into tests/golden/lego_part.npz, together with the reference's small .bin files
verbatim and the oracle's rendering of the part made with the full table.
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PART = os.path.join(ROOT, "tests", "golden", "lego_part.npz")
GRID = 128


def read_bin(path):
    """[int32 dtype][int32 numel][payload]  (taichi_ngp.py:34-65, utils.cpp:100-120)."""
    return parse_bin(np.fromfile(path, dtype=np.uint8))


def parse_bin(raw):
    code, numel = raw[:8].view(np.int32)
    dt = {0: np.float32, 1: np.float16, 2: np.int32, 3: np.int16, 4: np.uint32, 5: np.uint16}[int(code)]
    return raw[8:].view(dt)[:numel]


def deployment_layout():
    sys.path.insert(0, ROOT)
    from taichi_nerfs_b200.layout import make_hash_layout
    return make_hash_layout(2 ** 21, 4, 32, 128, 4)


def box_cells(lo, hi):
    """Morton indices of the cells of the occupancy grid with lo <= (x, y, z) < hi."""
    sys.path.insert(0, ROOT)
    from oracle import oracle as O
    axes = [np.arange(a, b, dtype=np.int32) for a, b in zip(lo, hi)]
    xyz = np.stack(np.meshgrid(*axes, indexing='ij'), -1).reshape(-1, 3)
    return O.morton3d(xyz)


def restrict_bitfield(bits, lo, hi):
    """The occupancy bitfield with every cell outside the box cleared."""
    keep = np.zeros(GRID ** 3, np.uint8)
    keep[box_cells(lo, hi)] = 1
    return bits & np.packbits(keep, bitorder='little')


def entries_read_by_cells(cells):
    """Sorted indices of the hash-table entries (rows of 4 features) that any point of the given occupancy cells
    reads: the 27 points {0, 1/2, 1}^3 of a cell reach every grid cell of every level that the cell overlaps."""
    sys.path.insert(0, ROOT)
    from oracle import oracle as O
    lay = deployment_layout()
    u = np.array([0, 0.5, 1], np.float32)
    off = np.stack(np.meshgrid(u, u, u, indexing='ij'), -1).reshape(-1, 3)
    c = O.morton3d_invert(np.asarray(cells, np.int32)).astype(np.float32)
    p = np.clip(((c[:, None, :] + off[None]) / GRID).reshape(-1, 3), 0, 1).astype(np.float32)
    g = O.hash_encode_bwd(p, np.ones((p.shape[0], lay.out_dim), np.float32), lay)
    return np.nonzero(g.reshape(-1, 4).any(1))[0].astype(np.uint32)


def load_part(path=PART):
    """The stored part of the shipped model: dense table (zeros outside the kept entries), MLP weights, the box's
    occupancy bitfield, pose, the camera directions of the stored view and the oracle's golden rendering of it."""
    z = np.load(path)
    lay = deployment_layout()
    table = np.zeros((lay.total_param_size // 4, 4), np.float32)
    table[z["hash_index"]] = z["hash_values"]
    bits = np.load(os.path.join(ROOT, "tests", "golden", "lego_bitfield.npz"))["bitfield"]
    part = {"table": table.reshape(-1), "sigma_w": parse_bin(z["sigma_weights_bin"]),
            "rgb_w": parse_bin(z["rgb_weights_bin"]), "pose": parse_bin(z["pose_bin"]).reshape(3, 4),
            "bits": restrict_bitfield(bits, z["box_lo"], z["box_hi"]), "directions": z["directions"],
            "gold_rgb": z["gold_rgb"], "gold_opacity": z["gold_opacity"], "raw": z}
    # the deployment.npy keys of modules.utils.load_deployment_model
    part["blob"] = {"model.hash_encoder.params": part["table"], "model.xyz_encoder.params": part["sigma_w"],
                    "model.rgb_net.params": part["rgb_w"], "model.density_bitfield": part["bits"],
                    "pose": part["pose"]}
    return part


def sh16(d):
    sys.path.insert(0, ROOT)
    from oracle import oracle as O
    return O.dir_encode(d)


def deployment_mlp(emb, dirs, sigma_w, rgb_w):
    """sigma_rgb_layer, kernels.py:449-518: sigma net 16->16(relu)->16, rgb net [SH16|h16]->16(relu)->3."""
    W1 = sigma_w[:256].reshape(16, 16)          # temp_i = sum_j emb_j * w[i*16+j]
    W2 = sigma_w[256:512].reshape(16, 16)       # out_j += relu(temp_i) * w[256 + j*16 + i]
    h = np.maximum(emb @ W1.T, 0) @ W2.T
    sigma = np.exp(h[:, 0])
    d = dirs / np.linalg.norm(dirs, axis=1, keepdims=True)
    sh = sh16(((d + 1) / 2).astype(np.float32))  # dir_encode_func, kernels.py:139-172
    x = np.concatenate([sh, h], 1).astype(np.float32)
    W3 = rgb_w[:512].reshape(16, 32)
    W4 = rgb_w[512:512 + 48].reshape(3, 16)     # s_c += relu(temp_i) * w[512 + c*16 + i]
    o = np.maximum(x @ W3.T, 0) @ W4.T
    return sigma.astype(np.float32), (1 / (1 + np.exp(-o))).astype(np.float32)


def render(table, sigma_w, rgb_w, bits, pose, directions, T_threshold=1e-2, max_samples=1024):
    """(rgb [h, w, 3], opacity [h, w], samples per ray, samples [h, w]) of the camera directions [h, w, 3]."""
    sys.path.insert(0, ROOT)
    from oracle import oracle as O
    lay = deployment_layout()
    assert lay.total_param_size == table.size

    h, w = directions.shape[:2]
    dirs_cam = directions.reshape(-1, 3)
    rays_d = (dirs_cam @ pose[:, :3].T).astype(np.float32)        # new_kernels.py:12
    rays_o = np.tile(pose[:, 3], (rays_d.shape[0], 1)).astype(np.float32)
    hits = O.ray_aabb_intersect(rays_o, rays_d, 0.5)
    noise = np.zeros(rays_d.shape[0], np.float32)
    rays_a, xyzs, sdirs, deltas, ts, S = O.raymarching_train(rays_o, rays_d, hits, bits, noise, 1, 0.5, 0.0, GRID,
                                                             max_samples)
    emb = O.hash_encode_fwd((xyzs + 0.5).astype(np.float32), table, lay)  # kernels.py:397 (xyz + 0.5)
    sigma, rgbs = deployment_mlp(emb, sdirs, sigma_w, rgb_w)
    tot, opacity, depth, rgb, ws = O.composite_train_fwd(sigma, rgbs, deltas, ts, rays_a, T_threshold)
    return rgb.reshape(h, w, 3), opacity.reshape(h, w), S / rays_d.shape[0], rays_a[:, 2].reshape(h, w)


def stats(rgb, opacity, spr):
    obj = opacity > 0.5
    col = rgb[obj].mean(0) / np.maximum(opacity[obj].mean(), 1e-6)
    return {"coverage": float(obj.mean()), "semi_transparent_fraction": float(((opacity > 0.05) & (opacity < 0.95)).mean()),
            "object_mean_rgb": [float(c) for c in col], "samples_per_ray": float(spr),
            "opacity_max": float(opacity.max())}
