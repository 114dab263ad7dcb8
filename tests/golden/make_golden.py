"""Generates the small golden fixtures under tests/golden/ from a checkout of the reference project.

    python tests/golden/make_golden.py <reference checkout>

Outputs (committed):
  lego_bitfield.npz      — the trained Lego occupancy bitfield shipped with the reference's mobile
                           demo (deployment/InstantNGP/taichi_ngp/compiled/density_bitfield.bin,
                           128^3 bits, 3.94 % occupied), zlib-compressed.  Used as the "occupancy (A)"
                           workload of BASELINE.md §4 and as a real-world marching fixture.
  layout_constants.json  — hash-layout constants printed by the reference itself
                           (notebooks/pipeline.ipynb cell 1; deployment/InstantNGP/utils/app_fp32.cpp:70-71).
  lego_part.npz          — the part of the shipped trained Lego model inside one box of the occupancy grid
                           (oracle/kat_lego.py): the hash-table entries its cells read, the small .bin files
                           verbatim, the headers of all six, the camera directions of one view of the part and the
                           oracle's rendering of that view made with the FULL shipped table.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import kat_lego  # noqa: E402

LEGO_FILES = ("hash_embedding", "sigma_weights", "rgb_weights", "density_bitfield", "pose", "directions")
BOX_LO, BOX_HI = (40, 40, 40), (64, 64, 64)   # 2976 occupied cells, 8.5 k table entries: ~140 KB
VIEW_STEP = 4                                   # every 4th pixel of the shipped 300x600 directions


def make_part(comp):
    raw = {n: np.fromfile(os.path.join(comp, n + ".bin"), dtype=np.uint8) for n in LEGO_FILES}
    table = kat_lego.parse_bin(raw["hash_embedding"])
    sigma_w, rgb_w = kat_lego.parse_bin(raw["sigma_weights"]), kat_lego.parse_bin(raw["rgb_weights"])
    pose = kat_lego.parse_bin(raw["pose"]).reshape(3, 4)
    bits = kat_lego.restrict_bitfield(kat_lego.parse_bin(raw["density_bitfield"]).view(np.uint8), BOX_LO, BOX_HI)
    directions = kat_lego.parse_bin(raw["directions"]).reshape(600, 300, 3)[::VIEW_STEP, ::VIEW_STEP]

    # the view: the rows / columns of the shipped camera in which the part is visible, plus a margin
    _, opacity, _, _ = kat_lego.render(table, sigma_w, rgb_w, bits, pose, directions)
    rows, cols = np.nonzero((opacity > 1e-3).any(1))[0], np.nonzero((opacity > 1e-3).any(0))[0]
    r0, r1 = max(rows[0] - 3, 0), min(rows[-1] + 4, directions.shape[0])
    c0, c1 = max(cols[0] - 3, 0), min(cols[-1] + 4, directions.shape[1])
    directions = np.ascontiguousarray(directions[r0:r1, c0:c1])
    rgb, opacity, _, _ = kat_lego.render(table, sigma_w, rgb_w, bits, pose, directions)

    occupied = np.nonzero(np.unpackbits(bits, bitorder='little'))[0]
    idx = kat_lego.entries_read_by_cells(occupied)
    sparse = np.zeros_like(table).reshape(-1, 4)
    sparse[idx] = table.reshape(-1, 4)[idx]
    rgb2, opacity2, _, _ = kat_lego.render(sparse.reshape(-1), sigma_w, rgb_w, bits, pose, directions)
    assert np.array_equal(rgb, rgb2) and np.array_equal(opacity, opacity2), "kept entries miss some the part reads"

    np.savez_compressed(
        os.path.join(HERE, "lego_part.npz"),
        box_lo=np.array(BOX_LO, np.int32), box_hi=np.array(BOX_HI, np.int32),
        hash_index=idx, hash_values=table.reshape(-1, 4)[idx],
        bin_names=np.array(LEGO_FILES), bin_headers=np.stack([raw[n][:8].view(np.int32) for n in LEGO_FILES]),
        bin_sizes=np.array([raw[n].size for n in LEGO_FILES], np.int64),
        sigma_weights_bin=raw["sigma_weights"], rgb_weights_bin=raw["rgb_weights"], pose_bin=raw["pose"],
        directions=directions, gold_rgb=rgb, gold_opacity=opacity)
    print("part:", occupied.size, "cells,", idx.size, "entries, view", directions.shape[:2],
          kat_lego.stats(rgb, opacity, 0))


def main(ref):
    comp = os.path.join(ref, "deployment/InstantNGP/taichi_ngp/compiled")
    bits = kat_lego.read_bin(os.path.join(comp, "density_bitfield.bin")).view(np.uint8)
    assert bits.size == 128 ** 3 // 8
    np.savez_compressed(os.path.join(HERE, "lego_bitfield.npz"), bitfield=bits)
    pose = kat_lego.read_bin(os.path.join(comp, "pose.bin")).reshape(3, 4)

    # constants the reference prints / hard-codes
    consts = {
        "source": {
            "lego_16_1024": "notebooks/pipeline.ipynb cell 1 (per_level_scale, offset_, total_hash_size)",
            "deployment": "deployment/InstantNGP/utils/app_fp32.cpp:70-71, taichi_ngp/kernels.py (offsets)",
        },
        "lego_16_1024": {"per_level_scale": 1.3195079107728942, "total_entries": 5710032,
                         "total_params": 11420064},
        "deployment": {"total_params": 11176096, "offsets_entries": [0, 32768, 165424, 696872]},
        "deployment_pose": pose.tolist(),
        "bitfield_occupied_fraction": float(np.unpackbits(bits).mean()),
    }
    with open(os.path.join(HERE, "layout_constants.json"), "w") as f:
        json.dump(consts, f, indent=1)
    print("bitfield occupied:", consts["bitfield_occupied_fraction"])
    make_part(comp)


if __name__ == "__main__":
    main(sys.argv[1])
