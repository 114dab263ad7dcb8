"""Known-answer test against the reference's shipped trained Lego deployment model (the part of it stored in
tests/golden/lego_part.npz, see oracle/kat_lego.py)."""
import json
import os

import numpy as np

from conftest import GOLDEN
from oracle import kat_lego


def test_oracle_renders_the_shipped_lego_model():
    P = kat_lego.load_part()
    rgb, opacity, spr, counts = kat_lego.render(P["table"], P["sigma_w"], P["rgb_w"], P["bits"], P["pose"],
                                                P["directions"])
    # the oracle's rendering of the same view with the full shipped table (tests/golden/make_golden.py)
    np.testing.assert_allclose(rgb, P["gold_rgb"], atol=1e-5)
    np.testing.assert_allclose(opacity, P["gold_opacity"], atol=1e-5)
    st, gold = kat_lego.stats(rgb, opacity, spr), kat_lego.stats(P["gold_rgb"], P["gold_opacity"], spr)
    # a trained scene is (almost) binary in opacity; wrong hash indexing / weight layout gives fog.  The box that cuts
    # the part out of the scene leaves a rim of partly covered pixels, hence more than the whole model's 1.5 %
    assert st["semi_transparent_fraction"] < 0.1
    assert 0.3 < st["coverage"] < 0.5 and abs(st["coverage"] - gold["coverage"]) < 0.03
    assert np.allclose(st["object_mean_rgb"], gold["object_mean_rgb"], atol=0.03)
    r, g, b = st["object_mean_rgb"]
    assert r > g > b and r - b > 0.15         # the yellow bulldozer on the tan base plate
    # opaque pixels can only occur where marching produced samples inside the trained occupancy grid
    assert not (opacity[counts == 0] > 1e-6).any()
    # image is not noise: neighbouring pixels agree (total variation far below that of random colours)
    tv = np.abs(np.diff(rgb, axis=0)).mean() + np.abs(np.diff(rgb, axis=1)).mean()
    assert tv < 0.2   # uniform-random colours give ~0.67


def test_deployment_bin_container_and_layout():
    P = kat_lego.load_part()
    z = P["raw"]
    head = {str(n): (int(c), int(k), int(s)) for n, (c, k), s in zip(z["bin_names"], z["bin_headers"], z["bin_sizes"])}
    itemsize = {0: 4, 1: 2, 2: 4, 3: 2, 4: 4, 5: 2}
    for n, (code, numel, size) in head.items():
        assert size == 8 + numel * itemsize[code], n                  # [int32 dtype][int32 numel][payload]
    assert head["hash_embedding"][:2] == (0, kat_lego.deployment_layout().total_param_size)   # float32 table
    assert head["density_bitfield"][1] * itemsize[head["density_bitfield"][0]] == 128 ** 3 // 8
    assert head["directions"][1] == 600 * 300 * 3
    assert P["sigma_w"].dtype == np.float32 and P["sigma_w"].size == 512
    assert P["rgb_w"].size == 768 and P["pose"].size == 12
    with open(os.path.join(GOLDEN, "layout_constants.json")) as f:
        assert np.allclose(P["pose"], json.load(f)["deployment_pose"])
