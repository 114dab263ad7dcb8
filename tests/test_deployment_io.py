"""Deployment containers (SURVEY §8f rank 4): deployment.npy layout and the .bin [dtype, numel] files."""
import os
import types

import numpy as np
import pytest
import torch

DEPLOY_CFG = dict(scale=0.5, pos_encoder_type='hash', levels=4, feature_per_level=4, base_res=32, max_res=128,
                  log2_T=21, xyz_net_width=16, rgb_net_width=16, rgb_net_depth=1)   # reference train.py:88-99


def _model(seed):
    from modules.networks import NGP
    torch.manual_seed(seed)
    m = NGP(**DEPLOY_CFG)
    with torch.no_grad():
        m.pos_encoder.hash_table.uniform_(-1, 1)
        m.density_bitfield.copy_(torch.randint(0, 256, m.density_bitfield.shape, dtype=torch.uint8))
    return m


def test_bin_container_round_trip_and_errors(tmp_path):
    from modules.utils import read_aot_array, write_aot_array
    rng = np.random.default_rng(0)
    for i, dt in enumerate([np.float32, np.float16, np.int32, np.int16, np.uint32, np.uint16]):
        a = (rng.random(37) * 100).astype(dt)
        p = write_aot_array(str(tmp_path), a.reshape(37, 1), f"a{i}")
        raw = np.fromfile(p, dtype=np.uint8)
        assert list(raw[:8].view(np.int32)) == [i, 37]                     # header: dtype code, numel
        assert raw.size == 8 + a.nbytes
        b = read_aot_array(p)
        assert b.dtype == dt and np.array_equal(a, b)
    with pytest.raises(TypeError):
        write_aot_array(str(tmp_path), np.zeros(3, np.float64), "bad")
    p = write_aot_array(str(tmp_path), np.zeros(4, np.float32), "trunc")
    with open(p, "r+b") as f:
        f.truncate(8 + 12)
    with pytest.raises(ValueError, match="invalid buffer size"):
        read_aot_array(p)
    with open(p, "r+b") as f:
        f.write(np.array([9], np.int32).tobytes())
    with pytest.raises(ValueError, match="invalid buffer dtype"):
        read_aot_array(p)


def test_deployment_npy_and_bin_round_trip(tmp_path):
    from modules.utils import export_aot_weights, load_deployment_model, save_deployment_model
    src = _model(1)
    ds = types.SimpleNamespace(poses=torch.randn(25, 3, 4))
    save_deployment_model(src, ds, str(tmp_path))
    blob = np.load(os.path.join(tmp_path, 'deployment.npy'), allow_pickle=True).item()
    # layout the mobile kernels index (deployment/InstantNGP/taichi_ngp/kernels.py:449-518): 16x16 | 16x16, 16x32 | 16x16
    assert blob['model.xyz_encoder.params'].shape == (512,) and blob['model.rgb_net.params'].shape == (768,)
    assert np.all(blob['model.rgb_net.params'][512 + 48:] == 0)          # rows 3..15 of the padded output layer
    assert blob['model.hash_encoder.params'].size == src.pos_encoder.hash_table.numel()

    dst = _model(2)
    extra = load_deployment_model(dst, os.path.join(tmp_path, 'deployment.npy'))
    assert extra['poses'].shape == (25, 3, 4)
    for (k, a), b in zip(src.state_dict().items(), dst.state_dict().values()):
        if k.startswith(('pos_encoder', 'xyz_encoder', 'rgb_net', 'density_bitfield')):
            assert torch.equal(a, b), k

    export_aot_weights(blob, str(tmp_path / 'aot'), directions=np.ones((6, 3), np.float32))
    assert sorted(os.listdir(tmp_path / 'aot')) == ['density_bitfield.bin', 'directions.bin', 'hash_embedding.bin',
                                                    'pose.bin', 'rgb_weights.bin', 'sigma_weights.bin']
    dst2 = _model(3)
    extra = load_deployment_model(dst2, str(tmp_path / 'aot'))
    assert np.array_equal(extra['pose'].reshape(3, 4), ds.poses[20].numpy())   # taichi_ngp.py:84-85 ships pose 20
    for (k, a), b in zip(src.state_dict().items(), dst2.state_dict().values()):
        if k.startswith(('pos_encoder', 'xyz_encoder', 'rgb_net', 'density_bitfield')):
            assert torch.equal(a, b), k
    with pytest.raises(ValueError):
        from modules.networks import NGP
        load_deployment_model(NGP(scale=0.5), blob)                            # stock architecture: shapes differ


def test_shipped_lego_files_load_into_the_model(tmp_path):
    """A folder of .bin files in the reference's container format: the small files are the shipped ones byte for byte,
    the table and the bitfield carry the shipped headers over the stored part of the model (oracle/kat_lego.py), and
    directions.bin holds the stored view's camera directions (a subsample of the shipped file) under its own header."""
    from modules.networks import NGP
    from modules.utils import load_deployment_model, read_aot_array
    from oracle import kat_lego
    P = kat_lego.load_part()
    z = P["raw"]
    head = {str(n): h for n, h in zip(z["bin_names"], z["bin_headers"])}
    payload = {"sigma_weights": z["sigma_weights_bin"][8:], "rgb_weights": z["rgb_weights_bin"][8:],
               "pose": z["pose_bin"][8:], "hash_embedding": P["table"], "density_bitfield": P["bits"]}
    for n, a in payload.items():
        with open(tmp_path / (n + ".bin"), "wb") as f:
            f.write(head[n].astype(np.int32).tobytes() + np.ascontiguousarray(a).tobytes())
    with open(tmp_path / "directions.bin", "wb") as f:
        f.write(np.array([head["directions"][0], P["directions"].size], np.int32).tobytes() + P["directions"].tobytes())
    m = NGP(**DEPLOY_CFG)
    extra = load_deployment_model(m, str(tmp_path))
    assert extra['pose'].size == 12 and np.array_equal(extra['pose'].reshape(3, 4), P["pose"])
    assert np.array_equal(extra['model.directions'], P["directions"].reshape(-1))
    emb = read_aot_array(str(tmp_path / "hash_embedding.bin"))
    assert torch.equal(m.pos_encoder.hash_table.detach().reshape(-1), torch.from_numpy(emb.copy()))
    assert np.array_equal(m.density_bitfield.numpy(), P["bits"])
    assert torch.equal(m.xyz_encoder.hidden_layers[0].weight.detach().reshape(-1), torch.from_numpy(P["sigma_w"][:256]))
