"""Host-side pieces of station-array runs (no GPU): the stations-file loader and the sharding of
(station, chain) pairs over ranks."""
import numpy as np
import pytest
from rfsurfhmc_b200.distributed import gather_chains, shard_station_chains
from rfsurfhmc_b200.fixtures import driver_bounds, f1_true_model
from rfsurfhmc_b200.model.stations import load_stations

ND, NP = 197, 14


def _default():
    return driver_bounds(f1_true_model())


def test_loader_accepts_the_documented_shapes(tmp_path):
    S = 3
    dobs = np.arange(S * ND, dtype=float).reshape(S, ND)
    st = load_stations({"dobs": dobs}, ND, NP, _default())
    assert st["names"] == ["station0000", "station0001", "station0002"]
    assert np.array_equal(st["sigma1"], np.ones(S)) and np.array_equal(st["sigma2"], np.ones(S))
    assert st["bounds"].shape == (S, NP, 2) and all(np.array_equal(b, _default()) for b in st["bounds"])
    bounds = np.repeat(_default()[None], S, axis=0) * np.array([1.0, 0.9, 1.1])[:, None, None]
    path = tmp_path / "st.npz"
    np.savez(path, dobs=dobs, names=np.array(["A", "B", "C"]), sigma1=[1.0, 2.0, 3.0], sigma2=[0.5, 0.5, 1.0],
             bounds=bounds)
    st = load_stations(str(path), ND, NP, _default())
    assert st["names"] == ["A", "B", "C"] and st["sigma1"].tolist() == [1.0, 2.0, 3.0]
    assert np.array_equal(st["dobs"], dobs) and np.array_equal(st["bounds"], bounds)


@pytest.mark.parametrize("patch,key", [
    ({"dobs": None}, "dobs"),
    ({"dobs": np.zeros(ND)}, "dobs"),
    ({"dobs": np.zeros((2, ND + 1))}, "dobs"),
    ({"names": np.array(["a"])}, "names"),
    ({"names": np.array(["a", "a"])}, "names"),
    ({"names": np.array(["a", "x/y"])}, "names"),
    ({"sigma1": np.ones(3)}, "sigma1"),
    ({"sigma2": np.array([1.0, 0.0])}, "sigma2"),
    ({"bounds": np.zeros((2, NP - 2, 2))}, "bounds"),
    ({"bounds": np.zeros((NP, 2))}, "bounds"),
])
def test_loader_rejects_wrong_shapes_naming_the_key(patch, key):
    src = {"dobs": np.zeros((2, ND))}
    src.update(patch)
    src = {k: v for k, v in src.items() if v is not None}
    with pytest.raises(ValueError, match=f"'{key}'"):
        load_stations(src, ND, NP, _default())


@pytest.mark.parametrize("S,K", [(1, 1), (3, 4), (5, 3), (7, 2), (2, 9)])
def test_station_chain_sharding_covers_every_pair_once(S, K):
    for ws in range(1, 9):
        if S * K < ws:
            continue
        pairs = []
        for r in range(ws):
            sta, cid = shard_station_chains(S, K, r, ws)
            assert len(sta) == len(cid) >= 1
            pairs += list(zip(sta.tolist(), cid.tolist()))
        # rank order concatenated = station-major order, which is what gather_chains returns
        assert pairs == [(s, k) for s in range(S) for k in range(K)], (S, K, ws)
    sta, cid = shard_station_chains(S, K, 0, 1)
    assert np.array_equal(gather_chains(np.stack([sta, cid], 1), S * K), np.stack([sta, cid], 1))
