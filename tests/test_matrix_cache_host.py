"""CPU suite: the matrix-cache file read as CSC arrays (api.deserialize_csc) holds exactly what the dense reader
(api.deserialize_mat) gives, in the reference's byte layout, without a dense matrix being built."""
import numpy as np
import pytest


@pytest.mark.parametrize("N,density", [(1, 1.0), (2, 0.0), (33, 0.3), (257, 0.31), (1000, 0.05)])
def test_deserialize_csc_equals_dense_reader(tmp_path, N, density):
    from daisyriot_b200 import api
    rng = np.random.RandomState(N)
    mask = rng.uniform(0, 1, (N, N)) < density
    F = np.where(mask, rng.uniform(1e-6, 1.0, (N, N)), 0.0).astype(np.float32)
    cols, rows = np.nonzero(mask.T)
    vals = F[rows, cols]
    outer = np.concatenate([[0], np.cumsum(mask.sum(axis=0))]).astype(np.int32)
    path = str(tmp_path / "radmat.bin")
    api.serialize_mat(path, vals, rows.astype(np.int32), outer, N)
    v, i, o = api.deserialize_csc(path)
    assert v.dtype == np.float32 and i.dtype == np.int32 and o.dtype == np.int32
    assert o.size == N + 1 and o[N] == v.size == i.size  # the closing sentinel the file does not store
    dense = np.zeros((N, N), np.float32)
    for c in range(N):
        dense[i[o[c]:o[c + 1]], c] = v[o[c]:o[c + 1]]
    assert np.array_equal(dense.view(np.uint32), api.deserialize_mat(path).view(np.uint32))
    assert np.array_equal(dense.view(np.uint32), F.view(np.uint32))


def test_deserialize_csc_rejects_a_truncated_file(tmp_path):
    from daisyriot_b200 import api
    path = str(tmp_path / "radmat.bin")
    api.serialize_mat(path, np.ones(3, np.float32), np.arange(3, dtype=np.int32), np.array([0, 3, 3, 3], np.int32), 3)
    data = open(path, "rb").read()
    open(path, "wb").write(data[:-4])
    with pytest.raises(ValueError):
        api.deserialize_csc(path)
