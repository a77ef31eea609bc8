"""CPU: the input pipeline (phoenix_b200/io.py, SURVEY 8 f4) on synthetic files."""
import os

import numpy as np
import torch

from phoenix_b200 import io as pio


def _write_expression_csv(path, dim, lengths, rng):
    with open(path, "w") as fh:
        width = max(lengths)
        fh.write(",".join([str(dim), str(len(lengths))] + [""] * (width - 2)) + "\n")
        for T in lengths:
            vals = rng.random((dim, T))
            for r in vals:
                fh.write(",".join("%.9g" % v for v in r) + "\n")
            fh.write(",".join("%g" % (2.5 * i) for i in range(T)) + "\n")


def test_readcsv_synthetic_shapes_and_values(tmp_path):
    rng = np.random.default_rng(3)
    fp = os.path.join(str(tmp_path), "x.csv")
    _write_expression_csv(fp, 7, [5, 3], rng)
    data_np, data_pt, t_np, t_pt, dim, ntraj, d0_np, d0_pt = pio.readcsv(fp, "cpu", 0, 2.0)
    assert (dim, ntraj) == (7, 2)
    assert data_np[0].shape == (5, 1, 7) and data_np[1].shape == (3, 1, 7) and data_np[0].dtype == np.float32
    assert t_pt[1].tolist() == [0.0, 2.5, 5.0] and t_pt[0].dtype == torch.float32
    assert torch.equal(data_pt[0], torch.tensor(data_np[0])) and np.array_equal(data_np[0], d0_np[0])
    raw = np.loadtxt(fp, delimiter=",", skiprows=1, max_rows=7, usecols=range(5))
    assert np.allclose(data_np[0][:, 0, :], (2.0 * raw.T).astype(np.float32))


def test_read_prior_matrix_dense_and_triplets(tmp_path):
    d = os.path.join(str(tmp_path), "dense.csv")
    m = np.zeros((5, 5))
    m[1, 3], m[4, 0] = 1.0, -0.5
    np.savetxt(d, m, delimiter=",")
    assert torch.equal(pio.read_prior_matrix(d), torch.from_numpy(m).float())
    t = os.path.join(str(tmp_path), "trip.csv")
    np.savetxt(t, np.array([[2, 4, 1.0], [5, 1, -0.5]]), delimiter=",")
    assert torch.equal(pio.read_prior_matrix(t, sparse=True, num_genes=5), torch.from_numpy(m).float())

