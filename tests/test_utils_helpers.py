"""CPU: the input-side helpers (SURVEY 8f rank 1) against a dense restatement of the reference algorithm
(utils.py:92-110) and, when the reference checkout is present, against the reference functions themselves."""
import argparse

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import utils as U


def _dense_add_noisy_edges(adj, noise_level):
    """reference utils.py:92-110 restated densely (np.float -> float)."""
    level = noise_level * 10
    np.random.seed(0)
    adj = sp.coo_matrix(adj)
    noise = (np.random.rand(adj.shape[0], adj.shape[1]) < level).astype(float)
    mask = np.ones(adj.shape)
    mask[adj.row, adj.col] = 0
    mask[np.arange(len(mask)), np.arange(len(mask))] = 0
    return sp.csr_matrix(adj + noise * mask)


def _graph(n, m, seed):
    rng = np.random.RandomState(seed)
    r, c = rng.randint(0, n, m), rng.randint(0, n, m)
    keep = r != c
    a = sp.coo_matrix((np.ones(keep.sum()), (r[keep], c[keep])), shape=(n, n))
    a.sum_duplicates()
    a.data[:] = 1.0
    return a


@pytest.mark.parametrize("n,level,chunk", [(300, 0.002, 64), (1000, 0.00014, 1024), (257, 0.01, 100)])
def test_add_noisy_edges_matches_dense_reference_algorithm(n, level, chunk):
    a = _graph(n, 4 * n, n)
    U._NOISY_CACHE.clear()
    got = U.add_noisy_edges(a, noise_level=level, chunk_rows=chunk)
    want = _dense_add_noisy_edges(a, level)
    assert (got != want).nnz == 0
    assert got.nnz > a.nnz                      # some noise was added
    again = U.add_noisy_edges(a, noise_level=level)   # memoised path
    assert (again != want).nnz == 0


def test_add_noisy_edges_matches_reference_module():
    from oracle import ref_loader

    if not ref_loader.reference_available():
        pytest.skip("no reference checkout (set DGG_REFERENCE_ROOT)")
    ref = ref_loader.load_reference(("utils",))["utils"]
    a = _graph(400, 1500, 3)
    U._NOISY_CACHE.clear()
    got = U.add_noisy_edges(a, noise_level=0.001)
    want = ref.add_noisy_edges(a, noise_level=0.001)
    assert (got != want).nnz == 0
    t1 = U.sparse_mx_to_torch_sparse_tensor(got).coalesce()
    t2 = ref.sparse_mx_to_torch_sparse_tensor(want).coalesce()
    assert torch.equal(t1.indices(), t2.indices()) and torch.equal(t1.values(), t2.values())
    out = torch.randn(50, 7)
    lab = torch.randint(0, 7, (50,))
    assert float(U.accuracy(out, lab)) == float(ref.accuracy(out, lab))


def test_str2bool_and_accuracy():
    assert U.str2bool("Yes") is True and U.str2bool("0") is False and U.str2bool(True) is True
    with pytest.raises(argparse.ArgumentTypeError):
        U.str2bool("maybe")
    out = torch.tensor([[0.1, 0.9], [0.8, 0.2], [0.3, 0.7]])
    assert float(U.accuracy(out, torch.tensor([1, 0, 0]))) == pytest.approx(2 / 3)


def test_cached_device_adj_cpu():
    ei = torch.tensor([[0, 1, 2, 3], [1, 0, 3, 2]])
    U._DEVICE_CACHE.clear()
    a = U.cached_device_adj(ei, 5, noise_level=0.0, device="cpu")
    b = U.cached_device_adj(ei, 5, noise_level=0.0, device="cpu")
    assert a is b and a.is_coalesced() and a.shape == (5, 5) and a._nnz() == 4
