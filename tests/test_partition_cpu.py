"""Row partitioning and shard extraction of the sharded path, on the CPU: work-balanced bounds that
match the oracle, and shards that concatenate back to the global arrays bit for bit."""
import numpy as np
import pytest


@pytest.mark.parametrize("scale", [9, 12])
def test_partition_and_shard_round_trip(sp, orc, scale):
    import gpu_spmv_b200.dist as D
    import gpu_spmv_b200.gen as gen
    n, rp, ci, va = gen.rmat_pagerank_csr(scale, 8, 11, "cpu")
    for parts in (2, 3, 8):
        bounds = D.partition_rows(rp, parts)
        assert bounds == orc.partition_rows(n, rp.numpy(), parts).tolist()
        assert gen.partition_bounds(rp, parts) == bounds  # the rule partition_rows applies to CUDA tensors
        pieces = [D.extract_shard(rp, ci, va, bounds[p], bounds[p + 1]) for p in range(parts)]
        assert np.array_equal(np.concatenate([p[1].numpy() for p in pieces]), ci.numpy())
        assert np.array_equal(np.concatenate([p[2].numpy() for p in pieces]).view(np.uint32), va.numpy().view(np.uint32))
        rebuilt = np.concatenate([[0]] + [p[0].numpy()[1:] + rp.numpy()[bounds[i]] for i, p in enumerate(pieces)])
        assert np.array_equal(rebuilt, rp.numpy())


def test_partition_properties(sp, orc):
    """Bounds are monotone, cover all rows, balance nnz, and match the oracle."""
    rng = np.random.default_rng(3)
    for _ in range(50):
        rows = int(rng.integers(1, 500))
        lens = rng.integers(0, 30, rows)
        if rng.random() < 0.3:
            lens[int(rng.integers(0, rows))] = 5000
        rp = np.zeros(rows + 1, np.int32)
        rp[1:] = np.cumsum(lens)
        for parts in (1, 2, 3, 8):
            for w in (1, 3):  # (rows + nnz)-balanced variants match the oracle and stay monotone
                bw = sp.partition_rows(rp, rows, parts, w)
                assert bw[0] == 0 and bw[-1] == rows and np.all(np.diff(bw) >= 0)
                assert np.array_equal(bw, orc.partition_rows(rows, rp, parts, w))
            b = sp.partition_rows(rp, rows, parts)
            assert b[0] == 0 and b[-1] == rows and np.all(np.diff(b) >= 0)
            assert np.array_equal(b, orc.partition_rows(rows, rp, parts))
            nnz = int(rp[-1])
            for p in range(1, parts):
                assert rp[b[p]] >= (nnz * p) // parts and (b[p] == 0 or rp[b[p] - 1] < (nnz * p) // parts or b[p] == b[p - 1])


def test_merge_path_search_matches_oracle(sp, orc):
    rng = np.random.default_rng(4)
    for _ in range(20):
        rows = int(rng.integers(1, 60))
        lens = rng.integers(0, 9, rows)
        rp = np.zeros(rows + 1, np.int32)
        rp[1:] = np.cumsum(lens)
        nnz = int(rp[-1])
        for d in range(rows + nnz + 1):
            assert sp.merge_path_search(d, rp, rows, nnz) == orc.merge_path_search(d, rp, rows, nnz)
    with pytest.raises(ValueError):
        sp.merge_path_search(rows + nnz + 1, rp, rows, nnz)
