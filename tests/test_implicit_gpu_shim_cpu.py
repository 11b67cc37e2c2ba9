"""CPU: the `implicit.gpu` stand-ins (`rectools_b200/implicit_gpu.py`, the lowest seam of SURVEY section 8b) make the UNMODIFIED
reference `ImplicitRanker(..., use_gpu=True)` (rank_implicit.py:148-185, :250-262) produce the same triplets as its CPU path.
The top-k provider behind `KnnQuery.topk` is the oracle here (injected); on a B200 it is the engine (tests/test_gpu_parity.py).
Runs the reference package itself, so it needs it staged in oracle/_ref (`oracle.stage_reference`); skipped without it."""
import numpy as np
import pytest
from scipy import sparse

from oracle import stage_reference

pytestmark = pytest.mark.skipif(not stage_reference.available(), reason="reference package neither staged nor checked out")


def _oracle_backend(items, queries, k, item_norms, csr):
    from oracle.topk_oracle import implicit_topk

    ids, scores = implicit_topk(items, queries, k, item_norms, csr, accum="f32")
    return ids.astype(np.int32), scores.astype(np.float32), (scores > -1e38).sum(axis=1).astype(np.int32)


@pytest.fixture()
def patched():
    added = stage_reference.add_to_path()
    from rectools_b200 import implicit_gpu

    implicit_gpu.patch_implicit_gpu(backend=_oracle_backend)
    import rectools.models.rank.rank_implicit as ri

    yield ri
    implicit_gpu.unpatch_implicit_gpu()
    import implicit.gpu

    assert implicit.gpu.HAS_CUDA is False and ri.HAS_CUDA is False
    stage_reference.remove_from_path(added)


@pytest.mark.parametrize("distance", ["DOT", "COSINE", "EUCLIDEAN"])
@pytest.mark.parametrize("with_filter, with_whitelist", [(False, False), (True, False), (True, True)])
def test_unmodified_ranker_use_gpu_matches_cpu_path(patched, distance, with_filter, with_whitelist):
    ri = patched
    from rectools.models.rank import Distance

    rng = np.random.default_rng(3)
    u = rng.standard_normal((40, 8)).astype(np.float32)
    i = rng.standard_normal((90, 8)).astype(np.float32)
    sids = rng.permutation(40)[:25]
    csr = None
    if with_filter:
        csr = sparse.random(25, 90, density=0.2, random_state=1, format="csr", dtype=np.float32)
        csr.data[:] = 1.0
    wl = np.sort(rng.choice(90, 30, replace=False)) if with_whitelist else None
    dist = getattr(Distance, distance)
    assert ri.HAS_CUDA is True
    cpu = ri.ImplicitRanker(dist, u, i, use_gpu=False).rank(sids, k=7, filter_pairs_csr=csr, sorted_object_whitelist=wl)
    gpu = ri.ImplicitRanker(dist, u, i, use_gpu=True).rank(sids, k=7, filter_pairs_csr=csr, sorted_object_whitelist=wl)
    np.testing.assert_array_equal(np.asarray(cpu[0]), np.asarray(gpu[0]))
    np.testing.assert_array_equal(np.asarray(cpu[1]), np.asarray(gpu[1]))
    np.testing.assert_allclose(np.asarray(cpu[2]), np.asarray(gpu[2]), rtol=1e-5, atol=1e-6)


def test_all_filtered_rows_and_empty_filter(patched):
    ri = patched
    from rectools.models.rank import Distance

    u = np.eye(3, dtype=np.float32)
    i = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 1]], dtype=np.float32)
    full = sparse.csr_matrix(np.ones((3, 4), dtype=np.float32))  # everything viewed: no rows come back
    s, ids, sc = ri.ImplicitRanker(Distance.DOT, u, i, use_gpu=True).rank([0, 1, 2], k=2, filter_pairs_csr=full)
    assert len(s) == len(ids) == len(sc) == 0
    empty = sparse.csr_matrix((3, 4), dtype=np.float32)  # rank_implicit.py:169-173: no COOMatrix is built
    s, ids, sc = ri.ImplicitRanker(Distance.DOT, u, i, use_gpu=True).rank([0, 1, 2], k=2, filter_pairs_csr=empty)
    np.testing.assert_array_equal(ids, [0, 3, 1, 3, 2, 3])
