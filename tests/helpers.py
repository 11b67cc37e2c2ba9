"""Shared helpers for the parity tests (CPU and GPU)."""
import os

import numpy as np
from scipy import sparse

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_rank_case(case: int):
    inp = np.load(os.path.join(GOLDEN, f"rank_inputs_{case}.npz"))
    out = np.load(os.path.join(GOLDEN, f"rank_outputs_{case}.npz"))
    shape = tuple(int(x) for x in inp["csr_shape"])
    csr = sparse.csr_matrix(
        (np.ones(len(inp["csr_indices"]), dtype=np.float32), inp["csr_indices"], inp["csr_indptr"]), shape=shape
    )
    return inp, out, csr


def golden_keys(out):
    return sorted({k.rsplit("|", 1)[0] for k in out.files})


def parse_key(key: str):
    impl, dist, k, f, w = key.split("|")
    k = int(k[1:])
    return impl, dist, (None if k < 0 else k), f == "f1", w == "w1"


def synth_factors(n_users, n_items, d, seed=0):
    """SURVEY §8(d) synthetic inputs: standard_normal / sqrt(d), fp32, fixed seeds."""
    u = (np.random.default_rng(seed).standard_normal((n_users, d), dtype=np.float32) / np.sqrt(d)).astype(np.float32)
    i = (np.random.default_rng(seed + 1).standard_normal((n_items, d), dtype=np.float32) / np.sqrt(d)).astype(np.float32)
    return u, i


def synth_viewed_csr(n_users, n_items, per_user, seed=2):
    """~`per_user` viewed items per user (uniform draws, sorted within a row; rare duplicates are kept -- the filter
    is a set-membership test so they are harmless), int32 indices / int64 indptr, data = ones."""
    rng = np.random.default_rng(seed)
    cols = rng.integers(0, n_items, size=(n_users, per_user), dtype=np.int32)
    cols.sort(axis=1)
    indptr = np.arange(n_users + 1, dtype=np.int64) * per_user
    return sparse.csr_matrix((np.ones(cols.size, np.float32), cols.reshape(-1), indptr), shape=(n_users, n_items))


def ragged_to_padded(subjects, ids, scores, subject_ids, k):
    """Flat (subject, id, score) triplet -> [n, k] id / score arrays + counts (order preserved)."""
    n = len(subject_ids)
    out_ids = np.full((n, k), -1, dtype=np.int64)
    out_sc = np.full((n, k), np.nan, dtype=np.float32)
    counts = np.zeros(n, dtype=np.int64)
    pos = 0
    subjects = np.asarray(subjects)
    for r, sid in enumerate(subject_ids):
        c = 0
        while pos < len(subjects) and subjects[pos] == sid and c < k:
            out_ids[r, c] = ids[pos]
            out_sc[r, c] = scores[pos]
            pos += 1
            c += 1
        counts[r] = c
    return out_ids, out_sc, counts


def assert_same_ranking(ids, scores, ref_ids, ref_scores, rtol=2e-5, atol=2e-6, tie_tol=None, msg=""):
    """ids must be identical; where they differ the two rankings must be a permutation inside a near-tie window
    (`tie_tol`, relative to the score scale) -- the reference leaves tie order undefined (pure_svd.py:78-80)."""
    ids, ref_ids = np.asarray(ids), np.asarray(ref_ids)
    scores, ref_scores = np.asarray(scores, dtype=np.float64), np.asarray(ref_scores, dtype=np.float64)
    assert ids.shape == ref_ids.shape, f"{msg}: shape {ids.shape} vs {ref_ids.shape}"
    np.testing.assert_allclose(scores, ref_scores, rtol=max(rtol, tie_tol or 0), atol=atol, err_msg=msg)
    bad = np.nonzero(ids != ref_ids)[0]
    if len(bad) == 0:
        return 0
    assert tie_tol is not None, f"{msg}: {len(bad)} id mismatches, first at {bad[:5]}"
    scale = max(1e-30, float(np.abs(ref_scores).max()))
    for p in bad:
        # the item the reference put here must sit at a neighbouring position with an (almost) equal score
        assert abs(scores[p] - ref_scores[p]) <= tie_tol * scale, f"{msg}: non-tie mismatch at {p}"
    return len(bad)


class OracleRanker:
    """CPU stand-in with the `B200Ranker` surface the host code uses (`rank`, `rank_padded`), backed by the oracle.  Test
    infrastructure only: it lets the host-side logic around the ranker be checked against the reference without a GPU."""

    def __init__(self, distance, subjects_factors, objects_factors, num_threads=0, use_gpu=False):  # pylint: disable=unused-argument
        self.distance = "dot"  # the oracle returns final scores (COSINE / EUCLIDEAN post-scaling included)
        self._dist = str(getattr(distance, "value", distance))
        self._u = np.asarray(subjects_factors, dtype=np.float32)
        self._i = np.asarray(objects_factors, dtype=np.float32)

    def rank(self, subject_ids, k=None, filter_pairs_csr=None, sorted_object_whitelist=None):
        from oracle.topk_oracle import rank_oracle

        return rank_oracle(self._dist, self._u, self._i, subject_ids, k, filter_pairs_csr, sorted_object_whitelist, accum="f32")

    def rank_padded(self, subject_ids, k=None, filter_pairs_csr=None, sorted_object_whitelist=None, flags=0):  # pylint: disable=unused-argument
        subject_ids = np.asarray(subject_ids, dtype=np.int64)
        n_pos = self._i.shape[0] if sorted_object_whitelist is None else len(sorted_object_whitelist)
        k_out = min(n_pos if k is None else k, n_pos)
        ids = np.full((len(subject_ids), k_out), -1, dtype=np.int32)
        scores = np.full((len(subject_ids), k_out), -np.finfo(np.float32).max, dtype=np.float32)
        counts = np.zeros(len(subject_ids), dtype=np.int32)
        for r, sid in enumerate(subject_ids):
            csr = filter_pairs_csr[r] if filter_pairs_csr is not None else None
            _, oi, os_ = self.rank([sid], k, csr, sorted_object_whitelist)
            counts[r] = len(oi)
            ids[r, : len(oi)] = oi
            scores[r, : len(oi)] = os_
        return subject_ids, ids, scores, counts


class OracleTorchRanker:
    """CPU stand-in with the `TorchRanker` constructor signature (rank_torch.py:59-67), backed by the oracle.  Keeps the torch
    path's filter semantics: CSR VALUES != 0 filter (rank_torch.py:143).  Test infrastructure only."""

    def __init__(self, distance, device, subjects_factors, objects_factors, batch_size=128, dtype=None):  # pylint: disable=unused-argument
        self._dist = str(getattr(distance, "value", distance))
        to_np = lambda t: t.detach().cpu().float().numpy() if hasattr(t, "detach") else np.asarray(t, dtype=np.float32)
        self._u, self._i = to_np(subjects_factors), to_np(objects_factors)

    def rank(self, subject_ids, k=None, filter_pairs_csr=None, sorted_object_whitelist=None):
        from oracle.topk_oracle import rank_oracle

        if filter_pairs_csr is not None:
            filter_pairs_csr = filter_pairs_csr.copy()
            filter_pairs_csr.eliminate_zeros()
        return rank_oracle(self._dist, self._u, self._i, subject_ids, k, filter_pairs_csr, sorted_object_whitelist, accum="f64")


class FakeIdMap:
    """The part of `rectools.dataset.IdMap` (identifiers.py:40-126) the vectorised recommend() touches."""

    def __init__(self, external_ids):
        self.external_ids = np.asarray(external_ids)
        self._to_internal = {e: i for i, e in enumerate(self.external_ids.tolist())}

    @property
    def external_dtype(self):
        return self.external_ids.dtype

    @property
    def size(self):
        return self.external_ids.size


class _Table:  # stands in for the interactions DataFrame (cache key; must be weak-referenceable)
    pass


class FakeDataset:
    """`rectools.dataset.Dataset` surface used by `rectools_b200.recommend` (dataset.py:314-348)."""

    def __init__(self, user_ext, item_ext, ui_csr):
        from types import SimpleNamespace

        self.user_id_map, self.item_id_map = FakeIdMap(user_ext), FakeIdMap(item_ext)
        self.interactions = SimpleNamespace(df=_Table())
        self._csr = ui_csr
        self.n_hot_users = ui_csr.shape[0]
        self.n_matrix_builds = 0

    def get_user_item_matrix(self, include_weights=True):  # pylint: disable=unused-argument
        self.n_matrix_builds += 1
        return self._csr.copy()


class FakeVectorModel:
    """`VectorModel` / `ModelBase` surface used by `rectools_b200.recommend` (base.py:652-733, vector.py:50-79, :136-150)."""

    require_recommend_context = False

    def __init__(self, u2i_dist, user_vectors, item_vectors, i2i_dist="cosine"):
        self.u2i_dist, self.i2i_dist, self._u, self._i = u2i_dist, i2i_dist, user_vectors, item_vectors

    def _check_is_fitted(self):
        pass

    @staticmethod
    def _check_k(k):
        if k <= 0:
            raise ValueError("`k` must be positive integer")

    @staticmethod
    def _custom_transform_dataset_u2i(dataset, users, on_unsupported_targets, context=None):  # pylint: disable=unused-argument
        return dataset

    @staticmethod
    def _get_sorted_item_ids_to_recommend(items_to_recommend, dataset):
        if items_to_recommend is None:
            return None
        m = dataset.item_id_map._to_internal  # pylint: disable=protected-access
        return np.unique([m[i] for i in np.asarray(items_to_recommend).tolist() if i in m])

    @staticmethod
    def _custom_transform_dataset_i2i(dataset, target_items, on_unsupported_targets):  # pylint: disable=unused-argument
        return dataset

    @staticmethod
    def _split_targets_by_hot_warm_cold(targets, dataset, entity):
        id_map = dataset.user_id_map if entity == "user" else dataset.item_id_map
        n_hot = dataset.n_hot_users if entity == "user" else id_map.size
        m = id_map._to_internal  # pylint: disable=protected-access
        t = np.asarray(targets).tolist()
        known = np.asarray([m[x] for x in t if x in m], dtype=np.int64)
        cold = np.asarray([x for x in t if x not in m])
        return known[known < n_hot], known[known >= n_hot], cold

    @staticmethod
    def _check_targets_are_valid(hot, warm, cold, entity, on_unsupported_targets):  # pylint: disable=unused-argument
        return hot, warm, cold

    def _get_u2i_vectors(self, dataset):  # pylint: disable=unused-argument
        return self._u, self._i

    def _get_i2i_vectors(self, dataset):  # pylint: disable=unused-argument
        return self._i, self._i

    def recommend(self, *args, **kwargs):
        raise AssertionError("the vectorised path should not have delegated")

    def recommend_to_items(self, *args, **kwargs):
        raise AssertionError("the vectorised path should not have delegated")


def fake_rectools(monkeypatch):
    """Stand-in modules for the names `rectools_b200.install()` / `make_similarity_module()` rebind or subclass
    (`rectools.models.{vector,ease}.ImplicitRanker`, `VectorModel` / `ModelBase.recommend{,_to_items}`,
    `rectools.models.nn.transformers.similarity.DistanceSimilarityModule`), registered in `sys.modules` for one test.
    Test infrastructure only: the behaviour of the reference behind those names is pinned by tests/golden."""
    import enum
    import sys
    import types

    import torch

    class Distance(enum.Enum):  # rectools/models/rank/rank.py: the values are the contract
        DOT = "dot"
        COSINE = "cosine"
        EUCLIDEAN = "euclidean"

    class ImplicitRanker:  # the stock ranker the two modules import by name
        pass

    class ModelBase:
        def recommend(self, *args, **kwargs):
            raise NotImplementedError

        def recommend_to_items(self, *args, **kwargs):
            raise NotImplementedError

    class VectorModel(ModelBase):
        pass

    class DistanceSimilarityModule(torch.nn.Module):
        def __init__(self, distance="dot"):
            super().__init__()
            self.distance = Distance(distance)

        def forward(self, session_embs, item_embs, candidate_item_ids=None):  # any fixed function: inherited or not
            logits = session_embs @ item_embs.T
            return logits if candidate_item_ids is None else torch.gather(logits, -1, candidate_item_ids)

    mods = {name: types.ModuleType(name) for name in (
        "rectools", "rectools.models", "rectools.models.base", "rectools.models.vector", "rectools.models.ease",
        "rectools.models.nn", "rectools.models.nn.transformers", "rectools.models.nn.transformers.similarity")}
    mods["rectools.models.base"].ModelBase = ModelBase
    mods["rectools.models.vector"].__dict__.update(VectorModel=VectorModel, ImplicitRanker=ImplicitRanker, Distance=Distance)
    mods["rectools.models.ease"].__dict__.update(ImplicitRanker=ImplicitRanker, Distance=Distance)
    mods["rectools.models.nn.transformers.similarity"].DistanceSimilarityModule = DistanceSimilarityModule
    for name, mod in mods.items():
        parent, _, child = name.rpartition(".")
        if parent:
            setattr(mods[parent], child, mod)
        monkeypatch.setitem(sys.modules, name, mod)
    return types.SimpleNamespace(**mods)
