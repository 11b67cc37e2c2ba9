"""CPU: the vectorised `recommend()` (SURVEY section 8f rank 1) returns the same table as the unmodified reference
`ModelBase.recommend` (rectools/models/base.py:385-519).  The reference tables, the fitted `PureSVDModel(factors=8)` vectors
and the interactions they were computed from are stored in tests/golden/recommend_puresvd.npz (oracle/make_golden.py); the
model and dataset are duck-typed stand-ins over those arrays and the B200 ranker is replaced by the oracle-backed stand-in
(`tests/helpers.OracleRanker`), so only the host logic is compared."""
import os
import sys
import warnings

import numpy as np
import pandas as pd
import pytest
from scipy import sparse

from tests.helpers import GOLDEN, FakeIdMap, FakeVectorModel, OracleRanker, fake_rectools


class GoldenDataset:
    """`rectools.dataset.Dataset` surface used by `rectools_b200.recommend`, over an interactions DataFrame of internal ids."""

    def __init__(self, user_ext, item_ext, inter_user, inter_item):
        self.user_id_map, self.item_id_map = FakeIdMap(user_ext), FakeIdMap(item_ext)
        self.interactions = type("Interactions", (), {})()
        self.interactions.df = pd.DataFrame({"user_id": inter_user, "item_id": inter_item, "weight": 1.0})

    @property
    def n_hot_users(self):  # dataset.py:176-184
        return int(self.interactions.df["user_id"].max()) + 1

    def get_user_item_matrix(self, include_weights=True):
        df = self.interactions.df
        data = df["weight"].to_numpy(np.float32) if include_weights else np.ones(len(df), np.float32)
        shape = (self.user_id_map.size, self.item_id_map.size)
        return sparse.csr_matrix((data, (df["user_id"].to_numpy(), df["item_id"].to_numpy())), shape=shape)


class GoldenModel(FakeVectorModel):
    """PureSVD's distances (pure_svd.py:88-89) and `ModelBase._check_targets_are_valid` (base.py:703-732): unsupported
    targets raise, warn or are dropped."""

    def __init__(self, user_vectors, item_vectors):
        super().__init__("dot", user_vectors, item_vectors, i2i_dist="cosine")

    @staticmethod
    def _check_targets_are_valid(hot, warm, cold, entity, on_unsupported_targets):
        for kind, targets in (("warm", warm), ("cold", cold)):
            if np.size(targets) == 0:
                continue
            msg = f"some of the given {entity}s are {kind}"
            if on_unsupported_targets == "warn":
                warnings.warn(msg)
            elif on_unsupported_targets == "raise":
                raise ValueError(msg)
        return hot, np.asarray([], dtype=np.int64), np.asarray([])


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(GOLDEN, "recommend_puresvd.npz"))


def _build(g, prefix=""):
    dataset = GoldenDataset(g[prefix + "user_ext"], g[prefix + "item_ext"], g[prefix + "inter_user"], g[prefix + "inter_item"])
    return GoldenModel(g[prefix + "user_vectors"], g[prefix + "item_vectors"]), dataset


@pytest.fixture()
def fitted(golden):
    model, dataset = _build(golden)
    # the interactions table in external ids (what the reference's fixture was built from)
    df = pd.DataFrame({"user_id": dataset.user_id_map.external_ids[golden["inter_user"]],
                       "item_id": dataset.item_id_map.external_ids[golden["inter_item"]]})
    return model, dataset, df


def _ref(g, name):
    return pd.DataFrame({str(col): g[f"{name}|{col}"] for col in g[name + "|columns"]})


def _same(ref, got):
    pd.testing.assert_frame_equal(ref.reset_index(drop=True), got.reset_index(drop=True), check_exact=False, rtol=2e-5, atol=1e-6)


def _delegate_to(ref, calls):
    def reference_recommend(*args, **kwargs):
        calls.append((args, kwargs))
        return ref

    return reference_recommend


@pytest.mark.parametrize("filter_viewed", [True, False])
@pytest.mark.parametrize("add_rank_col", [True, False])
def test_all_users_match_reference(golden, fitted, filter_viewed, add_rank_col):
    from rectools_b200.recommend import recommend

    model, dataset, _ = fitted
    users = dataset.user_id_map.external_ids
    ref = _ref(golden, f"all_f{int(filter_viewed)}_r{int(add_rank_col)}")
    got = recommend(model, users, dataset, 7, filter_viewed, add_rank_col=add_rank_col, ranker_factory=OracleRanker)
    assert list(ref.columns) == list(got.columns) and [str(t) for t in ref.dtypes] == [str(t) for t in got.dtypes]
    _same(ref, got)


def test_user_subset_whitelist_and_ragged_rows(golden, fitted):
    from rectools_b200.recommend import recommend

    model, dataset, df = fitted
    users = np.random.default_rng(1).permutation(dataset.user_id_map.external_ids)[:57]
    np.testing.assert_array_equal(users, golden["subset|users"])
    # a whitelist smaller than k plus the viewed filter: users get fewer than k rows (rank_implicit.py:107-118)
    items = golden["subset|items"]
    assert set(items.tolist()) == set(df["item_id"].value_counts().index[:4].tolist())
    ref = _ref(golden, "subset")
    got = recommend(model, users, dataset, 6, True, items_to_recommend=items, ranker_factory=OracleRanker)
    assert len(ref) < 57 * 4 + 1 and ref.groupby("user_id").size().min() < 4
    _same(ref, got)
    # second call: the viewed-items CSR comes from the cache
    from rectools_b200 import recommend as rmod

    assert id(dataset.interactions.df) in sys.modules[rmod.__module__]._CSR_CACHE  # pylint: disable=protected-access
    _same(ref, recommend(model, users, dataset, 6, True, items_to_recommend=items, ranker_factory=OracleRanker))


def test_cold_targets_are_delegated(golden, fitted):
    """Cold targets: refused, or dropped (on_unsupported_targets="ignore") and the rest ranked as the reference does."""
    from rectools_b200.recommend import recommend

    model, dataset, _ = fitted
    users = np.concatenate([dataset.user_id_map.external_ids[:5], [10**9]])
    with pytest.raises(ValueError):
        recommend(model, users, dataset, 3, True, ranker_factory=OracleRanker)
    got = recommend(model, users, dataset, 3, True, on_unsupported_targets="ignore", ranker_factory=OracleRanker)
    _same(_ref(golden, "cold"), got)


def test_install_patches_vector_model_recommend(monkeypatch):
    rt = fake_rectools(monkeypatch)
    vector, ModelBase = rt.rectools.models.vector, rt.rectools.models.base.ModelBase

    import rectools_b200

    rectools_b200.install(fast_recommend=True)
    try:
        assert "recommend" in vector.VectorModel.__dict__ and "recommend_to_items" in vector.VectorModel.__dict__
    finally:
        rectools_b200.uninstall()
    assert "recommend" not in vector.VectorModel.__dict__ and vector.VectorModel.recommend is ModelBase.recommend
    assert vector.VectorModel.recommend_to_items is ModelBase.recommend_to_items


@pytest.mark.parametrize("filter_itself", [True, False])
@pytest.mark.parametrize("with_whitelist", [False, True])
def test_recommend_to_items_matches_reference(golden, fitted, filter_itself, with_whitelist):
    """SURVEY 8f rank 2: i2i = the same ranker with item vectors as subjects, k + 1 results, self-filter on the padded arrays."""
    from rectools_b200.recommend import recommend_to_items

    model, dataset, df = fitted
    targets = np.random.default_rng(2).permutation(dataset.item_id_map.external_ids)[:40]
    np.testing.assert_array_equal(targets, golden["i2i|targets"])
    wl = None
    if with_whitelist:  # small enough that some targets get fewer than k rows; contains some of the targets themselves
        wl = golden["i2i|whitelist"]
        assert set(wl[3:].tolist()) == set(df["item_id"].value_counts().index[:4].tolist())
    ref = _ref(golden, f"i2i_f{int(filter_itself)}_w{int(with_whitelist)}")
    got = recommend_to_items(model, targets, dataset, 5, filter_itself, items_to_recommend=wl, ranker_factory=OracleRanker)
    assert list(ref.columns) == list(got.columns) and [str(t) for t in ref.dtypes] == [str(t) for t in got.dtypes]
    _same(ref, got)


def test_recommend_to_items_repeated_targets_are_delegated(golden, fitted):
    from rectools_b200.recommend import recommend_to_items

    model, dataset, _ = fitted
    t = dataset.item_id_map.external_ids[:3]
    targets = np.concatenate([t, t[:1]])
    ref, calls = _ref(golden, "i2i_repeated"), []
    _same(ref, recommend_to_items(model, targets, dataset, 4, ranker_factory=OracleRanker, reference_recommend=_delegate_to(ref, calls)))
    assert len(calls) == 1 and calls[0][0][0] is targets and calls[0][0][2] == 4


def test_repeated_users_are_delegated(golden, fitted):
    """ADVICE r1: with repeated target users the reference's rank column runs across the repeats (`groupby(user).cumcount()`,
    base.py:778-791): the vectorised path hands such calls to the reference method."""
    from rectools_b200.recommend import recommend

    model, dataset, _ = fitted
    u = dataset.user_id_map.external_ids[:3]
    users = np.array([u[0], u[1], u[0]])
    ref, calls = _ref(golden, "users_repeated"), []
    got = recommend(model, users, dataset, 3, True, ranker_factory=OracleRanker, reference_recommend=_delegate_to(ref, calls))
    assert len(calls) == 1 and calls[0][0][0] is users and calls[0][0][2:4] == (3, True)
    _same(ref, got)
    assert got["rank"].max() == 6


def test_viewed_csr_cache_notices_in_place_edits(fitted):
    """VERDICT r1 #9: the cached viewed-items CSR is stamped with a digest of the (user, item) columns."""
    from rectools_b200.recommend import viewed_csr

    _, dataset, _ = fitted
    a = viewed_csr(dataset)
    assert viewed_csr(dataset) is a
    df = dataset.interactions.df
    old = df.loc[df.index[0], "item_id"]
    new = (old + 1) % dataset.item_id_map.size
    try:
        df.loc[df.index[0], "item_id"] = new
        b = viewed_csr(dataset)
        assert b is not a and (b != a).nnz > 0
    finally:
        df.loc[df.index[0], "item_id"] = old
    assert (viewed_csr(dataset) != a).nnz == 0


def test_warm_users_are_still_told_apart_with_the_cached_hot_count(golden):
    """`n_hot_users` is answered from the stamped CSR cache entry (not a scan of the table per call): a user known only from
    the feature table is warm exactly as for the reference (base.py:676-700) -- refused, or dropped with a warning."""
    from rectools_b200.recommend import _viewed_entry, recommend

    model, dataset = _build(golden, "warm|")
    users = np.sort(golden["warm|user_ext"][: int(golden["warm|n_hot_users"][0])])  # np.unique of the interactions' users
    warm_id = int(golden["warm|user_ext"][-1])
    assert dataset.user_id_map.size == len(users) + 1 and warm_id not in set(users.tolist())
    assert _viewed_entry(dataset)[1] == dataset.n_hot_users == len(users) == golden["warm|n_hot_users"][0]
    _same(_ref(golden, "warm_hot"), recommend(model, users[:50], dataset, 5, True, ranker_factory=OracleRanker))
    targets = np.append(users[:5], warm_id)
    with pytest.raises(ValueError, match="warm"):
        recommend(model, targets, dataset, 5, True, ranker_factory=OracleRanker)
    with pytest.warns(UserWarning):
        got = recommend(model, targets, dataset, 5, True, on_unsupported_targets="warn", ranker_factory=OracleRanker)
    _same(_ref(golden, "warm_warn"), got)
    assert warm_id not in set(got["user_id"])


def test_threaded_table_columns_match_reference(golden, fitted, monkeypatch):
    """Above 2^20 output rows the id gather / repeat / rank columns are written by row blocks on a thread pool: force that
    path at test size and compare with the reference table (u2i with unfilled slots, u2i full, i2i)."""
    import importlib

    rec = importlib.import_module("rectools_b200.recommend")  # (the package attribute of that name is the function)
    monkeypatch.setattr(rec, "_PAR_MIN", 1)
    model, dataset, _ = fitted
    users = dataset.user_id_map.external_ids
    for k, add_rank_col in ((7, True), (7, False), (dataset.item_id_map.size, True)):  # the last: ragged rows (-1 slots)
        ref = _ref(golden, f"threaded_k{k}_r{int(add_rank_col)}")
        _same(ref, rec.recommend(model, users, dataset, k, True, add_rank_col=add_rank_col, ranker_factory=OracleRanker))
    items = dataset.item_id_map.external_ids[:40]
    _same(_ref(golden, "threaded_i2i"), rec.recommend_to_items(model, items, dataset, 6, ranker_factory=OracleRanker))
    table = np.arange(10, dtype=np.int64) * 3
    ids = np.array([[1, -1], [9, 0]], dtype=np.int32)
    assert rec.external_ids_of(table, ids, np.int64).tolist() == [[3, 0], [27, 0]]
    assert rec._repeat_rows(np.array([5, 6, 7]), 2).tolist() == [5, 5, 6, 6, 7, 7]
    assert rec._tile_rows(np.array([1, 2]), 3).tolist() == [1, 2, 1, 2, 1, 2]
