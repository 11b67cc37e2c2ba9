"""GPU: the UNMODIFIED reference models with the real B200 engine under them (SURVEY 8 rows a9 / a11 / a13 / f3 / f4).

`oracle/_ref` holds the reference package as staged by `__graft_entry__.build()` (git-ignored; it travels to the GPU box
like the built `.so`), `oracle/implicit_stub` stands in for the third-party `implicit` (its top-k = the CPU oracle).  Every
test computes the expectation with the stock reference path (`ImplicitRanker` -> stub top-k on the CPU, `TorchRanker` on the
CPU) and then the same call after `rectools_b200.install()` / with `make_similarity_module()`: the frames must agree
(ids exact; near-ties of the fp32 reference arithmetic may swap neighbours within `tie_tol`).  The similarity-module seam
compares with the stock module's results stored in tests/golden/similarity_module.npz and runs without the package."""
import os

import numpy as np
import pytest

from oracle import stage_reference
from tests.helpers import GOLDEN, assert_same_ranking, fake_rectools

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(not stage_reference.available(), reason="reference package not staged (oracle/_ref)")


@pytest.fixture(scope="module")
def ref():
    added = stage_reference.add_to_path()
    import rectools  # noqa: F401

    yield
    import rectools_b200

    rectools_b200.uninstall()
    stage_reference.remove_from_path(added)


def _same_reco(ref_df, got_df, target_col="user_id", tie_tol=3e-6):
    assert list(ref_df.columns) == list(got_df.columns)
    assert [str(t) for t in ref_df.dtypes] == [str(t) for t in got_df.dtypes]
    np.testing.assert_array_equal(ref_df[target_col].to_numpy(), got_df[target_col].to_numpy())
    if "rank" in ref_df:
        np.testing.assert_array_equal(ref_df["rank"].to_numpy(), got_df["rank"].to_numpy())
    assert_same_ranking(got_df["item_id"].to_numpy(), got_df["score"].to_numpy(), ref_df["item_id"].to_numpy(), ref_df["score"].to_numpy(),
                        rtol=3e-5, atol=3e-6, tie_tol=tie_tol)


def _factors(n, d, seed):
    return (np.random.default_rng(seed).standard_normal((n, d), dtype=np.float32) / np.sqrt(d)).astype(np.float32)


@needs_reference
@pytest.mark.parametrize("fast_recommend", [True, False])
def test_puresvd_and_injected_als_recommend_through_the_engine(ref, fast_recommend):
    """`install()` + `PureSVDModel.recommend()` and `ImplicitALSWrapperModel.recommend()` (pre-fitted factors injected as in
    tests/models/test_implicit_als.py:193-197) vs the stock reference path; u2i with / without filter and whitelist, i2i."""
    from rectools.models import PureSVDModel

    import rectools_b200
    from tests.ref_models import injected_als, synthetic_dataset

    n_users, n_items = 6000, 3000
    dataset = synthetic_dataset(n_users, n_items, 30, seed=1)
    models = {
        "puresvd": PureSVDModel(factors=32, random_state=0).fit(dataset),
        "als": injected_als(_factors(n_users, 64, 1), _factors(n_items, 64, 2)),
    }
    users = np.random.default_rng(3).permutation(dataset.user_id_map.external_ids)[:5000]
    wl = dataset.item_id_map.external_ids[::7]
    targets = dataset.item_id_map.external_ids[:400]
    calls = {
        "u2i": lambda m: m.recommend(users, dataset, k=10, filter_viewed=True),
        "u2i_nofilter": lambda m: m.recommend(users[:1000], dataset, k=5, filter_viewed=False, add_rank_col=False),
        "u2i_whitelist": lambda m: m.recommend(users, dataset, k=10, filter_viewed=True, items_to_recommend=wl),
        "i2i": lambda m: m.recommend_to_items(targets, dataset, k=6),
    }
    expected = {(name, call): fn(model) for name, model in models.items() for call, fn in calls.items()}
    rectools_b200.install(device=0, fast_recommend=fast_recommend)
    try:
        import rectools.models.vector as vector

        assert vector.ImplicitRanker is rectools_b200.B200ImplicitRanker
        for (name, call), exp in expected.items():
            got = calls[call](models[name])
            _same_reco(exp, got, "target_item_id" if call == "i2i" else "user_id")
        from rectools_b200 import integration

        assert len(integration._ENGINE_CACHE) >= 1  # pylint: disable=protected-access
        stats = next(iter(integration._ENGINE_CACHE.values())).last_stats  # pylint: disable=protected-access
        assert stats["path"] in (0, 1)
    finally:
        rectools_b200.uninstall()


@needs_reference
def test_in_place_refit_reaches_the_device(ref):
    """VERDICT r1 weak #3: factors changed IN PLACE between two `recommend()` calls must give fresh results."""
    import rectools_b200
    from tests.ref_models import injected_als, synthetic_dataset

    dataset = synthetic_dataset(3000, 2000, 10, seed=2)
    u, i = _factors(3000, 32, 5), _factors(2000, 32, 6)
    model = injected_als(u, i)
    users = dataset.user_id_map.external_ids
    rectools_b200.install(device=0)
    try:
        first = model.recommend(users, dataset, k=5, filter_viewed=False)
        # "refit": the implicit model's arrays are rewritten in place (same objects, same addresses)
        model.model.item_factors[1234] = 10.0 * model.model.user_factors[:50].mean(axis=0)
        model.model.user_factors[17] *= -1.0
        second = model.recommend(users, dataset, k=5, filter_viewed=False)
    finally:
        rectools_b200.uninstall()
    expected = model.recommend(users, dataset, k=5, filter_viewed=False)  # stock path on the changed factors
    _same_reco(expected, second)
    assert not first["item_id"].equals(second["item_id"])


@needs_reference
def test_ease_sparse_subjects_through_install(ref):
    """SURVEY 8 f-4: `EASEModel._recommend_u2i` hands the user x item CSR as SUBJECT factors (ease.py:134-161); the engine
    scores it sparse (SpMM + streaming top-k) instead of densifying users x items."""
    from rectools.models import EASEModel

    import rectools_b200
    from tests.ref_models import synthetic_dataset

    dataset = synthetic_dataset(5000, 1200, 25, seed=4)
    model = EASEModel(regularization=200.0).fit(dataset)
    users = dataset.user_id_map.external_ids[::2]
    exp = model.recommend(users, dataset, k=10, filter_viewed=True)
    exp_wl = model.recommend(users[:500], dataset, k=40, filter_viewed=True, items_to_recommend=dataset.item_id_map.external_ids[::3])
    rectools_b200.install(device=0)
    try:
        import rectools.models.ease as ease

        assert ease.ImplicitRanker is rectools_b200.B200ImplicitRanker
        got = model.recommend(users, dataset, k=10, filter_viewed=True)
        got_wl = model.recommend(users[:500], dataset, k=40, filter_viewed=True, items_to_recommend=dataset.item_id_map.external_ids[::3])
    finally:
        rectools_b200.uninstall()
    _same_reco(exp, got, tie_tol=1e-5)
    _same_reco(exp_wl, got_wl, tie_tol=1e-5)


@pytest.mark.parametrize("distance", ["dot", "cosine"])
def test_transformer_similarity_module_seam(monkeypatch, distance):
    """SURVEY 8 a13 / f-3: `DistanceSimilarityModule._recommend_u2i` (similarity.py:117-140) with `B200TorchRanker` under it
    (`make_similarity_module()`), called the way `TransformerLightningModuleBase._recommend_u2i` does (lightning.py:402-426):
    device-resident `item_embs` with the PAD row first, whitelist = the non-PAD items (nn/transformers/base.py:543-544),
    filter CSR over all token columns.  DOT = SASRec / BERT4Rec, COSINE = HSTU's default (hstu.py:696-703)."""
    import torch
    from scipy import sparse

    from rectools_b200.integration import make_similarity_module

    DistanceSimilarityModule = fake_rectools(monkeypatch).rectools.models.nn.transformers.similarity.DistanceSimilarityModule
    gold = np.load(os.path.join(GOLDEN, "similarity_module.npz"))

    n_users, n_tokens, d, k = 3000, 20_001, 64, 10  # token 0 = PAD
    rng = np.random.default_rng(7)  # (numpy: the same values on every host, unlike torch's vectorised CPU sampler)
    user_embs = torch.from_numpy(rng.standard_normal((n_users, d), dtype=np.float32) / np.float32(d**0.5))
    item_embs = torch.from_numpy(rng.standard_normal((n_tokens, d), dtype=np.float32) / np.float32(d**0.5))
    item_embs[0] = 0.0
    user_ids = np.random.default_rng(0).permutation(n_users)[:2000]
    rng = np.random.default_rng(1)
    cols = rng.integers(1, n_tokens, size=(len(user_ids), 30))
    rows = np.repeat(np.arange(len(user_ids)), 30)
    ui = sparse.csr_matrix((np.ones(cols.size, np.float32), (rows, cols.reshape(-1))), shape=(len(user_ids), n_tokens))
    ui.sum_duplicates()
    ui.data[:] = 1.0
    whitelist = np.arange(1, n_tokens)

    e_users, e_ids, e_scores = (gold[f"gpu|{distance}|f32|{name}"] for name in ("users", "ids", "scores"))
    ours = make_similarity_module()(distance=distance)
    assert isinstance(ours, DistanceSimilarityModule)
    dev = torch.device("cuda:0")
    o_users, o_ids, o_scores = ours._recommend_u2i(user_embs, item_embs.to(dev), user_ids, k, whitelist, ui)  # pylint: disable=protected-access
    np.testing.assert_array_equal(o_users, e_users)
    assert_same_ranking(o_ids, o_scores, e_ids, e_scores, rtol=3e-5, atol=3e-6, tie_tol=3e-6)
    assert not (np.asarray(o_ids) == 0).any()  # the PAD token is never recommended
    # bf16 item embeddings stay 16-bit all the way to the engine (exact widening there): same ids as the fp32 path on the
    # bf16-rounded values
    emb16 = item_embs.to(torch.bfloat16)
    e2 = tuple(gold[f"gpu|{distance}|bf16|{name}"] for name in ("users", "ids", "scores"))  # the stock module on emb16.float()
    o2 = ours._recommend_u2i(user_embs, emb16.to(dev), user_ids, k, whitelist, ui)  # pylint: disable=protected-access
    assert_same_ranking(o2[1], o2[2], e2[1], e2[2], rtol=3e-5, atol=3e-6, tie_tol=3e-6)
