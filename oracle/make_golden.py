"""Generate tests/golden/*.npz by running the UNMODIFIED reference here (test infrastructure only).

Needs a checkout of the reference (RecTools 0.17.0) on the path, next to the `implicit` stub:

    PYTHONPATH=<rectools checkout>:oracle/implicit_stub python oracle/make_golden.py

What is recorded (inputs + the reference's outputs, fp32 / int64):
  * torch_*    -- `rectools.models.rank.TorchRanker` (rank_torch.py:77-177): an independent in-repo implementation
                  of the Ranker contract (torch CPU matmul + torch.topk), DOT and COSINE, with/without
                  `filter_pairs_csr`, with/without `sorted_object_whitelist`, k in {1, 10, None}.
  * implicit_* -- `rectools.models.rank.ImplicitRanker` (rank_implicit.py:187-280) driven through the `implicit` stub
                  whose `topk` is oracle/topk_oracle.py::implicit_topk (pins prologue/epilogue semantics, incl. the
                  < k rows case and EUCLIDEAN).
  * puresvd_c1 -- BASELINE config 1: `PureSVDModel(factors=32)` fit on synthetic 6 040 x 3 706 interactions
                  (MovieLens-1M shape), `recommend(k=10, filter_viewed=True)`; stores the fitted factor matrices
                  (user rows of the ranked users only, the others zero: the file stays small), the filter CSR
                  the model builds (vector.py:58-60) and the returned (user, item, score) table.
  * recommend_puresvd -- `PureSVDModel(factors=8)` on 300 x 120 synthetic interactions: the model's vectors, the
                  interactions and the tables of every `recommend()` / `recommend_to_items()` call of
                  tests/test_recommend_cpu.py (keys `<call>|<column>`).
  * similarity_module -- the stock `DistanceSimilarityModule._recommend_u2i` (scorer: `TorchRanker`) on the inputs of
                  tests/test_transformer_seam_cpu.py and of tests/test_gpu_models.py::test_transformer_similarity_module_seam.
Seeds are fixed; continuous random factors => no intra-user score ties.
"""

from __future__ import annotations

import os
import sys

import numpy as np
import pandas as pd
from scipy import sparse

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "..", "tests", "golden")


def _random_case(seed: int, n_subj: int, n_obj: int, d: int, nnz_per_row: int):
    rng = np.random.default_rng(seed)
    s = (rng.standard_normal((n_subj, d)) / np.sqrt(d)).astype(np.float32)
    o = (rng.standard_normal((n_obj, d)) / np.sqrt(d)).astype(np.float32)
    subject_ids = rng.permutation(n_subj)[: max(1, n_subj * 3 // 4)].astype(np.int64)
    rows, cols = [], []
    for r in range(len(subject_ids)):
        m = int(rng.integers(0, nnz_per_row + 1))
        c = rng.choice(n_obj, size=min(m, n_obj), replace=False)
        rows.extend([r] * len(c))
        cols.extend(c.tolist())
    csr = sparse.csr_matrix(
        (np.ones(len(rows), dtype=np.float32), (rows, cols)), shape=(len(subject_ids), n_obj), dtype=np.float32
    )
    csr.sort_indices()
    whitelist = np.sort(rng.choice(n_obj, size=max(2, n_obj // 3), replace=False)).astype(np.int64)
    return s, o, subject_ids, csr, whitelist


def _save(name: str, **arrays) -> None:
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"wrote {path}: {os.path.getsize(path) / 1024:.1f} KiB")


def ranker_cases() -> None:
    """One `rank_inputs_<c>.npz` per seeded case + one `rank_outputs_<c>.npz` holding every (impl, distance, k,
    filter, whitelist) combination under keys `<impl>|<distance>|k<k>|f<0/1>|w<0/1>|{subjects,ids,scores}`."""
    from rectools.models.rank import Distance, ImplicitRanker, TorchRanker

    for case, (n_subj, n_obj, d, nnz) in enumerate([(48, 300, 16, 12), (33, 1000, 40, 60), (17, 64, 7, 70)]):
        s, o, subject_ids, csr, whitelist = _random_case(100 + case, n_subj, n_obj, d, nnz)
        _save(
            f"rank_inputs_{case}",
            subjects=s,
            objects=o,
            subject_ids=subject_ids,
            csr_indptr=csr.indptr.astype(np.int64),
            csr_indices=csr.indices.astype(np.int32),
            csr_shape=np.asarray(csr.shape, dtype=np.int64),
            whitelist=whitelist,
        )
        outputs = {}
        for dist in (Distance.DOT, Distance.COSINE, Distance.EUCLIDEAN):
            rankers = (
                ("torch", TorchRanker(distance=dist, device="cpu", subjects_factors=s, objects_factors=o)),
                ("implicit", ImplicitRanker(dist, s, o)),
            )
            for k in (1, 10, 100) if case == 1 else (1, 10, None):
                for use_filter in (False, True):
                    for use_wl in (False, True):
                        for impl, ranker in rankers:
                            u, i, sc = ranker.rank(
                                subject_ids=subject_ids,
                                k=k,
                                filter_pairs_csr=csr if use_filter else None,
                                sorted_object_whitelist=whitelist if use_wl else None,
                            )
                            key = f"{impl}|{dist.value}|k{-1 if k is None else k}|f{int(use_filter)}|w{int(use_wl)}"
                            outputs[key + "|subjects"] = np.asarray(u, dtype=np.int64)
                            outputs[key + "|ids"] = np.asarray(i, dtype=np.int32)
                            outputs[key + "|scores"] = np.asarray(sc, dtype=np.float32)
        _save(f"rank_outputs_{case}", **outputs)


def puresvd_c1() -> None:
    from rectools import Columns
    from rectools.dataset import Dataset
    from rectools.models import PureSVDModel

    rng = np.random.default_rng(0)
    n_users, n_items, draws = 6040, 3706, 1_000_000
    users = rng.integers(0, n_users, size=draws)
    items = (rng.zipf(1.3, size=draws) - 1) % n_items
    df = pd.DataFrame({Columns.User: users, Columns.Item: items}).drop_duplicates()
    df[Columns.Weight] = 1.0
    df[Columns.Datetime] = pd.Timestamp("2024-01-01")
    dataset = Dataset.construct(df)
    model = PureSVDModel(factors=32, random_state=0).fit(dataset)

    ext_users = np.sort(dataset.user_id_map.external_ids)[:768]
    reco = model.recommend(users=ext_users, dataset=dataset, k=10, filter_viewed=True)
    reco_nf = model.recommend(users=ext_users, dataset=dataset, k=10, filter_viewed=False)

    user_vectors, item_vectors = model._get_u2i_vectors(dataset)  # pylint: disable=protected-access
    int_users = dataset.user_id_map.convert_to_internal(ext_users)
    ui = dataset.get_user_item_matrix(include_weights=False)[int_users]
    ui.sort_indices()

    def table(r):
        return dict(
            users=dataset.user_id_map.convert_to_internal(r[Columns.User].to_numpy()).astype(np.int64),
            items=dataset.item_id_map.convert_to_internal(r[Columns.Item].to_numpy()).astype(np.int64),
            scores=r[Columns.Score].to_numpy().astype(np.float32),
        )

    t, tn = table(reco), table(reco_nf)
    _save(
        "puresvd_c1",
        user_factors=np.where(np.isin(np.arange(len(user_vectors)), int_users)[:, None], user_vectors, 0).astype(np.float32),
        item_factors=item_vectors.astype(np.float32),
        subject_ids=int_users.astype(np.int64),
        csr_indptr=ui.indptr.astype(np.int64),
        csr_indices=ui.indices.astype(np.int32),
        csr_shape=np.asarray(ui.shape, dtype=np.int64),
        out_subjects=t["users"],
        out_ids=t["items"],
        out_scores=t["scores"],
        out_nf_subjects=tn["users"],
        out_nf_ids=tn["items"],
        out_nf_scores=tn["scores"],
        n_interactions=np.asarray([len(df)], dtype=np.int64),
    )


def _tables(out: dict, name: str, df: pd.DataFrame) -> None:
    out[name + "|columns"] = np.asarray(list(df.columns))
    for col in df.columns:
        out[name + "|" + col] = df[col].to_numpy()


def recommend_cases() -> None:
    """The fixture and the reference calls of tests/test_recommend_cpu.py."""
    import warnings

    from rectools import Columns
    from rectools.dataset import Dataset
    from rectools.models import PureSVDModel

    rng = np.random.default_rng(0)
    n_users, n_items, n_inter = 300, 120, 6000
    df = pd.DataFrame(
        {
            Columns.User: rng.integers(0, n_users, n_inter) * 7 + 1000,  # external ids != internal ids
            Columns.Item: rng.integers(0, n_items, n_inter) * 3 + 5,
            Columns.Weight: 1.0,
            Columns.Datetime: pd.Timestamp("2024-01-01"),
        }
    ).drop_duplicates([Columns.User, Columns.Item])
    dataset = Dataset.construct(df)
    model = PureSVDModel(factors=8, random_state=0).fit(dataset)
    out: dict = {}

    def dataset_arrays(prefix, ds, m):
        inter = ds.interactions.df
        out[prefix + "user_ext"] = ds.user_id_map.external_ids
        out[prefix + "item_ext"] = ds.item_id_map.external_ids
        out[prefix + "inter_user"] = inter[Columns.User].to_numpy().astype(np.int64)  # internal ids
        out[prefix + "inter_item"] = inter[Columns.Item].to_numpy().astype(np.int64)
        out[prefix + "user_vectors"], out[prefix + "item_vectors"] = m._get_u2i_vectors(ds)  # pylint: disable=protected-access

    dataset_arrays("", dataset, model)
    users = dataset.user_id_map.external_ids
    for fv in (True, False):
        for rc in (True, False):
            _tables(out, f"all_f{int(fv)}_r{int(rc)}", model.recommend(users, dataset, k=7, filter_viewed=fv, add_rank_col=rc))
    sub = np.random.default_rng(1).permutation(users)[:57]
    top4 = df[Columns.Item].value_counts().index[:4].to_numpy()
    out["subset|users"], out["subset|items"] = sub, top4
    _tables(out, "subset", model.recommend(sub, dataset, k=6, filter_viewed=True, items_to_recommend=top4))
    cold = np.concatenate([users[:5], [10**9]])
    _tables(out, "cold", model.recommend(cold, dataset, k=3, filter_viewed=True, on_unsupported_targets="ignore"))
    targets = np.random.default_rng(2).permutation(dataset.item_id_map.external_ids)[:40]
    wl = np.concatenate([targets[:3], top4])
    out["i2i|targets"], out["i2i|whitelist"] = targets, wl
    for fi in (True, False):
        for use_wl in (False, True):
            _tables(out, f"i2i_f{int(fi)}_w{int(use_wl)}",
                    model.recommend_to_items(targets, dataset, k=5, filter_itself=fi, items_to_recommend=wl if use_wl else None))
    t = dataset.item_id_map.external_ids[:3]
    _tables(out, "i2i_repeated", model.recommend_to_items(np.concatenate([t, t[:1]]), dataset, k=4))
    u = users[:3]
    _tables(out, "users_repeated", model.recommend(np.array([u[0], u[1], u[0]]), dataset, k=3, filter_viewed=True))
    for k, rc in ((7, True), (7, False), (dataset.item_id_map.size, True)):
        _tables(out, f"threaded_k{k}_r{int(rc)}", model.recommend(users, dataset, k=k, filter_viewed=True, add_rank_col=rc))
    _tables(out, "threaded_i2i", model.recommend_to_items(dataset.item_id_map.external_ids[:40], dataset, k=6))

    # a user known only from the feature table: warm for the reference (base.py:676-700)
    hot = np.unique(df[Columns.User].values)
    warm_id = int(hot.max()) + 7
    feats = pd.DataFrame({"id": np.append(hot, warm_id), "feature": "f", "value": 1.0})
    wds = Dataset.construct(df, user_features_df=feats)
    wmodel = PureSVDModel(factors=8, random_state=0).fit(wds)
    dataset_arrays("warm|", wds, wmodel)
    out["warm|n_hot_users"] = np.asarray([wds.n_hot_users], dtype=np.int64)
    _tables(out, "warm_hot", wmodel.recommend(hot[:50], wds, k=5, filter_viewed=True))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _tables(out, "warm_warn", wmodel.recommend(np.append(hot[:5], warm_id), wds, k=5, filter_viewed=True, on_unsupported_targets="warn"))
    _save("recommend_puresvd", **out)


def similarity_module_cases() -> None:
    """`DistanceSimilarityModule(distance)._recommend_u2i` of the reference on the inputs of tests/test_transformer_seam_cpu.py
    (they are rebuilt there from the same seeds)."""
    import torch
    from rectools.models.nn.transformers.similarity import DistanceSimilarityModule
    from scipy import sparse as sp

    out = {}
    for distance, n_extra in (("dot", 1), ("cosine", 1), ("dot", 2)):
        n_users, n_tokens, d, k = 150, 400 + n_extra, 16, 7
        rng = np.random.default_rng(3)  # (numpy: the same values on every host, unlike torch's vectorised CPU sampler)
        user_embs = torch.from_numpy(rng.standard_normal((n_users, d), dtype=np.float32))
        item_embs = torch.from_numpy(rng.standard_normal((n_tokens, d), dtype=np.float32))
        item_embs[:n_extra] = 0.0
        user_ids = np.random.default_rng(0).permutation(n_users)[:90]
        dense = (np.random.default_rng(1).random((len(user_ids), n_tokens)) < 0.05).astype(np.float32)
        dense[5, n_extra:] = 1.0
        dense[6, n_extra : n_tokens - 3] = 1.0
        whitelist = np.arange(n_extra, n_tokens)
        stock = DistanceSimilarityModule(distance=distance)
        users, ids, scores = stock._recommend_u2i(user_embs, item_embs, user_ids, k, whitelist, sp.csr_matrix(dense))  # pylint: disable=protected-access
        key = f"{distance}|{n_extra}"
        out[key + "|users"] = np.asarray(users, dtype=np.int64)
        out[key + "|ids"] = np.asarray(ids, dtype=np.int64)
        out[key + "|scores"] = np.asarray(scores, dtype=np.float32)
    for distance in ("dot", "cosine"):  # the GPU seam test: PAD token 0, fp32 and bf16-rounded item embeddings
        n_users, n_tokens, d, k = 3000, 20_001, 64, 10
        rng = np.random.default_rng(7)  # (numpy: the same values on every host, unlike torch's vectorised CPU sampler)
        user_embs = torch.from_numpy(rng.standard_normal((n_users, d), dtype=np.float32) / np.float32(d**0.5))
        item_embs = torch.from_numpy(rng.standard_normal((n_tokens, d), dtype=np.float32) / np.float32(d**0.5))
        item_embs[0] = 0.0
        user_ids = np.random.default_rng(0).permutation(n_users)[:2000]
        rng = np.random.default_rng(1)
        cols = rng.integers(1, n_tokens, size=(len(user_ids), 30))
        rows = np.repeat(np.arange(len(user_ids)), 30)
        ui = sp.csr_matrix((np.ones(cols.size, np.float32), (rows, cols.reshape(-1))), shape=(len(user_ids), n_tokens))
        ui.sum_duplicates()
        ui.data[:] = 1.0
        stock = DistanceSimilarityModule(distance=distance)
        for dtype, emb in (("f32", item_embs), ("bf16", item_embs.to(torch.bfloat16).float())):
            users, ids, scores = stock._recommend_u2i(user_embs, emb, user_ids, k, np.arange(1, n_tokens), ui)  # pylint: disable=protected-access
            key = f"gpu|{distance}|{dtype}"
            out[key + "|users"] = np.asarray(users, dtype=np.int32)
            out[key + "|ids"] = np.asarray(ids, dtype=np.int32)
            out[key + "|scores"] = np.asarray(scores, dtype=np.float32)
    _save("similarity_module", **out)


if __name__ == "__main__":
    try:
        import rectools  # noqa: F401  pylint: disable=unused-import
    except ImportError:
        sys.exit("make_golden.py needs the reference package (RecTools 0.17.0) on PYTHONPATH")
    ranker_cases()
    puresvd_c1()
    recommend_cases()
    similarity_module_cases()
