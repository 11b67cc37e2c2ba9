"""CPU: the transformer seam (SURVEY 8 a13).  `make_similarity_module()` subclasses the reference's
`DistanceSimilarityModule` and swaps the scorer of `_recommend_u2i` (similarity.py:117-140); here an oracle-backed stand-in
with the `TorchRanker` signature is plugged in, and the result is compared with what the stock module returned (its scorer
is the reference's own `TorchRanker`, an independent implementation of the same contract): tests/golden/similarity_module.npz,
made by oracle/make_golden.py from the same seeded inputs.  The base class is the stand-in of `tests.helpers.fake_rectools`.
The GPU twin with the real engine is tests/test_gpu_models.py::test_transformer_similarity_module_seam."""
import os

import numpy as np
import pytest
from scipy import sparse

from tests.helpers import GOLDEN, OracleTorchRanker, assert_same_ranking, fake_rectools


@pytest.mark.parametrize("distance, n_extra", [("dot", 1), ("cosine", 1), ("dot", 2)])
def test_similarity_module_subclass_matches_stock(monkeypatch, distance, n_extra):
    """n_extra = item extra tokens in front of the catalogue: PAD (SASRec / HSTU, data_preparator.py:141) or PAD + MASK
    (BERT4Rec, bert4rec.py:80); the default whitelist is the non-extra items (nn/transformers/base.py:543-544)."""
    import torch

    from rectools_b200.integration import make_similarity_module

    DistanceSimilarityModule = fake_rectools(monkeypatch).rectools.models.nn.transformers.similarity.DistanceSimilarityModule

    n_users, n_tokens, d, k = 150, 400 + n_extra, 16, 7
    rng = np.random.default_rng(3)  # (numpy: the same values on every host, unlike torch's vectorised CPU sampler)
    user_embs = torch.from_numpy(rng.standard_normal((n_users, d), dtype=np.float32))
    item_embs = torch.from_numpy(rng.standard_normal((n_tokens, d), dtype=np.float32))
    g = torch.Generator().manual_seed(3)
    item_embs[:n_extra] = 0.0
    user_ids = np.random.default_rng(0).permutation(n_users)[:90]
    dense = (np.random.default_rng(1).random((len(user_ids), n_tokens)) < 0.05).astype(np.float32)
    dense[5, n_extra:] = 1.0  # everything viewed: the user gets no rows
    dense[6, n_extra : n_tokens - 3] = 1.0  # three candidates left: fewer than k rows
    ui = sparse.csr_matrix(dense)
    whitelist = np.arange(n_extra, n_tokens)
    stock = DistanceSimilarityModule(distance=distance)
    gold = np.load(os.path.join(GOLDEN, "similarity_module.npz"))
    exp = tuple(gold[f"{distance}|{n_extra}|{name}"] for name in ("users", "ids", "scores"))
    cls = make_similarity_module(ranker_factory=OracleTorchRanker)
    assert issubclass(cls, DistanceSimilarityModule) and cls.__mro__[1] is DistanceSimilarityModule
    got = cls(distance=distance)._recommend_u2i(user_embs, item_embs, user_ids, k, whitelist, ui)  # pylint: disable=protected-access
    np.testing.assert_array_equal(got[0], exp[0])
    assert_same_ranking(got[1], got[2], exp[1], exp[2], rtol=3e-5, atol=3e-6, tie_tol=3e-6)
    assert len(got[1]) < len(user_ids) * k and (np.asarray(got[1]) >= n_extra).all()
    # the forward pass (training logits) is inherited untouched
    assert "forward" not in cls.__dict__
    sess = torch.randn((4, 5, d), generator=g)
    cand = torch.randint(0, n_tokens, (4, 5, 3), generator=g)
    ours = cls(distance=distance)
    np.testing.assert_array_equal(stock(sess, item_embs).numpy(), ours(sess, item_embs).numpy())
    np.testing.assert_array_equal(stock(sess, item_embs, cand).numpy(), ours(sess, item_embs, cand).numpy())
