"""CPU: `install()` / `uninstall()` rebind the ranker name that VectorModel / EASEModel use (vector.py:28, ease.py:31).
The rectools modules are the stand-ins of `tests.helpers.fake_rectools`."""
import pytest

from tests.helpers import fake_rectools


def test_install_rebinds_ranker(monkeypatch):
    rt = fake_rectools(monkeypatch)
    ease, vector = rt.rectools.models.ease, rt.rectools.models.vector

    import rectools_b200
    from rectools_b200.integration import B200ImplicitRanker

    orig = vector.ImplicitRanker
    rectools_b200.install(device=0, tc_mode="auto")
    try:
        assert vector.ImplicitRanker is B200ImplicitRanker and ease.ImplicitRanker is B200ImplicitRanker
        # constructor signature of ImplicitRanker (rank_implicit.py:58-65) is accepted; without a GPU it fails where one is needed
        import numpy as np
        import torch

        from rectools_b200 import _lib

        args = (vector.Distance.DOT, np.ones((2, 3)), np.ones((4, 3)))
        if torch.cuda.is_available():
            assert isinstance(vector.ImplicitRanker(*args, num_threads=2, use_gpu=False), B200ImplicitRanker)
        else:
            with pytest.raises(_lib.B200RankError):
                vector.ImplicitRanker(*args, num_threads=2, use_gpu=False)
    finally:
        rectools_b200.uninstall()
    assert vector.ImplicitRanker is orig and ease.ImplicitRanker is orig


def test_distance_enum_matches_reference_values():
    from rectools_b200 import Distance

    assert [d.value for d in Distance] == ["dot", "cosine", "euclidean"]
