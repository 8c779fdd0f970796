"""The drop-in recommenders accept the embedding sizes every kernel family is compiled for (8, 16, 32, 64, 128, 256)
and refuse the others up front with a ValueError (no CPU or generic fallback exists)."""
import types

import pytest


class _Probe:
    pass


def _make(emb_size):
    from arlib_b200.recommender._base import GraphRecommender

    class Rec(GraphRecommender):
        def _build_model(self):
            return _Probe()
    args = types.SimpleNamespace(topK="10,20", emb_size=emb_size)
    return Rec(args, data=None)


@pytest.mark.parametrize("emb_size", [8, 16, 32, 64, 128, 256])
def test_supported_widths_pass_the_gate(emb_size):
    assert isinstance(_make(emb_size).model, _Probe)


@pytest.mark.parametrize("emb_size", [4, 12, 24, 48, 100, 512])
def test_other_widths_raise_value_error(emb_size):
    with pytest.raises(ValueError, match="8, 16, 32, 64, 128, 256"):
        _make(emb_size)
