"""CPU tests (no GPU) of the sharded feature table: the row bounds, the pitch, the chunked fill plan, and the argument
checks of train(shard_features=True) and evaluate(features=...) that run before anything touches a device."""
import types

import pytest
import torch

from grapes_b200._lib import GrapesError
from grapes_b200.dist import feature_bounds, feature_pitch, fill_plan


@pytest.mark.parametrize("N,W", [(10, 1), (10, 3), (12, 4), (3, 8), (0, 2), (244_160_499, 8), (111_059_956, 7)])
def test_bounds_are_equal_contiguous_ranges(N, W):
    b = feature_bounds(N, W)
    per = -(-N // W)
    assert len(b) == W + 1 and b[0] == 0 and b[-1] == N
    assert all(b[r] <= b[r + 1] for r in range(W))
    assert all(b[r + 1] - b[r] == per for r in range(W) if (r + 1) * per <= N)      # full ranges first
    assert max(b[r + 1] - b[r] for r in range(W)) == per                            # no rank holds more than ceil(N / W)
    assert b == [min(N, r * per) for r in range(W + 1)]


def test_pitch_keeps_rows_aligned():
    for F in range(1, 40):
        ld = feature_pitch(F)
        assert ld >= F and ld % 4 == 0 and ld - F < 4      # 16-byte fp32 rows, 8-byte bf16 rows
    assert feature_pitch(602) == 604 and feature_pitch(128) == 128 and feature_pitch(130) == 132


@pytest.mark.parametrize("lo,hi,row_bytes,chunk", [(0, 100, 8, 64), (5, 5, 8, 64), (7, 1000, 3072, 1 << 20),
                                                   (0, 10, 1 << 31, 1 << 30), (30_520_000, 61_040_000, 256, 1 << 30)])
def test_fill_plan_covers_the_shard_in_bounded_chunks(lo, hi, row_bytes, chunk):
    plan = fill_plan(lo, hi, row_bytes, chunk)
    if hi == lo:
        assert plan == []
        return
    assert plan[0][0] == lo and plan[-1][1] == hi
    assert all(a < b for a, b in plan) and all(plan[i][1] == plan[i + 1][0] for i in range(len(plan) - 1))
    assert all((b - a) * row_bytes <= chunk for a, b in plan) or all(b - a == 1 for a, b in plan)


def _args(**kw):
    from grapes_b200.args import Arguments
    a = Arguments()
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_train_refuses_shard_features_with_embed_nodes():
    from grapes_b200.train import train
    with pytest.raises(GrapesError, match="embed_nodes"):
        train(_args(embed_nodes=True), shard_features=True)


def test_train_refuses_full_batch_evaluation_without_shard_eval():
    from grapes_b200.train import train
    with pytest.raises(GrapesError, match="shard_eval"):
        train(_args(eval_full_batch=True), shard_features=True, shard_eval=False)


def test_shard_features_is_keyword_only():
    import inspect
    from grapes_b200.eval import evaluate
    from grapes_b200.train import train
    assert inspect.signature(train).parameters["shard_features"].kind is inspect.Parameter.KEYWORD_ONLY
    assert inspect.signature(evaluate).parameters["features"].kind is inspect.Parameter.KEYWORD_ONLY


def test_full_batch_evaluation_of_a_sharded_table_needs_a_group():
    from grapes_b200.eval import evaluate
    data = types.SimpleNamespace(x=None, y=torch.zeros(4, dtype=torch.long), num_nodes=4)
    with pytest.raises(GrapesError, match="mini-batch"):
        evaluate(None, None, data, None, None, None, 0, "cpu", full_batch=True, features=object())
