"""CPU tests (no GPU) of the sharded learned table: the argument checks of train(shard_embeddings=True), which run before
anything touches a device, and the input check of ShardedEmbedding."""
import inspect

import pytest
import torch

from grapes_b200._lib import GrapesError


def _args(**kw):
    from grapes_b200.args import Arguments
    a = Arguments()
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_shard_embeddings_is_keyword_only():
    from grapes_b200.train import train
    assert inspect.signature(train).parameters["shard_embeddings"].kind is inspect.Parameter.KEYWORD_ONLY
    assert inspect.signature(train).parameters["shard_embeddings"].default is False


def test_train_refuses_shard_embeddings_without_embed_nodes():
    from grapes_b200.train import train
    with pytest.raises(GrapesError, match="shard_features"):
        train(_args(embed_nodes=False), shard_embeddings=True)


def test_train_refuses_full_batch_evaluation_without_shard_eval():
    from grapes_b200.train import train
    with pytest.raises(GrapesError, match="shard_eval"):
        train(_args(embed_nodes=True, eval_full_batch=True), shard_embeddings=True, shard_eval=False)


@pytest.mark.parametrize("x", [torch.zeros(10, 6), torch.zeros(10, 8, dtype=torch.bfloat16), torch.zeros(10)])
def test_sharded_learned_table_is_fp32_of_width_a_multiple_of_4(x):
    from grapes_b200.dist import ShardedEmbedding
    with pytest.raises(GrapesError, match="multiple of 4"):
        ShardedEmbedding.emulate(x, 2)
