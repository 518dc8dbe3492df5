"""Host plan of the packed (padding-free) layout: build_plan(packed=True) against the padded plan of the same batch.
CPU only."""
import numpy as np
import pytest

from oracle import gato_oracle as O


def _check_packed(batch, context_len, pad_seq):
    from neko_b200._lib import SampleDesc
    from neko_b200.policy.packing import build_plan
    pad = build_plan(batch, patch_size=16, context_len=context_len, pad_seq=pad_seq)
    pk = build_plan(batch, patch_size=16, context_len=context_len, pad_seq=pad_seq, packed=True)
    B, S, W = pad.B, pad.seq_len, pad.width
    lengths = S - pad.first_valid
    row_base = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    descs = np.frombuffer(pk.descs.tobytes(), dtype=SampleDesc)
    assert pk.packed and not pad.packed
    assert np.array_equal(descs["row_base"], row_base)
    assert np.array_equal(pk.cu_seqlens, np.concatenate([row_base, [lengths.sum()]]))
    assert pk.token_rows == pk.n_valid_tokens == int(lengths.sum()) == pad.n_valid_tokens
    assert pad.token_rows == B * W
    # everything but the row base is the padded plan's: seq_len / width / first_valid feed the dropout coordinates
    assert (pk.B, pk.seq_len, pk.width) == (B, S, W) and np.array_equal(pk.first_valid, pad.first_valid)
    assert np.array_equal(np.frombuffer(pad.descs.tobytes(), dtype=SampleDesc)["row_base"], np.zeros(B))
    # padded b*W + first_valid[b] + p  <->  packed row_base[b] + p, one to one and in the same order
    b_of = np.searchsorted(pad.loss_rows, np.arange(B) * W, side="left")
    bi = np.repeat(np.arange(B), np.diff(np.concatenate([b_of, [len(pad.loss_rows)]])))
    p = pad.loss_rows - bi * W - pad.first_valid[bi]
    assert np.array_equal(pk.loss_rows, row_base[bi] + p)
    # the fused cross entropy reads its target at row + 1: that row is still inside the sample
    assert (p + 1 < lengths[bi]).all() and (p >= 0).all()
    return pk


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
def test_packed_plan_configs(name):
    ctx = O.CONFIGS[name]["context_len"]
    pk = _check_packed(O.synth_batch(name), ctx, False)
    if name == "cfg5":
        assert 0 < pk.n_valid_tokens < pk.B * pk.seq_len     # the mixed batch carries padding that packing removes


@pytest.mark.parametrize("seed", range(8))
def test_packed_plan_random_mixed_batches(seed):
    from _random_batches import random_mixed_batch
    batch, ctx, pad_seq = random_mixed_batch(seed)
    _check_packed(batch, ctx, pad_seq)


def test_pack_sequences_flag_parses():
    from neko_b200.training.arguments import parse_args
    assert parse_args([]).pack_sequences is False
    assert parse_args(["--pack_sequences"]).pack_sequences is True
    assert parse_args(["--pack_sequences", "false"]).pack_sequences is False
