"""CPU checks of mixed negative sampling: the oracle's sampled-negative stream (oracle/twotower_sampled.py) and the option
checks that TwoTowerModel and ShardedTwoTowerNet share (twoTower.check_sampled_options)."""
import numpy as np
import pytest
import torch


def test_stream_is_the_philox_definition():
    from oracle import philox as P
    from oracle import twotower_sampled as OS
    M, seed, t, r, lo, hi = 37, 99, 2 ** 33 + 7, 5, 2, 1002
    got = OS.sampled_negatives(M, seed, t, r, lo, hi)
    for k in (0, 1, 36):
        ctr = np.array([[k, t & 0xFFFFFFFF, t >> 32, OS.TAG_TWOTOWER_NEG]], dtype=np.uint32)
        w = int(P.philox4x32_10(ctr, (seed, r))[0, 0])
        assert got[k] == lo + ((w * (hi - lo)) >> 32)
    assert got.dtype == np.int32 and got.min() >= lo and got.max() < hi


def test_stream_depends_on_step_replica_and_seed():
    from oracle import twotower_sampled as OS
    base = OS.sampled_negatives(500, 42, 1, 0, 2, 10 ** 6)
    assert np.array_equal(base, OS.sampled_negatives(500, 42, 1, 0, 2, 10 ** 6))
    for other in (OS.sampled_negatives(500, 42, 2, 0, 2, 10 ** 6), OS.sampled_negatives(500, 42, 1, 1, 2, 10 ** 6),
                  OS.sampled_negatives(500, 43, 1, 0, 2, 10 ** 6), OS.sampled_negatives(500, 42, 1 + 2 ** 32, 0, 2, 10 ** 6)):
        assert not np.array_equal(base, other)
    assert np.array_equal(OS.sampled_negatives(10, 42, 1, 0, 2, 10 ** 6), base[:10])    # draw k does not depend on M


def test_uniform_over_the_range():
    from oracle import twotower_sampled as OS
    ids = OS.sampled_negatives(200000, 7, 3, 0, 2, 12)
    counts = np.bincount(ids - 2, minlength=10)
    assert counts.min() > 19000 and counts.max() < 21000


def test_oracle_without_draws_is_the_retrieval_oracle():
    from oracle import twotower_retrieval as OR
    from oracle import twotower_sampled as OS
    a, b = OR.RetrievalOracle(20, 15, 8, 4, temperature=0.5), OS.SampledOracle(20, 15, 8, 4, temperature=0.5)
    u, i = np.array([2, 3, 4, 5]), np.array([2, 2, 7, 9])
    assert float(a.loss(u, i, cand_ids=i)) == float(b.loss(u, i, cand_ids=i, sampled=np.zeros(0, np.int32)))


def test_sampled_columns_extend_the_softmax():
    """By hand: logits over the batch's and the sampled columns, a sampled copy of the positive masked, weights."""
    from oracle import twotower_sampled as OS
    o = OS.SampledOracle(20, 15, 8, 4, temperature=2.0)
    u, i, smp, w = np.array([2, 3, 4]), np.array([2, 5, 5]), np.array([5, 9], np.int32), np.array([1.0, 0.5, 2.0], np.float32)
    with torch.no_grad():
        q, c = o.towers(u, np.concatenate([i, smp]))
        s = (q @ c.T) / 2.0
        ids = np.concatenate([i, smp])
        ref = 0.0
        for b in range(3):
            keep = [j for j in range(5) if j == b or ids[j] != i[b]]
            ref += w[b] * float(torch.logsumexp(s[b, keep], 0) - s[b, b])
        got = float(o.loss(u, i, cand_ids=i, sample_weight=w, sampled=smp))
    assert abs(got - ref) <= 1e-5 * abs(ref)


def test_option_checks():
    from binrec_b200.twoTower import check_sampled_options as chk
    assert chk(None, False, False, None, False) == 0 and chk(False, False, False, None, False) == 0
    assert chk(128, False, False, None, False) == 128 and chk(np.int64(3), False, False, False, False) == 3
    for bad in (0, -1, 2.5, True):
        with pytest.raises(ValueError, match="integer >= 1"):
            chk(bad, False, False, None, False)
    with pytest.raises(ValueError, match="rdZero"):
        chk(4, True, False, None, False)
    with pytest.raises(ValueError, match="global_negatives"):
        chk(4, False, True, None, False)
    with pytest.raises(ValueError, match="streamingFrequency"):
        chk(4, False, False, 0.01, False)
    with pytest.raises(ValueError, match="candidate probabilities"):
        chk(4, False, False, None, True)
