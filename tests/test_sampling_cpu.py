"""CPU: (1) the host parity samplers reproduce the reference's sampled indices BIT-EXACTLY under a
fixed seed (golden vectors from the unmodified reference, tests/golden/gen_sampling.py and
tests/golden/gen_reference_answers.py); (2) the oracle's Philox restatement is self-consistent (known-answer vector)."""
import os
import random

import numpy as np
import pytest

from oracle import sampling as osm

from _fixtures import load_reference_answers

GOLD = os.path.join(os.path.dirname(__file__), "golden", "sampling.npz")


def _setup():
    g = np.load(GOLD)
    n_users, n_items = int(g["n_users"]), int(g["n_items"])
    consumed = {u: g["idx"][g["indptr"][u]:g["indptr"][u + 1]].tolist() for u in range(n_users)}
    return g, n_users, n_items, consumed


def test_parity_mode_bit_exact_against_reference_golden():
    from librecommender_b200 import sampling as S

    g, n_users, n_items, consumed = _setup()
    seed = int(g["seed"])
    assert seed == S.collator_seed(42)
    for num_neg in (1, 3):
        rng = np.random.default_rng(seed)
        np.testing.assert_array_equal(S.negatives_from_random(rng, n_items, g["items_pos"], num_neg),
                                      g[f"random_{num_neg}"])
        rng = np.random.default_rng(seed)
        np.testing.assert_array_equal(S.negatives_from_random(rng, 50, g["items_pos"] % 50, num_neg),
                                      g[f"random_big_{num_neg}"])
        rng = np.random.default_rng(seed)
        np.testing.assert_array_equal(
            S.negatives_from_popular(rng, n_items, g["items_pos"], num_neg, probs=g["probs"]),
            g[f"popular_{num_neg}"])
        random.seed(seed)
        cs = [set(consumed[u]) for u in range(n_users)]
        got = S.negatives_from_unconsumed(cs, g["users"], g["items_pos"], n_items, num_neg)
        np.testing.assert_array_equal(got, g[f"unconsumed_{num_neg}"])
        osm.check_reference_invariants(got, g["users"], g["items_pos"], num_neg, n_items, consumed)


def random_negative_cases():
    gen = np.random.default_rng(9)
    for trial in range(5):
        n_items = int(gen.integers(20, 3000))
        pos = gen.integers(0, n_items, size=int(gen.integers(1, 500)))
        num_neg = int(gen.integers(1, 6))
        yield n_items, pos, num_neg


def test_parity_mode_vs_live_reference():
    from librecommender_b200 import sampling as S

    g = load_reference_answers()
    for trial, (n_items, pos, num_neg) in enumerate(random_negative_cases()):
        b = S.negatives_from_random(np.random.default_rng(trial), n_items, pos, num_neg)
        np.testing.assert_array_equal(g[f"negatives_{trial}"], b)


def test_probs_from_frequency_and_philox_known_answer():
    from librecommender_b200 import sampling as S

    item_consumed = {0: [1, 2, 2], 1: [3], 2: [0, 1, 2, 3]}
    p = S.neg_probs_from_frequency(item_consumed, 3, 0.75)
    np.testing.assert_allclose(p, osm.neg_probs_from_frequency(item_consumed, 3, 0.75))
    np.testing.assert_allclose(p.sum(), 1.0)
    # Random123 known-answer test for philox4x32-10: counter = key = 0
    out = osm.philox4x32_10(0, 0, 0, 0, 0, 0)
    assert [int(x) for x in out] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    out = osm.philox4x32_10(0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff)
    assert [int(x) for x in out] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
