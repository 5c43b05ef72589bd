"""The self-play step options on the CPU oracle (tests/selfplay_oracle.c): the categorical draw of the played action and the uniform root
prior; and the constants of include/eaz_b200.h against _abi."""
import os
import re

import numpy as np

from e_alphazero_b200 import _abi
from oracle import oracle as O
from tests import helpers as H
from tests import selfplay_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ties_go_to_the_lowest_index():
    w = np.full((3, 5), 0.2, np.float32)
    g = np.zeros((3, 5), np.float32)
    g[1, [1, 3]] = 0.5
    g[2, [2, 4]] = 0.25
    assert SO.sample_actions(w, g).tolist() == [0, 1, 2]


def test_temperature_scaling():
    # x = log w: log 0.6 - log 0.3 = log 2 = 0.693; noise 0.5 on action 1 loses at T = 1 (0.5 < 0.693), wins at T = 0.5 only if it
    # exceeds 2 log 2, so it still loses; at T = 2 the gap is log 2 / 2 = 0.347 < 0.5 and action 1 wins
    w = np.array([[0.6, 0.3, 0.1]], np.float32)
    g = np.array([[0.0, 0.5, 0.0]], np.float32)
    assert SO.sample_actions(w, g, 1.0)[0] == 0
    assert SO.sample_actions(w, g, 0.5)[0] == 0
    assert SO.sample_actions(w, g, 2.0)[0] == 1
    # a tiny temperature is the argmax of w whatever the noise; a huge one the argmax of the noise
    rng = np.random.default_rng(0)
    w = rng.dirichlet(np.ones(6), 500).astype(np.float32)
    g = rng.gumbel(size=(500, 6)).astype(np.float32)
    assert (SO.sample_actions(w, g, 1e-6) == w.argmax(1)).all()
    assert (SO.sample_actions(w, g, 1e30) == g.argmax(1)).all()


def test_invalid_actions_are_never_drawn():
    rng = np.random.default_rng(1)
    B, A = 4000, 7
    w = rng.dirichlet(np.ones(A), B).astype(np.float32)
    g = (rng.gumbel(size=(B, A)) * 30).astype(np.float32)  # noise large enough to overturn any weight
    inv = rng.random((B, A)) < 0.4
    inv[:, 0] &= rng.random(B) < 0.5
    inv[np.arange(B), rng.integers(0, A, B)] = False  # at least one valid action per row
    a = SO.sample_actions(w, g, 1.0, inv)
    assert not inv[np.arange(B), a].any()
    # the valid actions all occur: the mask removes, it does not bias towards the lowest index
    assert len(np.unique(a)) == A


def test_all_invalid_row_plays_zero():
    w = np.array([[0.1, 0.7, 0.2], [0.1, 0.7, 0.2]], np.float32)
    g = np.array([[0.0, 3.0, 9.0], [0.0, 3.0, 9.0]], np.float32)
    inv = np.array([[1, 1, 1], [1, 0, 1]], np.uint8)
    assert SO.sample_actions(w, g, 1.0, inv).tolist() == [0, 1]


def test_sampling_matches_the_distribution():
    # Gumbel-max at temperature T draws w^(1/T) / sum: frequencies over 200000 draws within 5 sigma
    rng = np.random.default_rng(2)
    w = np.array([0.5, 0.3, 0.15, 0.05], np.float32)
    n = 200000
    for T in (1.0, 0.5):
        g = rng.gumbel(size=(n, 4)).astype(np.float32)
        f = np.bincount(SO.sample_actions(np.tile(w, (n, 1)), g, T), minlength=4) / n
        p = w.astype(np.float64) ** (1 / T)
        p /= p.sum()
        assert (np.abs(f - p) < 5 * np.sqrt(p * (1 - p) / n)).all(), (T, f, p)


def test_stream_gumbel_is_standard_gumbel_and_salted():
    g = SO.stream_gumbel(7, 3, 256, 64)
    root = SO.stream_gumbel(7, 3, 256, 64, sample=False)
    assert not np.array_equal(g, root)  # the sample noise is its own stream
    assert not np.array_equal(g, SO.stream_gumbel(7, 4, 256, 64))  # and moves with the counter
    assert np.array_equal(g[100:], SO.stream_gumbel(7, 3, 156, 64, tree0=100))  # keyed by the tree index
    assert abs(g.mean() - np.euler_gamma) < 0.02 and abs(g.var() - np.pi ** 2 / 6) < 0.1


def test_uniform_prior_masks_invalid_actions():
    env = H.make_env("deepsea", seed=3, size=10)
    net = H.make_net(env, seed=4)
    B = 32
    root = H.make_root(env, net, B, seed=5, invalid_frac=0.3)
    cfg = _abi.default_search_config(num_simulations=16, root_prior=_abi.ROOT_PRIOR_UNIFORM)
    out = SO.search(cfg, env, net, root)
    inv = root["invalid_actions"].astype(bool)
    pl = out["children_prior_logits"][:, 0]
    assert (pl[~inv] == 0).all() and (pl[inv] == np.float32(-3.4028234663852886e38)).all()
    # only the root prior changes: the root value of the tree is the caller's
    assert np.array_equal(out["raw_values"][:, 0], root["value"])
    given = O.search(_abi.default_search_config(num_simulations=16), env, net, root)
    assert not np.array_equal(out["action_weights"], given["action_weights"])


def test_header_constants_match_abi():
    header = open(os.path.join(ROOT, "include", "eaz_b200.h")).read()
    consts = dict((k, int(v)) for k, v in re.findall(r"\bEAZ_((?:ROOT_PRIOR|ACTION)_[A-Z]+)\s*=\s*(\d+)", header))
    assert consts == dict(ROOT_PRIOR_GIVEN=_abi.ROOT_PRIOR_GIVEN, ROOT_PRIOR_UNIFORM=_abi.ROOT_PRIOR_UNIFORM, ACTION_SEARCH=_abi.ACTION_SEARCH,
                          ACTION_VISITS=_abi.ACTION_VISITS, ACTION_IMPROVED=_abi.ACTION_IMPROVED)
    cfg = _abi.default_search_config()
    assert (cfg.root_prior, cfg.action_sampling) == (0, 0)  # zero = off: zero-initialised structs keep the search's own action
    assert _abi.EazSearchConfig.action_sampling.offset == _abi.EazSearchConfig.noise_seed.offset + 8
    assert _abi.EazSearchInputs.sample_gumbel.offset == _abi.EazSearchInputs.net.offset + 8
