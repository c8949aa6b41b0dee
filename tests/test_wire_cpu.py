"""Flat episode wire format (section 8 f-2): lossless w.r.t. the per-moment decode, backward compatible."""
import os
import pickle
import sys

import numpy as np
import pytest

from conftest import GOLDEN
from handyrl_b200 import wire
from handyrl_b200.batch import decode_moments, flatten_moments, tree_leaves, make_batch
from handyrl_b200.replay import DeviceReplay

with open(os.path.join(GOLDEN, 'batch_cases.pkl'), 'rb') as f:
    CASES = pickle.load(f)


def same_flat(a, b):
    assert a.steps == b.steps and list(a.players) == list(b.players)
    for k in wire._FIELDS:
        x, y = getattr(a, k), getattr(b, k)
        assert x.dtype == y.dtype and np.array_equal(x, y), k
    for x, y in zip(tree_leaves(a.obs), tree_leaves(b.obs)):
        assert x.dtype == y.dtype and np.array_equal(x, y)


@pytest.mark.parametrize('name', sorted(CASES))
def test_pack_unpack_is_lossless(name):
    for ep in CASES[name]['episodes']:
        want = flatten_moments(decode_moments(ep['moment']), ep['outcome'])
        packed = wire.pack_episode(ep)
        assert packed['moment'] == ep['moment'] and packed['steps'] == ep['steps'] and packed['outcome'] == ep['outcome']
        same_flat(wire.episode_to_flat(packed), want)
        slim = wire.pack_episode(ep, drop_moments=True)
        assert slim['moment'] == [] and 'flat' in slim
        same_flat(wire.episode_to_flat(slim), want)
        assert wire.pack_episode(packed) is packed           # idempotent


def test_replay_accepts_both_formats():
    eps = CASES['geister_burnin']['episodes']
    a = DeviceReplay(4096, 64, device='cpu')
    b = DeviceReplay(4096, 64, device='cpu')
    for ep in eps:
        a.add(ep)
        b.add(wire.pack_episode(ep, drop_moments=True))
    for k in ('st_obs', 'st_prob', 'st_action', 'st_amask', 'st_value', 'st_reward', 'st_return', 'st_flags', 'st_turn', 'st_outcome'):
        assert (getattr(a, k) == getattr(b, k)).all(), k


def test_worker_hook_makes_the_reference_generator_ship_flat_episodes(monkeypatch):
    """The hook wraps Generator.generate of an importable `handyrl.generation`; here that module is a stand-in whose
    generate returns the episode the reference's own Generator produced (golden: generator_cases.pkl)."""
    import copy
    import types
    with open(os.path.join(GOLDEN, 'generator_cases.pkl'), 'rb') as f:
        golden = pickle.load(f)['tictactoe']

    class Generator:
        def __init__(self, env, args):
            self.args = args

        def generate(self, models, args):
            return copy.deepcopy(golden['episode'])

    gen = types.ModuleType('handyrl.generation')
    gen.Generator = Generator
    pkg = types.ModuleType('handyrl')
    pkg.generation = gen
    monkeypatch.setitem(sys.modules, 'handyrl', pkg)
    monkeypatch.setitem(sys.modules, 'handyrl.generation', gen)
    plain = Generator.generate
    assert wire.install_worker_hook() is plain and Generator.generate is not plain
    assert wire.install_worker_hook() is Generator.generate          # a second install does not wrap twice
    ep = Generator(None, golden['args']).generate({}, golden['episode']['args'])
    assert ep is not None and 'flat' in ep and ep['steps'] == len(decode_moments(ep['moment']))
    assert ep['moment'] == golden['episode']['moment'] and ep['outcome'] == golden['episode']['outcome']
    same_flat(wire.unpack_flat(ep['flat']), flatten_moments(decode_moments(ep['moment']), ep['outcome']))
