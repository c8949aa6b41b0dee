"""Generate the golden vectors by RUNNING THE REFERENCE (DeNA/HandyRL) on seeded inputs.

Run in the build container only (the reference is mounted at /root/reference there):

    python tests/golden/gen_golden.py

Outputs (committed):
    tests/golden/loss_cases.npz     compute_loss + autograd on synthetic batches (train.py:218-267)
    tests/golden/target_cases.npz   compute_target per algorithm (losses.py:63-80)
    tests/golden/batch_cases.pkl    make_batch on real self-play episodes (train.py:33-124)
    tests/golden/step_cases.pkl     3 full optimiser steps of the reference Trainer maths (train.py:366-371)
    tests/golden/rnn_cases.pkl      recurrent forward_prediction + compute_loss + parameter gradients (train.py:147-174)
    tests/golden/net_step_cases.pkl 3 optimiser steps of the reference's GeisterNet (DRC ConvLSTM, recurrent path) and
                                    GeeseNet (torus convolutions; `kaggle_environments` stubbed, SURVEY.md 8c)
    tests/golden/generator_cases.pkl one self-play episode from the reference's Generator (generation.py:20-93)

The reference has no golden vectors of its own for this path (SURVEY.md 8c), so the
vectors are the reference's own outputs.  The fp64 quirk of `selected_prob` is avoided by
feeding float32 tensors (SURVEY.md hard part 4).
"""
import os
import sys
import pickle
import random
import itertools

import numpy as np

REF = os.environ.get('HANDYRL_REFERENCE', '/root/reference')
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import handyrl.train as ref_train  # noqa: E402
import handyrl.losses as ref_losses  # noqa: E402
from handyrl.environment import make_env, prepare_env  # noqa: E402
from handyrl.generation import Generator  # noqa: E402
from handyrl.model import ModelWrapper  # noqa: E402

from handyrl_b200.synthetic import synthetic_batch, synthetic_outputs  # noqa: E402

ALGOS = ['MC', 'TD', 'UPGO', 'VTRACE']


class FixedOutputs(torch.nn.Module):
    """Stands in for the user's net: returns fixed leaf tensors so that only the
    reference's mask epilogue + loss maths is differentiated."""

    def __init__(self, outs):
        super().__init__()
        self.outs = outs

    def forward(self, obs, hidden=None):
        return {k: v.flatten(0, 2) for k, v in self.outs.items()}


def loss_case(name, *, B, T, P, A, turn_based, observation, has_value, has_return,
              burn_in, policy_target, value_target, reward_kind, lmb=0.7, gamma=0.8, seed=0):
    args = {
        'turn_based_training': turn_based, 'observation': observation,
        'gamma': gamma, 'lambda': lmb, 'burn_in_steps': burn_in, 'forward_steps': T - burn_in,
        'entropy_regularization': 0.1, 'entropy_regularization_decay': 0.1,
        'policy_target': policy_target, 'value_target': value_target,
    }
    batch = synthetic_batch(B, T, P, A, turn_based=turn_based, observation=observation,
                            reward_kind=reward_kind, gamma=gamma, seed=seed, burn_in=burn_in)
    outs = synthetic_outputs(batch, has_value=has_value, has_return=has_return, seed=seed + 1)
    leaves = {k: v.clone().requires_grad_(True) for k, v in outs.items()}
    losses, dcnt = ref_train.compute_loss(batch, FixedOutputs(leaves), None, args)
    losses['total'].backward()

    rec = {'meta': np.array(repr(dict(B=B, T=T, P=P, A=A, turn_based=turn_based, observation=observation,
                                     has_value=has_value, has_return=has_return, burn_in=burn_in,
                                     policy_target=policy_target, value_target=value_target,
                                     reward_kind=reward_kind, lmb=lmb, gamma=gamma, seed=seed)))}
    for k, v in batch.items():
        if k != 'observation':
            rec['in.' + k] = v.numpy()
    for k, v in outs.items():
        rec['out.' + k] = v.numpy()
        rec['grad.' + k] = leaves[k].grad.numpy()
    for k, v in losses.items():
        rec['loss.' + k] = np.float64(v.item())
    rec['loss.dcnt'] = np.float64(dcnt)
    return {name + '/' + k: v for k, v in rec.items()}


def gen_loss_cases():
    cases = {}
    n = 0
    # every policy_target x value_target, on the three layouts, TicTacToe-like and Geister-like
    for pt, vt in itertools.product(ALGOS, ALGOS):
        for layout, (turn_based, observation, P) in {
                'alt': (True, False, 2), 'sim': (False, False, 2), 'obs': (True, True, 2)}.items():
            has_return = (n % 2 == 1)
            cases.update(loss_case('%s_%s_%s' % (layout, pt, vt), B=6, T=9, P=P, A=9,
                                   turn_based=turn_based, observation=observation,
                                   has_value=True, has_return=has_return, burn_in=0,
                                   policy_target=pt, value_target=vt,
                                   reward_kind='step' if has_return or n % 3 == 0 else 'zero', seed=100 + n))
            n += 1
    # burn-in, no value head, 4 players, solo player, wide action space, long T
    extra = [
        dict(name='burnin_alt', B=5, T=10, P=2, A=9, turn_based=True, observation=False, has_value=True,
             has_return=True, burn_in=3, policy_target='UPGO', value_target='VTRACE', reward_kind='step'),
        dict(name='burnin_obs', B=5, T=10, P=2, A=7, turn_based=True, observation=True, has_value=True,
             has_return=True, burn_in=2, policy_target='TD', value_target='TD', reward_kind='step'),
        dict(name='novalue_alt', B=4, T=8, P=2, A=9, turn_based=True, observation=False, has_value=False,
             has_return=False, burn_in=0, policy_target='VTRACE', value_target='VTRACE', reward_kind='step'),
        dict(name='novalue_ret', B=4, T=8, P=2, A=9, turn_based=False, observation=False, has_value=False,
             has_return=True, burn_in=0, policy_target='UPGO', value_target='TD', reward_kind='step'),
        dict(name='geese4', B=4, T=8, P=4, A=4, turn_based=False, observation=False, has_value=True,
             has_return=False, burn_in=0, policy_target='VTRACE', value_target='VTRACE', reward_kind='zero'),
        dict(name='alt4', B=4, T=9, P=4, A=5, turn_based=True, observation=False, has_value=True,
             has_return=True, burn_in=0, policy_target='UPGO', value_target='VTRACE', reward_kind='step'),
        dict(name='solo1', B=5, T=8, P=1, A=6, turn_based=False, observation=False, has_value=True,
             has_return=True, burn_in=0, policy_target='TD', value_target='VTRACE', reward_kind='step'),
        dict(name='wide', B=3, T=6, P=2, A=214, turn_based=True, observation=True, has_value=True,
             has_return=True, burn_in=1, policy_target='TD', value_target='TD', reward_kind='step'),
        dict(name='wide512', B=2, T=5, P=2, A=512, turn_based=True, observation=False, has_value=True,
             has_return=False, burn_in=0, policy_target='UPGO', value_target='VTRACE', reward_kind='zero'),
        dict(name='odd33', B=3, T=7, P=2, A=33, turn_based=False, observation=False, has_value=True,
             has_return=False, burn_in=0, policy_target='UPGO', value_target='VTRACE', reward_kind='zero'),
        dict(name='a1', B=3, T=5, P=2, A=1, turn_based=True, observation=False, has_value=True,
             has_return=False, burn_in=0, policy_target='TD', value_target='TD', reward_kind='zero'),
        dict(name='t1', B=4, T=1, P=2, A=9, turn_based=True, observation=False, has_value=True,
             has_return=True, burn_in=0, policy_target='UPGO', value_target='VTRACE', reward_kind='step'),
        dict(name='long', B=3, T=70, P=2, A=9, turn_based=True, observation=False, has_value=True,
             has_return=False, burn_in=0, policy_target='UPGO', value_target='VTRACE', reward_kind='zero'),
        dict(name='cfg2_small', B=32, T=32, P=2, A=9, turn_based=True, observation=False, has_value=True,
             has_return=False, burn_in=0, policy_target='UPGO', value_target='VTRACE', reward_kind='zero'),
    ]
    for i, e in enumerate(extra):
        name = e.pop('name')
        cases.update(loss_case(name, seed=500 + i, **e))
    np.savez_compressed(os.path.join(HERE, 'loss_cases.npz'), **cases)
    print('loss cases:', len({k.split('/')[0] for k in cases}))


def gen_target_cases():
    g = torch.Generator().manual_seed(7)
    cases = {}
    B, T, P = 5, 11, 2
    for i, algo in enumerate(ALGOS):
        for bc in ('full', 'pa1'):
            values = torch.tanh(torch.randn((B, T, P, 1), generator=g))
            returns = torch.randn((B, T, P, 1), generator=g)
            rewards = 0.1 * torch.randn((B, T, P, 1), generator=g)
            rshape = (B, T, P, 1) if bc == 'full' else (B, T, 1, 1)
            rhos = torch.rand(rshape, generator=g)
            cs = torch.rand(rshape, generator=g)
            masks = (torch.rand((B, T, P, 1), generator=g) < 0.7).float()
            tg, adv = ref_losses.compute_target(algo, values, returns, rewards, 0.7, 0.9, rhos, cs, masks)
            name = '%s_%s' % (algo, bc)
            for k, v in dict(values=values, returns=returns, rewards=rewards, rhos=rhos, cs=cs, masks=masks,
                             targets=tg, advantages=adv).items():
                cases[name + '/' + k] = v.numpy()
        # value-stream flavour: returns (B,1,P,1) = outcome, rewards None, gamma 1
        values = torch.tanh(torch.randn((B, T, P, 1), generator=g))
        outcome = torch.randn((B, 1, P, 1), generator=g)
        rhos = torch.rand((B, T, 1, 1), generator=g)
        masks = (torch.rand((B, T, P, 1), generator=g) < 0.7).float()
        tg, adv = ref_losses.compute_target(algo, values, outcome, None, 0.7, 1, rhos, rhos, masks)
        name = '%s_outcome' % algo
        for k, v in dict(values=values, returns=outcome, rhos=rhos, cs=rhos, masks=masks,
                         targets=tg, advantages=adv).items():
            cases[name + '/' + k] = v.numpy()
    np.savez_compressed(os.path.join(HERE, 'target_cases.npz'), **cases)
    print('target cases:', len({k.split('/')[0] for k in cases}))


def play_episodes(env_name, n, train_args, seed):
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    env_args = {'env': env_name}
    prepare_env(env_args)
    env = make_env(env_args)
    model = ModelWrapper(env.net())
    gen = Generator(env, train_args)
    eps = []
    while len(eps) < n:
        players = env.players()
        ep = gen.generate({p: model for p in players}, {'player': players, 'model_id': {p: 0 for p in players}})
        if ep is not None:
            eps.append(ep)
    return eps, env


def gen_batch_cases():
    out = {}
    setups = {
        'tictactoe': ('TicTacToe', dict(turn_based_training=True, observation=False, burn_in_steps=0)),
        'tictactoe_obs': ('TicTacToe', dict(turn_based_training=True, observation=True, burn_in_steps=0)),
        'geister_burnin': ('Geister', dict(turn_based_training=True, observation=True, burn_in_steps=2)),
        'parallel_ttt': ('handyrl.envs.parallel_tictactoe', dict(turn_based_training=False, observation=False,
                                                                   burn_in_steps=0)),
    }
    for name, (env_name, over) in setups.items():
        args = {'gamma': 0.8, 'forward_steps': 8, 'compress_steps': 4, 'maximum_episodes': 1000,
                'batch_size': 6, 'num_batchers': 1}
        args.update(over)
        eps, _ = play_episodes(env_name, 8, args, seed=11)
        # select windows with the reference's own sampler (train.py:291-315)
        random.seed(5)
        batcher = ref_train.Batcher.__new__(ref_train.Batcher)
        batcher.args, batcher.episodes = args, eps
        selected = [batcher.select_episode() for _ in range(args['batch_size'])]
        random.seed(9)  # make_batch draws the solo player with `random` (train.py:58)
        batch = ref_train.make_batch(selected, args)
        from handyrl.util import map_r
        out[name] = {'args': args, 'episodes': eps, 'selected': selected,
                     'batch': map_r(batch, lambda t: t.numpy())}
    with open(os.path.join(HERE, 'batch_cases.pkl'), 'wb') as f:
        pickle.dump(out, f)
    print('batch cases:', list(out))


def gen_step_cases():
    """Three optimiser steps with the reference's update rule (train.py:327-331, 366-371)."""
    import torch.nn as nn
    import torch.optim as optim
    out = {}
    for name, layout in {'alt': (True, False), 'sim': (False, False)}.items():
        torch.manual_seed(3)
        env_args = {'env': 'TicTacToe'}
        prepare_env(env_args)
        net = make_env(env_args).net()
        B, T, P, A = 16, 8, 2, 9
        args = {'turn_based_training': layout[0], 'observation': layout[1], 'gamma': 0.8, 'lambda': 0.7,
                'burn_in_steps': 0, 'forward_steps': T, 'entropy_regularization': 0.1,
                'entropy_regularization_decay': 0.1, 'policy_target': 'UPGO', 'value_target': 'VTRACE',
                'batch_size': B}
        state0 = {k: v.clone().numpy() for k, v in net.state_dict().items()}
        params = list(net.parameters())
        # lr is deliberately large so that three steps move the weights well above fp32 noise
        opt = optim.Adam(params, lr=1e-3, weight_decay=1e-5)
        wrapped = ModelWrapper(net)
        wrapped.train()
        steps = []
        for s in range(3):
            batch = synthetic_batch(B, T, P, A, turn_based=layout[0], observation=layout[1], seed=40 + s)
            losses, dcnt = ref_train.compute_loss(batch, wrapped, None, args)
            opt.zero_grad()
            losses['total'].backward()
            gnorm = nn.utils.clip_grad_norm_(params, 4.0)
            opt.step()
            steps.append({'losses': {k: float(v.item()) for k, v in losses.items()}, 'dcnt': float(dcnt),
                          'grad_norm': float(gnorm)})
        out[name] = {'args': args, 'dims': (B, T, P, A), 'state0': state0, 'steps': steps, 'lr': 1e-3,
                     'state3': {k: v.clone().numpy() for k, v in net.state_dict().items()}}
    with open(os.path.join(HERE, 'step_cases.pkl'), 'wb') as f:
        pickle.dump(out, f)
    print('step cases:', list(out))


def gen_rnn_cases():
    """Recurrent path: the reference's forward_prediction (train.py:147-174, burn-in, hidden masking)
    and compute_loss driving a small recurrent net with a dict observation; parameter gradients."""
    from handyrl_b200.nets import GatedBoardNet
    out = {}
    for name, (turn_based, observation, burn_in) in {'alt_burn2': (True, False, 2), 'obs_burn1': (True, True, 1),
                                                       'sim_burn0': (False, False, 0)}.items():
        torch.manual_seed(21)
        net = GatedBoardNet()
        B, T, P, A = 4, 6, 2, 12
        args = {'turn_based_training': turn_based, 'observation': observation, 'gamma': 0.8, 'lambda': 0.7,
                'burn_in_steps': burn_in, 'forward_steps': T - burn_in, 'entropy_regularization': 0.1,
                'entropy_regularization_decay': 0.1, 'policy_target': 'TD', 'value_target': 'TD'}
        batch = synthetic_batch(B, T, P, A, turn_based=turn_based, observation=observation, reward_kind='step',
                                seed=77, burn_in=burn_in, with_obs=False)
        Pa = batch['action'].shape[2]
        g = torch.Generator().manual_seed(78)
        batch['observation'] = {'scalar': torch.rand((B, T, Pa, 4), generator=g),
                                'board': (torch.rand((B, T, Pa, 3, 4, 4), generator=g) < 0.3).float()}
        state0 = {k: v.clone().numpy() for k, v in net.state_dict().items()}
        wrapped = ModelWrapper(net)
        wrapped.train()
        hidden = wrapped.init_hidden([B, P])
        masked = ref_train.forward_prediction(wrapped, hidden, batch, args)
        masked = {k: v.detach().numpy() for k, v in masked.items()}
        # fresh copy: forward_prediction updated BatchNorm running stats
        net.load_state_dict({k: torch.from_numpy(v) for k, v in state0.items()})
        wrapped.train()
        losses, dcnt = ref_train.compute_loss(batch, wrapped, wrapped.init_hidden([B, P]), args)
        losses['total'].backward()
        from handyrl.util import map_r
        out[name] = {'args': args, 'dims': (B, T, P, A), 'state0': state0,
                     'batch': map_r(batch, lambda t: t.numpy()), 'masked_outputs': masked,
                     'losses': {k: float(v.item()) for k, v in losses.items()}, 'dcnt': float(dcnt),
                     'param_grads': {k: p.grad.numpy().copy() for k, p in net.named_parameters()},
                     'state1': {k: v.clone().numpy() for k, v in net.state_dict().items()}}
    with open(os.path.join(HERE, 'rnn_cases.pkl'), 'wb') as f:
        pickle.dump(out, f)
    print('rnn cases:', list(out))


def _reference_steps(net, args, batches, hidden_fn, lr=1e-4):
    """Three optimiser steps exactly as Trainer.train does them (train.py:358-371)."""
    import torch.nn as nn
    import torch.optim as optim
    state0 = {k: v.clone().numpy() for k, v in net.state_dict().items()}
    params = list(net.parameters())
    opt = optim.Adam(params, lr=lr, weight_decay=1e-5)
    wrapped = ModelWrapper(net)
    wrapped.train()
    steps = []
    for batch in batches:
        losses, dcnt = ref_train.compute_loss(batch, wrapped, hidden_fn(wrapped, batch), args)
        opt.zero_grad()
        losses['total'].backward()
        gnorm = nn.utils.clip_grad_norm_(params, 4.0)
        opt.step()
        steps.append({'losses': {k: float(v.item()) for k, v in losses.items()}, 'dcnt': float(dcnt),
                      'grad_norm': float(gnorm)})
    return state0, steps, {k: v.clone().numpy() for k, v in net.state_dict().items()}


def geister_batch(B, T, P, A, turn_based, observation, burn_in, seed):
    from handyrl_b200.synthetic import synthetic_geister_batch
    return synthetic_geister_batch(B, T, P, A, turn_based=turn_based, observation=observation, burn_in=burn_in, seed=seed)


def gen_net_step_cases():
    """configs[2] / configs[3] of BASELINE.json with the reference's own networks."""
    import types
    from handyrl.envs.geister import GeisterNet
    stub = types.ModuleType('kaggle_environments')      # the env cannot run here; only the net is needed
    stub.make = lambda *a, **k: None
    sys.modules.setdefault('kaggle_environments', stub)
    from handyrl.envs.kaggle.hungry_geese import GeeseNet
    out = {}
    for name, (turn_based, observation) in {'geister_obs': (True, True), 'geister_alt': (True, False)}.items():
        torch.manual_seed(5)
        net = GeisterNet()
        B, T, P, A, burn_in = 6, 6, 2, 214, 2
        args = {'turn_based_training': turn_based, 'observation': observation, 'gamma': 0.8, 'lambda': 0.7,
                'burn_in_steps': burn_in, 'forward_steps': T - burn_in, 'entropy_regularization': 0.1,
                'entropy_regularization_decay': 0.1, 'policy_target': 'TD', 'value_target': 'TD', 'batch_size': B}
        batches = [geister_batch(B, T, P, A, turn_based, observation, burn_in, 60 + s) for s in range(3)]
        state0, steps, state3 = _reference_steps(net, args, batches, lambda w, b: w.init_hidden([B, P]))
        # lr 1e-4: Adam's first steps move every weight by ~lr*sign(g), so weights whose gradient is rounding noise
        # (e.g. conv biases in front of BatchNorm: analytically zero) diverge by 2*lr between equally valid fp32 runs
        out[name] = {'net': 'geister', 'args': args, 'dims': (B, T, P, A), 'seeds': [60, 61, 62], 'state0': state0,
                     'steps': steps, 'lr': 1e-4, 'state3': state3}
    torch.manual_seed(6)
    net = GeeseNet()
    B, T, P, A = 8, 4, 4, 4
    args = {'turn_based_training': False, 'observation': False, 'gamma': 0.8, 'lambda': 0.7, 'burn_in_steps': 0,
            'forward_steps': T, 'entropy_regularization': 0.1, 'entropy_regularization_decay': 0.1,
            'policy_target': 'VTRACE', 'value_target': 'VTRACE', 'batch_size': B}
    from handyrl_b200.synthetic import synthetic_geese_batch
    batches = [synthetic_geese_batch(B, T, P, A, seed=80 + s) for s in range(3)]
    state0, steps, state3 = _reference_steps(net, args, batches, lambda w, b: None)
    out['geese'] = {'net': 'geese', 'args': args, 'dims': (B, T, P, A), 'seeds': [80, 81, 82], 'state0': state0,
                    'steps': steps, 'lr': 1e-4, 'state3': state3}
    with open(os.path.join(HERE, 'net_step_cases.pkl'), 'wb') as f:
        pickle.dump(out, f)
    print('net step cases:', list(out))


def gen_generator_cases():
    """One TicTacToe episode as the reference's Generator.generate returns it (generation.py:20-93): what a worker
    ships, and what wire.install_worker_hook wraps."""
    env_args = {'env': 'TicTacToe'}
    prepare_env(env_args)
    env = make_env(env_args)
    torch.manual_seed(3)
    model = ModelWrapper(env.net())
    random.seed(3)
    args = {'gamma': 0.8, 'compress_steps': 4}
    ep = Generator(env, args).generate({p: model for p in env.players()}, {'player': env.players(), 'model_id': {}})
    with open(os.path.join(HERE, 'generator_cases.pkl'), 'wb') as f:
        pickle.dump({'tictactoe': {'args': args, 'episode': ep}}, f)
    print('generator cases: tictactoe, %d steps' % ep['steps'])


if __name__ == '__main__':
    os.chdir('/tmp')
    if len(sys.argv) > 1 and sys.argv[1] in ('nets', 'generator'):
        {'nets': gen_net_step_cases, 'generator': gen_generator_cases}[sys.argv[1]]()
        sys.exit(0)
    gen_loss_cases()
    gen_target_cases()
    gen_batch_cases()
    gen_step_cases()
    gen_rnn_cases()
    gen_net_step_cases()
    gen_generator_cases()
