"""End to end: the reference's Learner, worker processes and server loop on top of handyrl_b200's Trainer.

    python tests/e2e_reference_learner.py [--uniform-net] [--epochs N]

With HANDYRL_REFERENCE naming a checkout of the original HandyRL (it is NOT part of this repo), that project's own
Learner, workers and server run.  Without one, a stand-in `handyrl` package drives the Trainer through the same
protocol (see StandInLearner).  With a CUDA device it trains a TicTacToe net through the GPU learner; with
`--uniform-net` (no GPU needed) the net is replaced by a parameter-free model, which exercises everything around the
optimiser step: install(), Learner.feed_episodes -> Trainer.episodes, the trainer thread protocol, update()
hand-offs, pickling the returned model for the workers and the workers unpickling it.
Prints E2E_OK on success.
"""
import argparse
import copy
import os
import pickle
import sys
import tempfile
import threading

REF = os.environ.get('HANDYRL_REFERENCE')
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REF:
    sys.path.insert(0, REF)
sys.path.insert(0, ROOT)


import torch  # noqa: E402


class UniformNet(torch.nn.Module):
    """Parameter-free stand-in for the environment's net (module level: the Learner pickles it for the workers)."""

    def forward(self, x, hidden=None):
        return {'policy': torch.zeros(x.shape[0], 9), 'value': torch.zeros(x.shape[0], 1)}


def stand_in_worker(conn, wid):
    """A worker process of StandInLearner: fetch the pickled model, run it, ship TicTacToe episodes in the reference's
    wire format; ends when the learner closes the connection."""
    from handyrl_b200.synthetic import tictactoe_episodes
    rounds = 0
    try:
        while True:
            conn.send(('model', None))
            model = pickle.loads(conn.recv())
            with torch.no_grad():
                assert model(torch.zeros(2, 3, 3, 3))['policy'].shape == (2, 9)
            conn.send(('episode', tictactoe_episodes(10, seed=1000 * wid + rounds)))
            conn.recv()
            rounds += 1
    except (EOFError, OSError):
        pass


class StandInLearner:
    """What the reference Learner does with its Trainer (train.py:403-630), for where no checkout of it is at hand: the
    Trainer is built through the module attribute `Trainer(args, copy.deepcopy(self.model))`, its run() goes on a
    thread, the server loop hands the model pickled to worker processes and feeds the episodes they return into
    trainer.episodes (oldest dropped beyond maximum_episodes), and every update_episodes returned episodes after
    minimum_episodes it calls trainer.update() and saves models/<epoch>.pth, until `epochs` epochs are done."""

    def __init__(self, args, net=None):
        import handyrl.train as module
        self.args = args['train_args']
        self.model = net
        self.model_epoch = 0
        self.num_returned_episodes = 0
        self.trainer = module.Trainer(self.args, copy.deepcopy(self.model))

    def update(self):
        model, steps = self.trainer.update()
        print('updated model(%d)' % steps)
        self.model_epoch += 1
        self.model = model if model is not None else self.model
        os.makedirs('models', exist_ok=True)
        torch.save(self.model.state_dict(), os.path.join('models', '%d.pth' % self.model_epoch))

    def feed_episodes(self, episodes):
        self.num_returned_episodes += len(episodes)
        self.trainer.episodes.extend(episodes)
        while len(self.trainer.episodes) > self.args['maximum_episodes']:
            self.trainer.episodes.popleft()

    def run(self):
        import multiprocessing as mp
        from multiprocessing.connection import wait
        threading.Thread(target=self.trainer.run, daemon=True).start()
        ctx = mp.get_context('spawn')
        conns, procs = [], []
        for wid in range(self.args['worker']['num_parallel']):
            mine, theirs = ctx.Pipe()
            procs.append(ctx.Process(target=stand_in_worker, args=(theirs, wid), daemon=True))
            procs[-1].start()
            theirs.close()
            conns.append(mine)
        next_update = self.args['minimum_episodes'] + self.args['update_episodes']
        while self.model_epoch < self.args['epochs']:
            for conn in wait(conns):
                req, data = conn.recv()
                if req == 'model':
                    conn.send(pickle.dumps(self.model))
                else:
                    self.feed_episodes(data)
                    conn.send(None)
            if self.num_returned_episodes >= next_update:
                next_update += self.args['update_episodes']
                self.update()
        for conn in conns:
            conn.close()
        for p in procs:
            p.join(timeout=30)


def install_stand_in():
    """A stand-in `handyrl` package: the module attributes install() replaces, and StandInLearner."""
    import types
    train = types.ModuleType('handyrl.train')
    for k in ('Trainer', 'Batcher', 'make_batch', 'forward_prediction', 'compute_loss'):
        setattr(train, k, None)
    train.Learner = StandInLearner
    losses = types.ModuleType('handyrl.losses')
    losses.compute_target = None
    pkg = types.ModuleType('handyrl')
    pkg.train, pkg.losses = train, losses
    sys.modules.update({'handyrl': pkg, 'handyrl.train': train, 'handyrl.losses': losses})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--uniform-net', action='store_true')
    ap.add_argument('--epochs', type=int, default=2)
    opt = ap.parse_args()
    os.chdir(tempfile.mkdtemp(prefix='hrl_e2e_'))           # the Learner writes models/<epoch>.pth into the cwd
    if not REF:
        install_stand_in()

    import handyrl_b200.train as b200
    ref = b200.install()                                       # the three lines INTEGRATION.md adds to main.py
    assert ref.Trainer is b200.Trainer

    args = {
        'env_args': {'env': 'TicTacToe'},
        'train_args': {
            'turn_based_training': True, 'observation': False, 'gamma': 0.8, 'forward_steps': 8, 'burn_in_steps': 0,
            'compress_steps': 4, 'entropy_regularization': 0.1, 'entropy_regularization_decay': 0.1,
            'update_episodes': 40, 'batch_size': 16, 'minimum_episodes': 40, 'maximum_episodes': 500,
            'epochs': opt.epochs, 'num_batchers': 1, 'eval_rate': 0.1, 'worker': {'num_parallel': 2}, 'lambda': 0.7,
            'policy_target': 'UPGO', 'value_target': 'VTRACE', 'eval': {'opponent': ['random']}, 'seed': 0,
            'restart_epoch': 0,
        },
        'worker_args': {'server_address': '', 'num_parallel': 2},
    }
    if REF:
        if opt.uniform_net:
            import handyrl.envs.tictactoe as ttt
            ttt.Environment.net = lambda self: UniformNet()
        from handyrl.environment import prepare_env
        prepare_env(args['env_args'])
        learner = ref.Learner(args=args)
    else:
        from handyrl_b200.nets import tictactoe_net
        learner = ref.Learner(args=args, net=UniformNet() if opt.uniform_net else tictactoe_net())
    assert isinstance(learner.trainer, b200.Trainer)
    learner.run()
    assert learner.model_epoch >= opt.epochs, learner.model_epoch
    assert os.path.exists(os.path.join('models', '%d.pth' % opt.epochs))
    if not opt.uniform_net:
        assert learner.trainer.steps > 0
        first = torch.load(os.path.join('models', '1.pth'))
        last = torch.load(os.path.join('models', '%d.pth' % opt.epochs))
        assert any(not torch.equal(first[k], last[k]) for k in first)
    print('E2E_OK epochs=%d steps=%d episodes=%d' % (learner.model_epoch, learner.trainer.steps, learner.num_returned_episodes))
    os._exit(0)          # the reference's daemon threads / worker pipes have no shutdown path


if __name__ == '__main__':
    main()
