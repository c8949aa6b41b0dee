"""install() swaps the learner hot path into an importable `handyrl`; the Trainer mirrors what the reference Learner touches."""
import os
import sys

import pytest

REF = os.environ.get('HANDYRL_REFERENCE')      # optional: a checkout of the original HandyRL


def test_install_swaps_reference_symbols(monkeypatch):
    """install() rebinds the learner hot path in the module namespaces of an importable `handyrl` (stand-in modules that
    carry the names it replaces).  The reference Learner builds its trainer through the module attribute (train.py:439),
    which is what makes the rebinding reach it; that is checked too where a checkout of the reference is given."""
    import types
    import handyrl_b200.train as b200
    from handyrl_b200 import ops
    ref_train = types.ModuleType('handyrl.train')
    for k in ('Trainer', 'Batcher', 'make_batch', 'forward_prediction', 'compute_loss'):
        setattr(ref_train, k, object())
    ref_losses = types.ModuleType('handyrl.losses')
    ref_losses.compute_target = object()
    pkg = types.ModuleType('handyrl')
    pkg.train, pkg.losses = ref_train, ref_losses
    for m in (pkg, ref_train, ref_losses):
        monkeypatch.setitem(sys.modules, m.__name__, m)
    assert b200.install() is ref_train
    assert ref_train.Trainer is b200.Trainer and ref_train.Batcher is b200.Batcher
    assert ref_train.make_batch is b200.make_batch and ref_train.compute_loss is b200.compute_loss
    assert ref_train.forward_prediction is b200.forward_prediction
    assert ref_losses.compute_target is ops.compute_target
    if REF:
        assert 'Trainer(args, copy.deepcopy(self.model))' in open(os.path.join(REF, 'handyrl', 'train.py')).read()


def test_trainer_constructor_mirrors_reference_attributes():
    """Attributes the reference Learner touches on its Trainer (train.py:439, 472, 482-483, 533)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip('covered by the GPU suite')
    from handyrl_b200.train import Trainer

    class NoParams(torch.nn.Module):
        def forward(self, x, h=None):
            return {'policy': x}

    args = {'batch_size': 4, 'forward_steps': 8, 'burn_in_steps': 0, 'num_batchers': 1, 'maximum_episodes': 10}
    tr = Trainer(args, NoParams())          # non-parametric model: allowed without a GPU (train.py:348-350)
    assert len(tr.episodes) == 0 and tr.steps == 0 and hasattr(tr, 'update') and hasattr(tr, 'run')
    tr.episodes.append({'steps': 3})
    tr.episodes.extend([{'steps': 4}])
    assert len(tr.episodes) == 2 and tr.episodes.popleft()['steps'] == 3
    assert tr.train() is tr.model            # sleeps 0.1 s and hands the model back


def test_reference_learner_and_workers_run_on_the_installed_trainer():
    """A Learner + worker processes + server loop for two epochs after install() (parameter-free net: runs without a GPU;
    everything around the optimiser step is the production code path): the reference's own where HANDYRL_REFERENCE names
    a checkout of it, otherwise a stand-in that drives the Trainer through the same protocol.  With a GPU, run
    `python tests/e2e_reference_learner.py` without --uniform-net for the full thing."""
    import subprocess
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'e2e_reference_learner.py')
    res = subprocess.run([sys.executable, script, '--uniform-net', '--epochs', '2'], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and 'E2E_OK epochs=2' in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]
    assert 'updated model' in res.stdout and 'started training' not in res.stdout.split('E2E_OK')[1]


def test_state_store_round_trip_and_cached_pickle():
    """f-4 pieces that need no GPU: every state_dict entry lives in ONE buffer and is rebuilt from a byte copy; the model
    handed to the Learner pickles as a memcpy of cached bytes and unpickles to the plain module class."""
    import copy
    import pickle
    import torch
    from handyrl_b200 import nets
    from handyrl_b200.train import StateStore, attach_pickle_cache
    torch.manual_seed(0)
    net = nets.tictactoe_net()
    net.train()
    net(torch.rand(8, 3, 3, 3))                       # move the BatchNorm statistics off their initial values
    want = {k: v.clone() for k, v in net.state_dict().items()}
    st = StateStore(net, 'cpu')
    flat = st.flat_param
    off = 0
    with torch.no_grad():
        for p in net.parameters():                    # what FlatAdam does with param_storage
            flat[off:off + p.numel()].copy_(p.reshape(-1))
            p.data = flat[off:off + p.numel()].view_as(p)
            off += p.numel()
    st.index_params(net)
    got = st.state_dict_from(st.bytes.clone(), want.keys())
    assert list(got) == list(want)
    for k in want:
        assert got[k].dtype == want[k].dtype and torch.equal(got[k], want[k]), k
    net.train()
    net(torch.rand(8, 3, 3, 3))                       # buffers are views of the store: updates land in it
    again = st.state_dict_from(st.bytes.clone(), want.keys())
    assert torch.equal(again['tower.0.1.running_mean'], net.state_dict()['tower.0.1.running_mean'])
    assert not torch.equal(again['tower.0.1.running_mean'], want['tower.0.1.running_mean'])
    assert int(again['tower.0.1.num_batches_tracked']) == 2

    tpl = nets.tictactoe_net()
    tpl.load_state_dict(again)
    tpl.eval()
    blob = pickle.dumps(tpl)
    model = attach_pickle_cache(pickle.loads(blob), blob)
    wire = pickle.dumps(model)                        # what Learner.server does per worker request (train.py:615)
    assert len(wire) < len(blob) + 200                # a wrapper around the cached bytes, not a second walk
    back = pickle.loads(wire)
    assert type(back) is nets.BoardNet and '__reduce_ex__' not in vars(back) and not back.training
    for k, v in back.state_dict().items():
        assert torch.equal(v, again[k])
    clone = copy.deepcopy(model)                      # Learner.server deep-copies the model for old model ids (:609)
    assert type(clone) is nets.BoardNet and torch.equal(clone.state_dict()['stem.weight'], again['stem.weight'])
    assert torch.equal(model(torch.ones(2, 3, 3, 3))['policy'], back(torch.ones(2, 3, 3, 3))['policy'])
