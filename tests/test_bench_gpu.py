"""bench.py on the GPU: --steps sets the timed steps, --dump-outputs writes the last timed step's results."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_steps_losses_and_state(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--quick', '--steps', '7', '--warmup', '3',
                          '--dump-outputs', str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])
    assert line['steps'] == 7
    files = sorted(os.listdir(tmp_path))
    assert 'losses.npy' in files and any(f.startswith('state.') for f in files)
    arrays = {f: np.load(os.path.join(tmp_path, f)) for f in files}
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    losses = arrays['losses.npy']
    assert losses.shape == (6,) and losses[5] > 0              # (p, v, r, ent, total, dcnt): the step saw data
