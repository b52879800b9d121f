"""bench.py --dump-outputs: the poses after the last timed step land in DIR/ligand_pos.npy, two runs with the same arguments
agree (seeded inputs), and one more timed step moves the poses (the dump follows --steps).  Small complex, few steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu

POSES, ATOMS = 4, 12


def _bench(out_dir, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', str(steps), '--warmup', '3',
                          '--n-res', '120', '--n-atoms', str(ATOMS), '--poses', str(POSES), '--quick', '--no-cpu-baseline',
                          '--dump-outputs', str(out_dir)], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1, out.stdout[-2000:]
    assert json.loads(lines[0])['steps'] == steps
    assert sorted(os.listdir(out_dir)) == ['ligand_pos.npy']
    return np.load(os.path.join(out_dir, 'ligand_pos.npy'))


def test_dump_outputs_is_the_last_timed_step(built_lib, tmp_path):
    a = _bench(tmp_path / 'a', steps=2)
    b = _bench(tmp_path / 'b', steps=2)
    c = _bench(tmp_path / 'c', steps=3)
    assert a.dtype == np.float32 and a.shape == (POSES, ATOMS, 3) and np.isfinite(a).all()
    # the kernels accumulate with float atomics, so repeated runs agree to rounding, not bit for bit
    scale = float(np.abs(a).max())
    assert np.abs(a - b).max() <= 1e-4 * scale
    assert np.abs(c - a).max() > 1e-3 * scale
