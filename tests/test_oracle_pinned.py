"""Pins the oracle port (oracle/port.py) against the committed fixtures: the outputs of the unmodified reference on
the same seeded inputs (tests/golden/*.npz, oracle/make_golden.py). CPU only."""
import pytest

from conftest import load_golden
from oracle import cases

RTOL, ATOL = 2e-5, 2e-6  # fp32: port and reference run the same torch CPU ops; slack covers thread-count summation order


@pytest.mark.parametrize('name', list(cases.CASES))
def test_port_matches_golden(name):
  out = cases.run_port(name, cases.make_inputs(name))
  bad = cases.compare(load_golden(name), out, rtol=RTOL, atol=ATOL)
  assert not bad, '\n'.join(bad)


def test_replay_index_stream_is_reference_stream():
  """memory.py:51-56 draws one np.random.randint per index from the GLOBAL stream; the port must consume it identically."""
  import numpy as np
  g = load_golden('replay_ring')
  out = cases.run_port('replay_ring', cases.make_inputs('replay_ring'))
  assert np.array_equal(g['sample_step'], out['sample_step'])
  assert np.array_equal(g['meta'], out['meta'])
