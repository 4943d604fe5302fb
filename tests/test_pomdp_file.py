"""
CPU tests of the Cassandra .POMDP reader / writer (pomdp_pbvi_exploration_b200.pomdp_file) against the tensors the
reference's own loader + Model constructor produced (tests/golden/model_*.npz), on a hand-written tiger specification,
on the reference's example files when a checkout of the reference is named by PBVI_REFERENCE_ROOT, and on round trips.
"""
import os

import numpy as np
import pytest

from conftest import load_golden
from pomdp_pbvi_exploration_b200.pomdp_file import load_POMDP_file, parse_POMDP, save_POMDP_file

# the example files ship with the reference (PimLb/POMDP_PBVI_Exploration), not with this repository
EXAMPLES = os.path.join(os.environ.get('PBVI_REFERENCE_ROOT', ''), 'Experiments', 'Example Models')
needs_examples = pytest.mark.skipif(not os.path.isabs(EXAMPLES) or not os.path.isdir(EXAMPLES),
                                    reason="needs the reference's example .POMDP files: set PBVI_REFERENCE_ROOT to a checkout of the reference")

TIGER = """
# tiger: listen / open-left / open-right; hearing accuracy 0.85
discount: 0.95
values: reward
states: tiger-left tiger-right
actions: listen open-left open-right
observations: tiger-left tiger-right

start:
0.5 0.5

T: listen
identity
T: open-left
uniform
T: open-right
uniform

O: listen
0.85 0.15
0.15 0.85
O: open-left
uniform
O: open-right
uniform

R: listen : * : * : * -1
R: open-left : tiger-left : * : * -100
R: open-left : tiger-right : * : * 10
R: open-right : tiger-left : * : * 10
R: open-right : tiger-right : * : * -100
"""


def _check_against_golden(model, tag):
    m = load_golden('model_' + tag)
    if 'transition_table' in m:                      # the dense S x A x S (x O) tables are only stored for models of up to 64 states
        assert np.array_equal(model.transition_table, m['transition_table'])
        assert np.array_equal(model.immediate_reward_table, m['reward_table'])
    assert np.array_equal(model.observation_table, m['obs_table'])
    assert np.array_equal(model.start_probabilities, m['start'])
    assert np.array_equal(model.reachable_states, m['reach'])
    assert np.array_equal(model.reachable_transitional_observation_table, m['rto'])
    assert np.array_equal(model.expected_rewards_table, m['rbar'])


def test_tiger_specification_matches_reference_tensors(tmp_path):
    path = tmp_path / 'tiger.POMDP'
    path.write_text(TIGER)
    model, solver = load_POMDP_file(str(path))
    assert solver.gamma == 0.95 and model.state_labels == ['tiger-left', 'tiger-right']
    _check_against_golden(model, 'tiger')


@needs_examples
@pytest.mark.parametrize('fname,tag', [('tiger.95.POMDP', 'tiger'), ('4x4.95.POMDP', 'grid4x4'), ('4x4.95-no_loop.POMDP', 'grid4x4_noloop'),
                                       ('tiger-grid.POMDP', 'tigergrid'), ('hallway.POMDP', 'hallway'), ('cheese.95.POMDP', 'cheese'),
                                       ('4x3.95.POMDP', 'grid4x3'), ('cit.POMDP', 'cit')])
def test_reference_example_files(fname, tag):
    model, solver = load_POMDP_file(os.path.join(EXAMPLES, fname))
    assert solver.gamma == pytest.approx(float(load_golden('model_' + tag)['gamma']))
    _check_against_golden(model, tag)


@needs_examples
def test_every_example_file_parses_to_stochastic_tables():
    """All 18 bundled files parse (the reference's reader rejects parr95, saci-s12-a6-z5 and shuttle), rows are distributions."""
    files = sorted(f for f in os.listdir(EXAMPLES) if f.endswith('.POMDP'))
    assert len(files) >= 15
    for f in files:
        spec = parse_POMDP(open(os.path.join(EXAMPLES, f)).read())
        np.testing.assert_allclose(spec['transitions'].sum(2), 1.0, atol=1e-4, err_msg=f)
        np.testing.assert_allclose(spec['observation_table'].sum(2), 1.0, atol=1e-4, err_msg=f)
        assert abs(spec["start"].sum() - 1.0) < 1e-4, f


# every model whose dense tables the reference's loader stored: the reader must give back exactly the reference's tensors
@pytest.mark.parametrize('tag', ['tiger', 'grid4x4', 'grid4x4_noloop', 'tigergrid', 'hallway', 'cheese', 'grid4x3', 'hanks', 'network',
                                 'maze4x5x2'])
def test_round_trip(tmp_path, tag):
    from pomdp_pbvi_exploration_b200 import Model
    m = load_golden('model_' + tag)
    S, A, O = m['rto'].shape[0], m['rto'].shape[1], m['rto'].shape[2]
    model = Model(states=S, actions=A, observations=O, transitions=m['transition_table'], rewards=m['reward_table'],
                  observation_table=m['obs_table'], start_probabilities=m['start'])
    path = str(tmp_path / 'm.POMDP')
    save_POMDP_file(model, path, float(m['gamma']))
    back, solver = load_POMDP_file(path)
    assert solver.gamma == float(m['gamma'])
    _check_against_golden(back, tag)


def test_grammar_corners():
    spec = parse_POMDP("""
discount: 0.9
values: cost
states: 3
actions: go stay
observations: 2
start include: 0 2
T: go : 0 : 1 1.0      # explicit entry
T: go : 1
0.0 0.5 0.5
T: go : 2   uniform
T: stay identity
O: * : * : 0 0.25
O: * : * : 1 0.75
O: stay : 2
1.0 0.0
R: go : 0 : * : * 2.5
R: stay : 1 : 1
1 2
R: go : 2
1 2
3 4
5 6
""")
    assert spec['states'] == ['s_0', 's_1', 's_2'] and spec['actions'] == ['go', 'stay']
    assert spec['start'].tolist() == [0.5, 0.0, 0.5]
    assert spec['transitions'][0, 0].tolist() == [0, 1, 0] and spec['transitions'][1, 0].tolist() == [0, 0.5, 0.5]
    assert np.allclose(spec['transitions'][2, 0], 1 / 3) and np.array_equal(spec['transitions'][:, 1, :], np.eye(3))
    assert spec['observation_table'][0, 0].tolist() == [0.25, 0.75] and spec['observation_table'][2, 1].tolist() == [1.0, 0.0]
    assert np.all(spec['rewards'][0, 0] == -2.5)                       # values: cost flips the sign
    assert spec['rewards'][1, 1, 1].tolist() == [-1, -2]
    assert spec['rewards'][2, 0].tolist() == [[-1, -2], [-3, -4], [-5, -6]]
    with pytest.raises(ValueError):
        parse_POMDP('discount: 0.9\nstates: 2\nactions: 1\nobservations: 1\nT: 0 : 0 : nowhere 1.0\n')
    with pytest.raises(ValueError):
        parse_POMDP('states: 2\nactions: 1\nobservations: 1\n')
