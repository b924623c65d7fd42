"""CPU: host logic of the batched grid-search back-end and the monitors (no GPU needed).  The comparisons with the
reference check against values recorded from this repository's code, which matched the reference when it was last run
live; see the provenance note in tests/helpers.py.  With the reference sources present the reference runs live too."""
import numpy as np
import pytest
import torch

from cobel_rl_b200.monitor import EscapeLatencyMonitor, RewardMonitor
from cobel_rl_b200.optimizer import EAOptimizer, GridSearchOptimizer
from helpers import check_stored


def _reference(module):
    import importlib
    from oracle import ref_loader
    ref_loader.load()
    return importlib.import_module('cobel.' + module)


def _f64(xs):
    """Arrays compared by value (np.array_equal), whatever their dtype."""
    return [np.asarray(x, dtype=np.float64) for x in xs]

PARAMS = {'x_1': [0, 1, 2, 3, 4], 'x_2': [0., 0.1, 0.2, 0.3, 0.4], 'x_3': np.array([0.9, 0.5, 0.6, 0.7, 0.8])}


@pytest.mark.parametrize('order', ['nested', 'systematic'])
def test_parameter_combinations_match_reference(order, tmp_path):
    def live():
        ref = _reference('optimizer').GridSearchOptimizer(str(tmp_path) + '/', PARAMS, 2, order,
                                                          rng=np.random.default_rng(4))
        return list(ref.parameter_combinations.items())
    ours = GridSearchOptimizer(str(tmp_path) + '/', PARAMS, 2, order, rng=np.random.default_rng(4))
    check_stored('GridSearchOptimizer.parameter_combinations %s' % order, list(ours.parameter_combinations.items()),
                    live)


def test_shuffled_order_is_a_permutation(tmp_path):
    # (the reference's 'shuffled' order raises AttributeError: it uses self.rng before assigning it,
    #  optimizer/grid_search.py:103 vs 107/161)
    nested = GridSearchOptimizer(str(tmp_path) + '/', PARAMS, 1, 'nested')
    shuffled = GridSearchOptimizer(str(tmp_path) + '/', PARAMS, 1, 'shuffled', rng=np.random.default_rng(4))
    assert set(shuffled.parameter_combinations) == set(nested.parameter_combinations)
    assert list(shuffled.parameter_combinations) != list(nested.parameter_combinations)


def test_batched_fit_equals_per_run_fit(tmp_path):
    """The doc example of the reference (grid_search.py:66-83): same fit dict as the sequential loop."""
    calls = []

    def sim_batch(task, params):
        calls.append(len(params['_run']))
        return params['x_1'] + params['x_2'] ** 2 + params['x_3'] ** 3 + 0.0 * params['_run']

    def loss(data_sim, data_exp):
        return sum((np.mean(data_sim[t]) - data_exp[t]) ** 2 for t in data_sim) / len(data_sim)

    data = {'task_1': 2 + 0.1 ** 2 + 0.7 ** 3}
    opt = GridSearchOptimizer(str(tmp_path) + '/', PARAMS, nb_runs=3)
    fit = opt.fit(sim_batch, {'task_1': {}}, data, loss, store_simulation_data=True)
    assert calls == [125 * 3]                               # one batched call: all combinations x runs
    assert len(fit) == 125 and min(fit, key=fit.get) == (2, 0.1, 0.7) and fit[(2, 0.1, 0.7)] < 1e-30
    for combo, f in fit.items():
        expect = (combo[0] + combo[1] ** 2 + combo[2] ** 3 - data['task_1']) ** 2
        assert f == pytest.approx(expect, rel=1e-12, abs=1e-30)
    # resume: a second optimizer on the same directory finds fit.pkl and runs nothing
    calls.clear()
    opt2 = GridSearchOptimizer(str(tmp_path) + '/', PARAMS, nb_runs=3)
    assert opt2.fit(sim_batch, {'task_1': {}}, data, loss) == fit and calls == []
    assert opt2.recompute_fit(data, loss, overwrite=True) == fit
    # chunked calls
    opt3 = GridSearchOptimizer(str(tmp_path) + '/', PARAMS, nb_runs=3, max_agents=60)
    fit3 = opt3.fit(sim_batch, {'task_1': {}}, data, loss, overwrite=True)
    assert fit3 == fit and max(calls) <= 60 and sum(calls) == 375


EA_TASKS = {'t1': {'x': 1.0}, 't2': {'x': -2.0}}
EA_DATA = {'t1': 0.3 * 1.0 + 0.5, 't2': 0.3 * -2.0 + 0.5}


def _ea_loss(sim, data):
    return float(sum((np.mean(sim[t]) - data[t]) ** 2 for t in sim))


def _ea_params(rng):
    return {'a': {'param_type': float, 'init_range': {'low': -1, 'high': 1}, 'mutator': (rng.normal, {'scale': 0.05})},
            'b': {'param_type': float, 'param_range': {'a_min': 0.0, 'a_max': 1.0}, 'mutator': (rng.normal, {'scale': 0.05})}}


def test_ea_optimizer_reference_constructor_cannot_run(reference, tmp_path):
    """optimizer/evolution.py:73-75: the default mutator is a set literal holding a dict."""
    from cobel.optimizer.evolution import EAOptimizer as Ref
    with pytest.raises(TypeError, match='unhashable'):
        Ref(str(tmp_path) + '/', _ea_params(np.random.default_rng(0)), 1, 1, np.random.default_rng(0))


def test_ea_optimizer_matches_reference_fit_method(tmp_path):
    """The reference's unmodified ``fit`` (on an object whose constructor is bypassed) against the batched back-end
    in ``bookkeeping='reference'`` mode: same run_<r>.pkl files, same returned fit, same rng consumption."""
    import os
    import pickle
    d_ref, d_our = str(tmp_path) + '/ref/', str(tmp_path) + '/our/'
    os.makedirs(d_ref); os.makedirs(d_our)

    def outcome(fit, d, rng):
        return fit, [pickle.load(open(d + 'run_%d.pkl' % r, 'rb')) for r in range(2)], rng.uniform()

    def live():
        import copy
        rng_ref = np.random.default_rng(11)
        ref = object.__new__(_reference('optimizer.evolution').EAOptimizer)
        ref.parameters = copy.deepcopy(_ea_params(rng_ref))      # evolution.py:65 (a bound mutator gets its own copy of the generator)
        for p in ref.parameters.values():               # what evolution.py:68-72 would have filled in
            p.setdefault('init_range', {'low': -1, 'high': 1})
            p.setdefault('param_range', {'a_min': None, 'a_max': None})
        ref.file_path, ref.nb_runs, ref.population_size, ref.rng, ref.present_files = d_ref, 2, 3, rng_ref, []
        f_ref = ref.fit(lambda task, ind: ind['a'] * task['x'] + ind['b'], EA_TASKS, EA_DATA, _ea_loss, generations=6,
                        individuals=5)
        return outcome(f_ref, d_ref, rng_ref)
    calls = []

    def sim_batch(task, params):
        calls.append(len(params['_run']))
        return params['a'] * task['x'] + params['b']
    rng_our = np.random.default_rng(11)
    ours = EAOptimizer(d_our, _ea_params(rng_our), 2, 3, rng_our, bookkeeping='reference')
    f_our = ours.fit(sim_batch, EA_TASKS, EA_DATA, _ea_loss, generations=6, individuals=5)
    assert len(f_our) >= 1
    assert calls == [5 * 3] * (2 * 6 * 2)            # one batched call per task and generation: individuals x repetitions
    # same fit, same run_<r>.pkl contents, same number of draws consumed (the next uniform)
    check_stored('EAOptimizer.fit reference bookkeeping', outcome(f_our, d_our, rng_our), live)


def test_ea_optimizer_intended_bookkeeping_converges_and_resumes(tmp_path):
    rng = np.random.default_rng(5)
    d = str(tmp_path) + '/'
    opt = EAOptimizer(d, _ea_params(rng), nb_runs=1, population_size=2, rng=rng)
    fit = opt.fit(lambda task, p: p['a'] * task['x'] + p['b'], EA_TASKS, EA_DATA, _ea_loss, generations=60, individuals=12)
    (a, b), f = next(iter(fit.items()))
    assert f < 1e-3 and abs(a - 0.3) < 0.05 and abs(b - 0.5) < 0.05 and 0.0 <= b <= 1.0
    import pickle
    hist = pickle.load(open(d + 'run_0.pkl', 'rb'))
    assert len(hist) == 60 and all(hist[i + 1][1] <= hist[i][1] for i in range(59))      # elitist: never worse
    # default mutator (the reference's is not constructible): rng.normal(value, 0.1); and resume from run_0.pkl
    opt2 = EAOptimizer(d, {'a': {'param_type': float}, 'b': {'param_type': float}}, rng=np.random.default_rng(1))
    assert opt2.parameters['a']['mutator'][1] == {'scale': 0.1}
    assert opt2.fit(None, EA_TASKS, EA_DATA, _ea_loss) == fit


def test_monitors_from_callbacks_and_results():
    el, rw = EscapeLatencyMonitor(4, 50, n_agents=3), RewardMonitor(4, n_agents=3)
    for t in range(4):
        logs = {'trial': t, 'steps': torch.tensor([t, 2 * t, 49]), 'trial_reward': torch.tensor([0.0, 1.0, t / 2])}
        el.update(logs); rw.update(logs)
    assert el.get_trace().tolist() == [[0, 1, 2, 3], [0, 2, 4, 6], [49] * 4]
    assert rw.get_trace()[2].tolist() == [0.0, 0.5, 1.0, 1.5]
    res = {'trial_steps': torch.arange(12).reshape(3, 4).int(), 'trial_reward': torch.ones(3, 4, dtype=torch.float64)}
    assert EscapeLatencyMonitor(4, 50, n_agents=3).from_result(res).get_trace()[1].tolist() == [4, 5, 6, 7]
    single = EscapeLatencyMonitor(2, 50)
    single.update({'trial': 1, 'steps': 7})
    assert single.get_trace().tolist() == [0, 7]


def test_response_and_q_monitors_match_reference():
    """monitor/behavior.py:212-301, 388-464: same traces as the reference's monitors fed the same logs."""
    import numpy as np
    from cobel_rl_b200.monitor import QMonitor, ResponseMonitor
    rewards = [0.0, 1.0, 0.0, 2.5, 0.0, 1.0]

    def feed(m):
        for t, r in enumerate(rewards):
            logs = {'trial': t, 'trial_reward': r}
            if t == 4:
                logs['response'] = 3
            m.update(dict(logs))
        return m

    def live_response():
        ref = feed(_reference('monitor.behavior').ResponseMonitor(6))
        return _f64([ref.get_trace(), ref.CRC])
    mine = feed(ResponseMonitor(6))
    check_stored('ResponseMonitor trace, cumulative', _f64([mine.get_trace(), mine.get_cumulative()]), live_response)

    class _Agent:
        def __init__(self):
            self.k = 0

        def predict_on_batch(self, batch):
            self.k += 1
            return np.arange(len(batch) * 4, dtype=float).reshape(len(batch), 4) * self.k
    def q_trace(m):
        a = _Agent()
        for t in range(3):
            m.update({'trial': t, 'agent': a})
        return _f64(m.get_trace())
    mine = q_trace(QMonitor(3, [0, 2, 5]))
    assert len(mine) == 3
    check_stored('QMonitor trace', mine, lambda: q_trace(_reference('monitor.behavior').QMonitor(3, [0, 2, 5])))
    # batched response monitor: one row per agent
    m = ResponseMonitor(3, n_agents=2)
    for t, r in enumerate(([0.0, 1.0], [2.0, 0.0], [0.0, 0.0])):
        m.update({'trial': t, 'trial_reward': np.array(r)})
    assert np.array_equal(m.get_trace(), [[0, 1, 0], [1, 0, 0]]) and np.array_equal(m.get_cumulative(), [[0, 1, 1], [1, 1, 1]])


def test_occupancy_map_and_match():
    """analysis/behavior_spatial.py:9-111 against the reference over random inputs, plus known answers."""
    import numpy as np
    import torch
    from cobel_rl_b200.analysis import get_occupancy_map, match
    rs = np.random.default_rng(0)
    for k in range(120):
        w, h = rs.uniform(1, 6, 2)
        b = rs.uniform(0.2, min(w, h))
        if k % 4 == 0:
            b, w, h = [0.5, 1.0, 0.25][k % 3], float(int(w) + 1), float(int(h) + 1)
        margins = ['expand', 'include', 'ignore'][k % 3]
        trajs = [np.round(rs.uniform(0, max(w, h) + 0.5, (int(rs.integers(1, 30)), 2)), 1 if k % 2 else 6) for _ in range(3)]
        live = lambda: _f64([_reference('analysis.behavior_spatial').get_occupancy_map(trajs, w, h, b, margins)])
        check_stored('get_occupancy_map %d' % k, _f64([get_occupancy_map(trajs, w, h, b, margins).numpy()]), live)
    for k in range(60):
        seq, tpl = rs.integers(0, 4, int(rs.integers(1, 20))), rs.integers(0, 4, int(rs.integers(1, 8)))
        check_stored('match %d' % k, _f64([match(seq, tpl)]),
                        lambda: _f64([_reference('analysis.behavior_spatial').match(seq, tpl)]))
    # a NaN-padded [N, T, 2] tensor gives the same map as the list of its valid rows
    pos = torch.tensor([[[0.5, 0.5], [1.5, 0.5], [float('nan')] * 2], [[0.5, 1.5], [0.5, 1.5], [1.5, 1.5]]], dtype=torch.float64)
    occ = get_occupancy_map(pos, 2.0, 2.0, 1.0)
    assert occ.tolist() == [[1.0, 2.0], [1.0, 1.0]]


def test_match_known_answers():
    import numpy as np
    from cobel_rl_b200.analysis import match
    assert match(np.array([1, 2, 3, 1, 2]), np.array([1, 2])).tolist() == [2, 0, 0, 2, 0]
    assert match(np.array([5]), np.array([5, 5, 5])).tolist() == [1]
