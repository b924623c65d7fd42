"""CPU: the product's world / graph builders produce exactly the reference's WorldDicts and node dictionaries (keys,
dtypes, values, neighbour order).  The comparison is with values recorded from this repository's builders, which matched
the reference when it was last run live; see the provenance note in tests/helpers.py.  With the reference sources
present its builders are called live as well."""
import numpy as np
import pytest

from cobel_rl_b200.misc import gridworld_tools as mg, topology_tools as mt
from cobel_rl_b200.memory.utils import metrics as mm
from helpers import check_stored, check_stored_record, world_form

WALLS = [(1, 2), (2, 1), (6, 7), (7, 6), (11, 12), (12, 11), (13, 8), (8, 13)]


def same_world(a, b):
    for k in b:
        x, y = a[k], b[k]
        if isinstance(y, np.ndarray):
            assert x.dtype == y.dtype and np.array_equal(x, y), k
        else:
            assert x == y, (k, x, y)


def check_builder(module, fn, *args, **kw):
    """``module.fn(*args, **kw)`` of the product against the same builder of the reference (``module`` names both)."""
    def live():
        import importlib
        from oracle import ref_loader
        ref_loader.load()
        return getattr(importlib.import_module('cobel.misc.' + module), fn)(*args, **kw)
    ours = getattr({'gridworld_tools': mg, 'topology_tools': mt}[module], fn)(*args, **kw)
    label = '%s.%s%r%s' % (module, fn, args, ('' if not kw else ' ' + repr(sorted(kw.items()))))
    if module == 'gridworld_tools':
        check_stored(label, world_form(ours), lambda: world_form(live()))
    else:
        check_stored(label, ours, live)
    return ours


def test_gridworld_builders():
    kw = dict(terminals=[4], rewards=np.array([[4, 10]]), goals=[4], starting_states=[12], invalid_transitions=WALLS)
    check_builder('gridworld_tools', 'make_gridworld', 5, 5, **kw)
    check_builder('gridworld_tools', 'make_open_field', 7, 4, 3, 2.5)
    check_builder('gridworld_tools', 'make_empty_field', 3, 6)
    cols = np.array([0, 0, 0, 1, 1, 1, 2, 2, 1, 0])
    check_builder('gridworld_tools', 'make_windy_gridworld', 7, 10, cols, 37, 1., 'up')
    check_builder('gridworld_tools', 'make_windy_gridworld', 7, 10, cols, 37, 1., 'down')
    check_builder('gridworld_tools', 'make_gridworld', 6, 6, invalid_states=[7, 8, 20])
    big = mg.make_open_field(100, 100, 0, 1, dense_sas=False)
    assert big['sas'] is None and big['succ'].shape == (10000, 4)


def test_maze_templates():
    # (world_form compares invalid_transitions as the sorted list of pairs: make_gridworld only tests membership)
    for stem in (1, 2, 3, 4):
        for arm in (1, 2, 3):
            for goal in ('left', 'right'):
                check_builder('gridworld_tools', 'make_t_maze', stem, arm, goal, 2.5)
            for goal in ('left-left', 'left-right', 'right-left', 'right-right'):
                check_builder('gridworld_tools', 'make_double_t_maze', stem, arm, goal)
                check_builder('gridworld_tools', 'make_two_sided_t_maze', stem, arm, goal)
    for ch in (1, 2, 3, 4, 5):
        for lw in (1, 2, 3):
            for goal in ('left', 'right'):
                check_builder('gridworld_tools', 'make_8_maze', ch, lw, goal, 3.0)
    for ch in (3, 4, 5, 6):
        for lw, arm in ((3, 1), (4, 1), (5, 2), (7, 2), (7, 3)):
            for chirality in ('left', 'right'):
                for goal in ('left', 'right'):
                    check_builder('gridworld_tools', 'make_two_choice_t_maze', ch, lw, arm, chirality, goal, 2.0)
    for ws, hs, dw, dh in ((1, 1, 1, 1), (2, 2, 2, 1), (1, 3, 4, 2), (3, 2, 1, 3)):
        check_builder('gridworld_tools', 'make_detour_maze', ws, hs, ws + dw, hs + dh, 2.0)
    for arm in (1, 2, 3, 4):
        for aw in (1, 2, 3):
            for goal in ('left', 'top', 'right', 'bottom'):
                check_builder('gridworld_tools', 'make_cross_maze', arm, aw, goal, 2.0)


def test_maze_templates_known_answers():
    """Runs everywhere (no reference needed): the T-maze of the reference's demo, drawn from the successor table."""
    w = mg.make_t_maze(3, 2)
    assert (w['height'], w['width']) == (4, 5) and list(w['starting_states']) == [17] and w['goals'] == [4]
    assert w['rewards'][4] == 1 and w['terminals'][4] == 1 and len(w['invalid_transitions']) == 20
    succ = w['succ']
    # stem: only up / down moves; arms: left / right along the top row, down only at the junction
    assert list(succ[17]) == [17, 12, 17, 17] and list(succ[12]) == [12, 7, 12, 17] and list(succ[7]) == [7, 2, 7, 12]
    assert list(succ[2]) == [1, 2, 3, 7] and list(succ[0]) == [0, 0, 1, 0] and list(succ[4]) == [3, 4, 4, 4]
    d = mg.make_double_t_maze(2, 1)
    assert (d['height'], d['width']) == (6, 7) and list(d['starting_states']) == [38] and d['goals'] == [6]
    assert len(d['invalid_transitions']) == 54
    t = mg.make_two_sided_t_maze(2, 2)
    assert (t['height'], t['width']) == (5, 4) and list(t['starting_states']) == [9] and t['goals'] == [19]
    assert len(t['invalid_transitions']) == 24
    e = mg.make_8_maze(3, 2)
    assert (e['height'], e['width']) == (5, 7) and list(e['starting_states']) == [4] and e['goals'] == [20]
    assert len(e['invalid_transitions']) == 40
    c = mg.make_two_choice_t_maze(3, 3, 1)
    assert (c['height'], c['width']) == (5, 9) and list(c['starting_states']) == [40] and c['goals'] == [26]
    assert len(c['invalid_transitions']) == 56
    d = mg.make_detour_maze(2, 2, 4, 3)
    assert (d['height'], d['width']) == (10, 9) and list(d['starting_states']) == [84] and d['goals'] == [3]
    assert len(d['invalid_transitions']) == 98
    x = mg.make_cross_maze(2, 2, 'left')
    assert x['height'] == x['width'] == 6 and list(x['starting_states']) == [14, 15, 20, 21] and list(x['goals']) == [12, 18]
    assert len(x['invalid_transitions']) == 32 and x['rewards'][12] == 1 and x['terminals'][18] == 1


def test_topology_builders():
    for args in [(10, 2, 1.0, 20., 'right'), (5, 1, 0.5, 1., 'left'), (4, 3)]:
        check_builder('topology_tools', 'linear_track', *args)
    for args in [(5,), ((3, 4),), (4, (0., 2.), 3., '5'), ((2, 5), ((0., 1.), (1., 3.)))]:
        check_builder('topology_tools', 'grid', *args)
    for args in [(4, 3, 1), (6, 3, 2), (2, 2, 3, 0.5, 2., 'left')]:
        check_builder('topology_tools', 't_maze', *args)
    for args in [(10,), (6,), (5, (0., 2.), 3., '7'), (2,), (9, (1.0, 4.0))]:
        check_builder('topology_tools', 'hexagonal', *args)
    for args in [(3, 1), (2, 2, 0.5, 30.0), (4, 3, 2.0, 90.0), (1, 1)]:
        check_builder('topology_tools', 'cross', *args)


def test_metrics():
    world = mg.make_gridworld(5, 5, terminals=[4], invalid_transitions=WALLS)

    def matrices(m):
        return {'DR_walls': m.DR(5, 5, world['sas'], 0.9, WALLS).D, 'DR_open': m.DR(5, 5, world['sas'], 0.9, []).D,
                'SR': m.SR(world['sas'], 0.8).D, 'Euclidean': m.Euclidean(4, 3).D}

    def live():
        from oracle import ref_loader
        return matrices(ref_loader.load().memory.utils.metrics)
    ours = matrices(mm)
    check_stored_record('metrics', ours, ['DR_walls', 'DR_open', 'SR'], live)
    check_stored_record('metrics_euclidean', ours, ['Euclidean'], live, rtol={'Euclidean': 1e-15})


def test_pickled_world_round_trip(tmp_path):
    """The gridworld editor's file format (misc/gridworld_gui.py:203-239: a pickled WorldDict)."""
    import pickle
    from cobel_rl_b200.interface.gridworld import successor_table
    ref_world = check_builder('gridworld_tools', 'make_t_maze', 3, 2)
    ref_world = {k: v for k, v in ref_world.items() if k != 'succ'}     # as the reference's editor saved it
    path = tmp_path / 'maze.pkl'
    with open(path, 'wb') as f:
        pickle.dump(ref_world, f)
    world = mg.load_world(path)
    same_world(world, ref_world)
    assert np.array_equal(world['succ'], mg.make_t_maze(3, 2)['succ']) and np.array_equal(successor_table(world), world['succ'])
    mg.save_world(world, tmp_path / 'again.pkl')
    again = mg.load_world(tmp_path / 'again.pkl')
    same_world(again, world)


def test_remove_obstructed_neighbors_known_answers():
    """misc/topology_tools.py:472-505 (the reference needs shapely, which this image does not have: the predicate
    is checked against hand-derived answers on a 5 x 5 grid graph)."""
    from cobel_rl_b200.misc import topology_tools as tt
    nodes, _ = tt.grid(5, (0.0, 4.0))
    wall = [[1.4, -0.5], [1.6, -0.5], [1.6, 2.5], [1.4, 2.5]]        # between the columns x = 1 and x = 2, rows y <= 2
    upd = tt.remove_obstructed_neighbors(nodes, [wall])
    cut = {(n, i) for n in nodes for i in range(4) if nodes[n]['neighbors'][i] != upd[n]['neighbors'][i]}
    by_pos = {nodes[n]['pose'][:2]: n for n in nodes}
    want = set()
    for y in (0.0, 1.0, 2.0):
        want |= {(by_pos[(1.0, y)], 2), (by_pos[(2.0, y)], 0)}          # right of x = 1, left of x = 2
    assert cut == want
    assert all(upd[n]['neighbors'][i] == n for n, i in cut)             # obstructed edges point back to the node
    assert nodes[by_pos[(1.0, 0.0)]]['neighbors'][2] == by_pos[(2.0, 0.0)]      # the input graph is not modified
    # the edge (1,3)-(2,3) passes the wall's top edge at distance 0.5: cut from buffer 0.5 on, not below
    e = (by_pos[(1.0, 3.0)], 2)
    assert tt.remove_obstructed_neighbors(nodes, [wall], 0.49)[e[0]]['neighbors'][2] == by_pos[(2.0, 3.0)]
    assert tt.remove_obstructed_neighbors(nodes, [wall], 0.5)[e[0]]['neighbors'][2] == e[0]
    # an edge that ends inside an obstacle, a shapely-like polygon object with a hole, and the assertion
    class Ring:
        def __init__(self, c): self.coords = c
    class Poly:
        exterior = Ring([(2.5, 2.5), (4.5, 2.5), (4.5, 4.5), (2.5, 4.5), (2.5, 2.5)])
        interiors = [Ring([(3.6, 3.6), (4.4, 3.6), (4.4, 4.4), (3.6, 4.4), (3.6, 3.6)])]
    upd = tt.remove_obstructed_neighbors(nodes, [Poly()])
    assert upd[by_pos[(2.0, 3.0)]]['neighbors'][2] == by_pos[(2.0, 3.0)]        # (2,3) -> (3,3) enters the polygon
    assert upd[by_pos[(3.0, 3.0)]]['neighbors'][1] == by_pos[(3.0, 3.0)]        # inside -> inside
    assert upd[by_pos[(0.0, 0.0)]]['neighbors'] == nodes[by_pos[(0.0, 0.0)]]['neighbors']
    with pytest.raises(AssertionError):
        tt.remove_obstructed_neighbors(nodes, [wall], -1.0)
