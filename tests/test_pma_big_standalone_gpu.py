"""GPU: the stand-alone PMA replay beyond 160 states or 1024 one-step backups (csrc/pma.cu replay_only, BIG branch).

PMAMemory.replay / PMA.replay / compute_need(None) there take the banded eliminations of train(): the band LU and
pma_sr_band_kernel for update_sr, the banded GTH for the stationary need.  Covered: the reference's train loop written
by hand on a 20x20 world against the oracle and against the fused train(); single replay calls on prepared tables at
the size limits the main kernel's shared memory allows (512 states at 3 actions, 1800 backups at 8 actions, and a
world that is BIG by its backups only); the numerical gates of tests/test_pma_sr_numerics_gpu.py on BIG banded T; and
the errors, raised before any launch or reported by the kernels."""
import numpy as np
import pytest
import torch

from oracle import tabular as tb
from oracle.philox import LazyStream
from helpers import EPS64, band_T, kappa_inf, ref_inverse, ref_stationary, reducible_T, unpack_run

pytestmark = pytest.mark.gpu

RTOL = {'SR': 1e-12}
WALLS20 = [(5, 6), (6, 5), (25, 26), (26, 25), (45, 46), (46, 45), (208, 228), (228, 208), (209, 229), (229, 209)]


# ---- worlds as successor tables ------------------------------------------------------------------------------------
def grid(h, w):
    """4-neighbour grid, moves off the grid stay put: half band w."""
    S = h * w
    r, c = np.divmod(np.arange(S), w)
    moves = [(0, -1), (-1, 0), (0, 1), (1, 0)]
    return np.stack([np.where((0 <= r + dr) & (r + dr < h) & (0 <= c + dc) & (c + dc < w), (r + dr) * w + c + dc,
                              np.arange(S)) for dr, dc in moves], axis=1).astype(np.int32)


def king(h, w):
    """8-neighbour grid, moves off the grid stay put: half band w + 1."""
    S = h * w
    r, c = np.divmod(np.arange(S), w)
    moves = [(dr, dc) for dr in (-1, 0, 1) for dc in (-1, 0, 1) if dr or dc]
    return np.stack([np.where((0 <= r + dr) & (r + dr < h) & (0 <= c + dc) & (c + dc < w), (r + dr) * w + c + dc,
                              np.arange(S)) for dr, dc in moves], axis=1).astype(np.int32)


def snake(h, w):
    """h x w cells joined into one corridor row by row, alternating direction; actions: back, forward, down (stays in
    the bottom row).  Half band w.  Three actions keep 512 states inside the main kernel's shared memory (at four
    actions it holds at most 454)."""
    S = h * w
    order = np.array([r * w + (c if r % 2 == 0 else w - 1 - c) for r in range(h) for c in range(w)])
    pos = np.empty(S, dtype=np.int64)
    pos[order] = np.arange(S)
    back, fwd = order[np.maximum(pos - 1, 0)], order[np.minimum(pos + 1, S - 1)]
    down = np.where(np.arange(S) + w < S, np.arange(S) + w, np.arange(S))
    return np.stack([back, fwd, down], axis=1).astype(np.int32)


WORLDS = {'snake32x16': (lambda: snake(32, 16), 16),      # 512 states, 1536 backups: the state limit
          'king15x15': (lambda: king(15, 15), 16),        # 225 states, 1800 backups
          'king12x12': (lambda: king(12, 12), 13)}        # 144 states, 1152 backups: BIG by its backups only


def _memory(succ, n, seed, gammas, gamma_q=0.9):
    import cobel_rl_b200 as cb
    from cobel_rl_b200.agent import PMA
    from cobel_rl_b200.memory import PMAMemory
    from cobel_rl_b200.policy import EpsilonGreedy
    from cobel_rl_b200.spaces import Discrete
    S, A = succ.shape
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    mem = PMAMemory(succ, EpsilonGreedy(0.1, rng=stream), 0.9, 0.9, list(gammas), gamma_q, rng=stream)
    ag = PMA(Discrete(S), Discrete(A), EpsilonGreedy(0.1, rng=stream), mem)
    return stream, mem, ag


def _launches():
    from cobel_rl_b200 import _lib
    return _lib.lib().cobel_launch_count()


# ---- 1. the reference's train loop by hand on 20 x 20 ------------------------------------------------------------
def test_pma_20x20_hand_written_loop_matches_oracle_and_fused_train():
    """agent/pma.py:199-257 written over the stand-alone methods on the world of test_pma_20x20_large_state_space (400
    states, band 20), three single-agent streams with their own gamma_q: replay(start), the steps, then
    replay(last, update_sr=True) (last = None on a time-out).  Against the oracle: every integer sequence, the tables
    and the draws bit-equal, SR within RTOL.  Against the fused train() of the same agents: integer sequences, Q and SR
    bit-equal -- both end on the same band factors of the same final T, refreshed by the same kernel."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import PMA
    from cobel_rl_b200.memory import PMAMemory
    from cobel_rl_b200.misc import gridworld_tools as mg
    from cobel_rl_b200.policy import EpsilonGreedy
    world = mg.make_gridworld(20, 20, terminals=[19], rewards=np.array([[19, 10.0]]), goals=[19], starting_states=[210],
                              invalid_transitions=WALLS20)
    W = tb.compile_gridworld(world)
    seed, trials, steps, batch, gq = 1, 3, 300, 16, [0.9, 0.95, 0.99]
    vmask = tb.valid_move_mask(W['succ'])
    hand, ended, timed_out = [], 0, 0
    for i, g in enumerate(gq):
        stream = cb.BatchStream(None, seed=seed, device='cuda:0', agent_id_base=i)
        env = Gridworld(world, rng=stream)
        k0 = int(stream.draw_count[0])
        mem = PMAMemory(world['sas'], EpsilonGreedy(0.1, rng=stream), 0.9, 0.9, 0.9, g, rng=stream)
        pol = EpsilonGreedy(0.1, rng=stream)
        ag = PMA(env.observation_space, env.action_space, pol, mem)
        ag.mask_actions = True
        ag.action_mask = vmask
        mask = ag.action_mask
        got = {k: [] for k in ('states', 'actions', 'trial_steps', 'replay', 'replay_len')}

        def replay(cur, update_sr=False):
            upd, _ = mem.replay(ag, mask, batch, cur, update_sr=update_sr)
            u = upd.cpu().numpy()
            u = u[u >= 0]
            got['replay'].extend(u.tolist()); got['replay_len'].append(len(u))

        for _ in range(trials):
            state, _info = env.reset()
            replay(state)
            step, last = 0, None
            for step in range(steps):
                action = pol.select_action(ag.Q[state], mask[state])
                nxt, reward, end, _trunc, _info = env.step(action)
                exp = {'state': state, 'action': action, 'reward': reward, 'next_state': nxt, 'terminal': 1 - int(end)}
                ag.update_q([exp])
                mem.store(exp)
                got['states'].append(state); got['actions'].append(action)
                state = nxt
                if end:
                    last = nxt
                    break
            got['trial_steps'].append(step)
            ended += last is not None
            timed_out += last is None
            replay(last, update_sr=True)
        torch.cuda.synchronize()
        got = {k: np.array(v, dtype=np.int32) for k, v in got.items()}
        got.update(Q=ag.Q.cpu().numpy(), Mr=mem.rewards.cpu().numpy(), Ms=mem.states.cpu().numpy(),
                   Mt=mem.terminals.cpu().numpy(), T=mem.T.cpu().numpy(), SR=mem.SR.cpu().numpy(),
                   draws=int(stream.draw_count[0]))
        assert float(mem.min_gap) > 1e-9, 'agent %d: a near tie of utilities decided a replay' % i
        rng = tb.Draws(LazyStream(seed, i), k0)
        st = tb.pma_init(tb.t0_from_succ(W['succ']), 400, 4)
        st['action_mask'] = vmask
        rec = tb.pma_train(W, st, rng, trials, steps, batch, gamma_q=g, mask_actions=True).arrays()
        rec.update(Q=st['Q'], Mr=st['Mr'], Ms=st['Ms'], Mt=st['Mt'], T=st['T'], SR=st['SR'], draws=rng.k)
        for k in ('states', 'actions', 'trial_steps', 'replay', 'replay_len', 'Q', 'Mr', 'Ms', 'Mt', 'T', 'draws'):
            assert np.array_equal(got[k], rec[k]), 'agent %d: %s differs from the oracle' % (i, k)
        err = np.abs(got['SR'] - rec['SR']).max() / np.abs(rec['SR']).max()
        assert err <= RTOL['SR'], 'agent %d: SR norm-wise relative error %.3g' % (i, err)
        hand.append(got)
    assert ended >= 1 and timed_out >= 1, 'both need paths of the end replay must run'

    stream = cb.BatchStream(len(gq), seed=seed, device='cuda:0')
    env = Gridworld(world, rng=stream)
    mem = PMAMemory(world['sas'], EpsilonGreedy(0.1, rng=stream), 0.9, 0.9, 0.9, gq, rng=stream)
    ag = PMA(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream), mem)
    ag.mask_actions = True
    ag.action_mask = vmask
    ag.record = True
    res = ag.train(env, trials, steps, batch)
    torch.cuda.synchronize()
    assert int(res['flags'].sum()) == 0 and float(mem.min_gap.min()) > 1e-9
    for i in range(len(gq)):
        fused = unpack_run(res, i, 4, W['succ'], W['reward'])
        fused.update(Q=ag.Q[i].cpu().numpy(), SR=mem.SR[i].cpu().numpy())
        for k in ('states', 'actions', 'trial_steps', 'replay', 'replay_len', 'Q', 'SR'):
            assert np.array_equal(hand[i][k], fused[k]), 'agent %d: %s differs from the fused train()' % (i, k)


# ---- 2. single replay calls on prepared tables against the oracle -------------------------------------------------
def _replay_states(mem, ag, L, state, update_sr):
    """cobel_pma_replay with a raw per-agent state vector (-1 = None), as PMAMemory.replay calls it: a call with
    given and None states mixed across the agents."""
    from cobel_rl_b200 import _lib
    from cobel_rl_b200.stream import cuda_stream
    from cobel_rl_b200.memory.pma import _check_flags
    st = mem._alloc_for
    n, dev = st.n_agents, st.device
    keep = []
    idx = torch.full((n, max(L, 1)), -1, dtype=torch.int32, device=dev)
    ln = torch.zeros((n, 1), dtype=torch.int32, device=dev)
    cnt = torch.zeros((2, n), dtype=torch.int64, device=dev)
    flags = torch.zeros(n, dtype=torch.int32, device=dev)
    tr = _lib.Trace(None, None, cnt[0].data_ptr(), cnt[1].data_ptr(), None, 0, idx.data_ptr(), max(L, 1), ln.data_ptr(),
                    1, flags.data_ptr(), None)
    p = mem._mem_params(keep, ag, L, tr)          # the agent's action mask (ag.mask_actions) included
    mem._set_band(p)
    st32 = torch.as_tensor(state, dtype=torch.int32, device=dev).contiguous()
    _lib.call('cobel_pma_replay', dev, p, st32.data_ptr(), 1 if update_sr else 0, cuda_stream(dev))
    _check_flags(flags)
    return idx


@pytest.mark.parametrize('update_sr', [False, True])
@pytest.mark.parametrize('wname', list(WORLDS))
def test_replay_calls_vs_oracle(wname, update_sr, monkeypatch):
    """13 agents (the last CTA of the main kernel and of the band kernels is partial) with random Q, experience tables
    and banded T, one gamma each.  A sequence of replay calls -- states given, None, and mixed per agent through the C
    ABI, each with L in {0, 1, 12} -- against oracle.tabular.pma_memory_replay: performed indices, Q and the draws bit
    for bit.  update_sr=False leaves SR bit-unchanged; update_sr=True refreshes it, and compute_need(s) then returns
    exactly the SR rows the next replay reads."""
    make, bw = WORLDS[wname]
    succ = make()
    S, A = succ.shape
    n, seed = 13, 4000 + S
    rs = np.random.default_rng(seed)
    gam = [0.5, 0.8, 0.9, 0.95, 0.99] * 3
    gam = gam[:n]
    stream, mem, ag = _memory(succ, n, seed, gam)
    assert mem.sr_band(bw)[0] == bw
    vmask = tb.valid_move_mask(succ)
    Ts = [band_T(S, bw, seed + i) for i in range(n)]
    SRs = [np.linalg.inv(np.eye(S) - g * T) for g, T in zip(gam, Ts)]
    Q = rs.normal(size=(n, S, A))
    Mr = np.where(rs.random((n, S, A)) < 0.3, rs.normal(size=(n, S, A)), 0.0)
    Mt = (rs.random((n, S, A)) < 0.9).astype(np.int32)
    ag.Q.copy_(torch.as_tensor(Q))
    mem.rewards.copy_(torch.as_tensor(Mr))
    mem.states.copy_(torch.as_tensor(np.broadcast_to(succ, (n, S, A)).copy()))
    mem.terminals.copy_(torch.as_tensor(Mt))
    mem.T.copy_(torch.as_tensor(np.stack(Ts)))
    mem.SR.copy_(torch.as_tensor(np.stack(SRs)))
    ag.mask_actions = True
    ag.action_mask = vmask
    sts, rngs = [], []
    for i in range(n):
        st = tb.pma_init(np.eye(S), S, A)                    # update_mask of the initial tables, as the memory's
        st.update(Q=Q[i].copy(), Mr=Mr[i].copy(), Ms=succ.copy(), Mt=Mt[i].copy(), T=Ts[i], SR=SRs[i], action_mask=vmask)
        sts.append(st)
        rngs.append(tb.Draws(LazyStream(seed, i), int(stream.draw_count[i])))
    # the oracle's need(None) is an eigen-decomposition per replay iteration; T does not change here, so compute it once
    need, cache = tb.pma_need, {}

    def cached_need(st, cur):
        if cur is not None:
            return need(st, cur)
        if id(st['T']) not in cache:
            cache[id(st['T'])] = need(st, None)
        return cache[id(st['T'])].copy()
    monkeypatch.setattr(tb, 'pma_need', cached_need)
    ran_none = ran_given = 0
    for kind in ('given', 'none', 'mixed'):
        for L in (0, 1, 12):
            given = rs.integers(0, S, n)
            cur = {'given': given, 'none': np.full(n, -1), 'mixed': np.where(np.arange(n) % 2 == 0, given, -1)}[kind]
            sr_before = mem.SR.clone()
            if kind == 'given':
                idx = mem.replay(ag, vmask, L, torch.as_tensor(given), update_sr=update_sr)[0]
            elif kind == 'none':
                idx = ag.replay(L, None, update_sr=update_sr)
            else:
                idx = _replay_states(mem, ag, L, cur, update_sr)
            torch.cuda.synchronize()
            idx = idx.cpu().numpy()
            what = '%s update_sr=%d %s L=%d' % (wname, update_sr, kind, L)
            if update_sr:
                SR = mem.SR.cpu().numpy()
                for i in range(n):
                    sts[i]['SR'] = np.linalg.inv(np.eye(S) - gam[i] * Ts[i])
                    err = np.abs(SR[i] - sts[i]['SR']).max() / np.abs(sts[i]['SR']).max()
                    assert err <= RTOL['SR'], '%s agent %d: SR error %.3g' % (what, i, err)
                rows = mem.compute_need(torch.as_tensor(given)).cpu().numpy()
                assert np.array_equal(rows, np.tile(SR[np.arange(n), given], (1, A))), what
            else:
                assert torch.equal(mem.SR, sr_before), what + ': SR changed'
            Qg = ag.Q.cpu().numpy()
            for i in range(n):
                c = None if cur[i] < 0 else int(cur[i])
                ran_none += c is None and L > 0
                ran_given += c is not None and L > 0
                perf, sts[i]['Q'] = tb.pma_memory_replay(sts[i], sts[i]['Q'], vmask, L, c, rngs[i], gamma_sr=gam[i])
                got = idx[i][idx[i] >= 0]
                assert got.tolist() == list(perf), '%s agent %d: replayed %s, oracle %s' % (what, i, got.tolist(), perf)
                assert np.array_equal(Qg[i], sts[i]['Q']), '%s agent %d: Q differs' % (what, i)
                assert int(stream.draw_count[i]) == rngs[i].k, '%s agent %d: draws' % (what, i)
    assert ran_none and ran_given
    assert float(mem.min_gap.min()) > 1e-9


# ---- 3. numerics on BIG banded T -------------------------------------------------------------------------------------
@pytest.mark.parametrize('wname, make, bw', [('grid20x20', lambda: grid(20, 20), 20), ('king15x15', lambda: king(15, 15), 16)])
def test_big_stationary_and_refresh_numerics(wname, make, bw):
    """compute_need(None) within 8 S eps of the extended-precision stationary vector, entry by entry, and SR after
    replay(..., update_sr=True) within 16 eps kappa_inf max|R| (the gates of tests/test_pma_sr_numerics_gpu.py)."""
    succ = make()
    S, A = succ.shape
    gam = [0.5, 0.9, 0.99] * 2
    n = len(gam)
    stream, mem, ag = _memory(succ, n, 77 + S, gam)
    Ts = [band_T(S, bw, 300 + i) for i in range(n)]
    mem.T.copy_(torch.as_tensor(np.stack(Ts)))
    need = mem.compute_need(None).cpu().numpy()
    state = torch.arange(n) * 37 % S
    ag.replay(0, state, update_sr=True)
    SR = mem.SR.cpu().numpy()
    worst_need = worst_sr = 0.0
    for i, g in enumerate(gam):
        assert np.array_equal(need[i], np.tile(need[i][:S], A))
        r = ref_stationary(Ts[i])
        rel = float((np.abs(np.asarray(need[i][:S], dtype=np.longdouble) - r) / r).max())
        worst_need = max(worst_need, rel / (8 * S * EPS64))
        M = np.eye(S) - g * Ts[i]
        R = ref_inverse(M)
        err = float(np.abs(np.asarray(SR[i], dtype=np.longdouble) - R).max())
        worst_sr = max(worst_sr, err / (16 * EPS64 * kappa_inf(M, R) * float(np.abs(R).max())))
    print('\n[%s] stationary %.3g of the gate, SR %.3g of the gate' % (wname, worst_need, worst_sr))
    assert worst_need <= 1 and worst_sr <= 1


# ---- 4. errors raised before any launch ------------------------------------------------------------------------------
def _snapshot(mem, ag, stream):
    return [t.clone() for t in (ag.Q, mem.rewards, mem.states, mem.terminals, mem.T, mem.SR, stream.draw_count)]


def _unchanged(before, mem, ag, stream):
    return all(torch.equal(a, b) for a, b in zip(before, _snapshot(mem, ag, stream)))


def _all_calls(mem, ag):
    return [lambda: ag.replay(8, 3), lambda: ag.replay(8, 3, update_sr=True), lambda: ag.replay(8, None),
            lambda: ag.replay(8, None, update_sr=True), lambda: mem.replay(ag, None, 8, 3), lambda: mem.compute_need(None)]


def test_unbanded_big_T_raises_before_any_launch():
    """A BIG T written outside the band through mem.T, or sr_band_max = -1: every row of the table of the stand-alone
    replay and compute_need(None) raise NotImplementedError, nothing is launched and nothing changes."""
    succ = grid(20, 20)
    stream, mem, ag = _memory(succ, 3, 11, [0.9] * 3)
    mem.T[0, 0, 399] = 0.25                               # far outside the band of 20
    for case in ('T outside the band', 'sr_band_max = -1'):
        if case == 'sr_band_max = -1':
            mem.T[0, 0, 399] = 0.0
            mem.sr_band_max = -1
        before, n0 = _snapshot(mem, ag, stream), _launches()
        for call in _all_calls(mem, ag):
            with pytest.raises(NotImplementedError, match='banded update_sr'):
                call()
        torch.cuda.synchronize()
        assert _launches() == n0, case
        assert _unchanged(before, mem, ag, stream), case


def test_bad_states_and_too_large_worlds_raise_before_any_launch():
    """A state of -2 or S raises IndexError; 23 x 23 (529 states) stays beyond the kernels."""
    from cobel_rl_b200.misc.gridworld_tools import make_open_field
    succ = grid(20, 20)
    stream, mem, ag = _memory(succ, 2, 12, [0.9] * 2)
    before, n0 = _snapshot(mem, ag, stream), _launches()
    for bad in (-2, 400, torch.tensor([3, 400])):
        with pytest.raises(IndexError):
            ag.replay(8, bad)
        with pytest.raises(IndexError):
            mem.replay(ag, None, 8, bad, update_sr=True)
        with pytest.raises(IndexError):
            mem.compute_need(bad)
    world = make_open_field(23, 23, 0, 1)
    stream2, mem2, ag2 = _memory(np.argmax(world['sas'], axis=2).astype(np.int32), 2, 13, [0.9] * 2)
    torch.cuda.synchronize()
    assert _launches() == n0
    for call in _all_calls(mem2, ag2):
        with pytest.raises(NotImplementedError, match='at most 512 states'):
            call()
    torch.cuda.synchronize()
    assert _launches() == n0
    assert _unchanged(before, mem, ag, stream)


# ---- 5. errors the kernels report ---------------------------------------------------------------------------------------
def test_lying_band_is_reported():
    """A caller that promises a narrower band than T has (as in test_pma_band_violation_is_reported) gets CobelError
    from pma_band_check_kernel, with or without update_sr."""
    from cobel_rl_b200 import _lib
    succ = grid(20, 20)
    stream, mem, ag = _memory(succ, 3, 14, [0.9] * 3)
    real = mem.sr_band
    mem.sr_band = lambda wb: (3, real(wb)[1], False)
    for call in (lambda: ag.replay(8, 5), lambda: ag.replay(8, None, update_sr=True), lambda: mem.compute_need(None)):
        with pytest.raises(_lib.CobelError, match='band'):
            call()


def test_reducible_big_T_raises():
    """Two closed classes: no unique stationary distribution, so the banded GTH of replay(None) and compute_need(None)
    raises CobelError."""
    from cobel_rl_b200 import _lib
    succ = grid(20, 20)
    stream, mem, ag = _memory(succ, 3, 15, [0.9] * 3)
    mem.T.copy_(torch.as_tensor(np.stack([reducible_T(400, 50 + i, bw=20) for i in range(3)])))
    with pytest.raises(_lib.CobelError, match='singular'):
        mem.compute_need(None)
    with pytest.raises(_lib.CobelError, match='singular'):
        ag.replay(8, None)
    with pytest.raises(_lib.CobelError, match='singular'):
        ag.replay(8, None, update_sr=True)
