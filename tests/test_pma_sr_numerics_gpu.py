"""GPU: PMA's update_sr eliminations against the extended-precision reference of tests/helpers.py, at every kernel
instantiation: the dense Gauss-Jordan / GTH of pma_sr_kernel<7> and <10>, the banded LU / row solve / GTH of
pma_band_factor_kernel and pma_band_solve_kernel for every half band 1..31, and every rung of the final refresh
pma_sr_band_kernel<BW>, BW in {4, 6, 8, 10, 12, 16, 24, 32}.

Each agent gets its own T (generators of tests/helpers.py: every band offset non-zero, entries spread over 1e-8..1)
and its own gamma; every batch covers gamma in {0, 0.5, 0.9, 0.99, 0.999}.

Gates (eps = fp64's unit round-off, R = the longdouble reference, kappa = kappa_inf(I - gamma T) from R):

* SR and every SR row the kernels solve for (the rows are entries of SR and share its gates):
    (1) max|X - R| <= 16 eps kappa max|R|.  Gauss-Jordan and LU without pivoting on a diagonally dominant matrix
        have a growth factor of at most 2 (Higham, Accuracy and Stability of Numerical Algorithms, Thm. 9.9 and
        ch. 14): the computed inverse is normwise within c eps kappa of the exact one with a small c.  16 covers c
        together with the S in ||R||_inf <= S max|R| that the entrywise form needs for the S of a gridworld row
        (at most 4 + 1 non-zeros) -- it does not cover a kernel that loses digits.
    (2) max|X - R| <= 32 max(max|X_lapack - R|, max|X_nopiv - R|, eps max|R|): the kernels may not be more than 32x
        (5 bits) less accurate than fp64 computations of the same inverse on the same input -- X_lapack =
        np.linalg.inv (LAPACK's partial-pivoting getrf / getri, what the reference's own PMAMemory uses) and X_nopiv =
        helpers.nopivot_inverse (the kernels' own elimination order, LU without pivoting and one triangular solve
        pair per column, run by NumPy).  X_nopiv is part of the baseline because of a measured finding: at gamma >=
        0.99 the unpivoted elimination is inherently up to ~65x less accurate than LAPACK's on these T (NumPy's fp64
        run of it shows 26..65x on the matrices where the B200 kernels showed 32..104x), while both stay 50x inside
        gate (1).  Against LAPACK alone, 10 of the ~1300 banded checks exceeded gate (2) by at most 3.3x.
* The stationary vector, elementwise: |x - r| / r <= 8 S eps.  GTH forms every quantity from non-negative numbers
  without a subtraction; an entry of x is reached through at most S elimination steps, each of which adds a few
  roundings of relative size eps (a product, an fma, the reciprocal of the row sum), so the relative error of every
  entry -- the ones of 1e-9 of a nearly decoupled chain included -- is a small multiple of S eps.
* Every COBEL_FLAG_* bit is 0 outside the singular cases.

Worst ratios error / gate seen on one B200 (1000 W power limit), printed by each test with -s:

    test                                   SR gate 1   SR gate 2   rows gate 1   rows gate 2   stationary
    dense, stand-alone (S = 1..160)        0.494       0.139       -             -             0.0495
    dense, inside train() (144, 160)       0.196       0.0346      -             -             0.00317
    band, fixed T (half bands 1..31)       0.113       0.733       0.0778        0.736         0.0461
    band, learned T (half bands 1..31)     0.0907      0.139       0.0289        0.137         0.0431
    band, 448 and 432 states               0.076       0.0522      0.0357        0.0394        0.00153

The dense gate-1 ratio grows about linearly with S (0.038 up to 17 states, 0.18 at 112, 0.49 at 160).
"""
import numpy as np
import pytest
import torch

from helpers import (EPS64, band_T, decoupled_T, dense_T, kappa_inf, nopivot_inverse, reducible_T, ref_inverse,
                     ref_stationary)

pytestmark = pytest.mark.gpu

GAMMAS = (0.0, 0.5, 0.9, 0.99, 0.999)
WORST = {}


def _note(key, value):
    WORST[key] = max(WORST.get(key, 0.0), value)


def sr_ratios(X, R, M, rows=None):
    """(error / gate 1, error / gate 2) of X against R = inv(M); `rows`: X holds only these rows of the inverse."""
    scale = float(np.abs(R).max())
    kappa = kappa_inf(M, R)
    M64 = np.asarray(M, dtype=np.float64)
    base = max(float(np.abs(np.linalg.inv(M64) - R).max()), float(np.abs(nopivot_inverse(M64) - R).max()))
    Rs = R if rows is None else R[rows]
    err = float(np.abs(np.asarray(X, dtype=np.longdouble) - Rs).max())
    return err / (16 * EPS64 * kappa * scale), err / (32 * max(base, EPS64 * scale))


def check_sr(X, R, M, what, rows=None, key='sr'):
    r1, r2 = sr_ratios(X, R, M, rows)
    _note(key + ' gate1', r1)
    _note(key + ' gate2', r2)
    assert r1 <= 1 and r2 <= 1, '%s: error / (16 eps kappa max|R|) = %.3g, error / (32 max(fp64 baseline error, eps max|R|)) = %.3g' % (
        what, r1, r2)


def check_stationary(x, T, what, key='need'):
    r = ref_stationary(T)
    S = T.shape[0]
    rel = np.abs(np.asarray(x, dtype=np.longdouble) - r) / r
    ratio = float(rel.max()) / (8 * S * EPS64)
    _note(key, ratio)
    assert ratio <= 1, '%s: worst relative error %.3g at state %d = %.3g of the gate 8 S eps (r = %.3g)' % (
        what, float(rel.max()), int(np.argmax(rel)), ratio, float(r[int(np.argmax(rel))]))


def report():
    return ', '.join('%s %.3g' % kv for kv in sorted(WORST.items()))


# ---- A. dense path, stand-alone: PMAMemory.update_sr() and compute_need(None) -----------------------------------
DENSE_S = [1, 2, 3, 7, 8, 15, 16, 17, 31, 32, 33, 63, 64, 65, 111, 112, 113, 127, 128, 129, 143, 144, 145, 159, 160]


def _dense_set(S, seed):
    """(name, T) per generator that makes sense at S states."""
    out = [('dense', dense_T(S, seed))]
    if S >= 2:
        out.append(('decoupled', decoupled_T(S, seed + 1)))
        out.append(('band', band_T(S, max(1, S // 8), seed + 2)))
    return out


@pytest.mark.parametrize('S', DENSE_S)
def test_dense_update_sr_and_stationary_stand_alone(S):
    """pma_sr_kernel<7> (S <= 112) and <10> (113..160) at every tile edge: SR = inv(I - gamma T) by the register-tiled
    Gauss-Jordan, and the dense GTH stationary vector of compute_need(None)."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.memory import PMAMemory
    from cobel_rl_b200.policy import EpsilonGreedy
    mats = _dense_set(S, 1000 + S)
    Ts = [T for _, T in mats for _ in GAMMAS]
    gam = [g for _ in mats for g in GAMMAS]
    names = ['%s gamma=%g' % (nm, g) for nm, _ in mats for g in GAMMAS]
    n = len(Ts)
    stream = cb.BatchStream(n, seed=S, device='cuda:0')
    succ = np.tile(np.arange(S)[:, None], (1, 4))
    mem = PMAMemory(succ, EpsilonGreedy(0.1, rng=stream), 0.9, 0.9, gam, 0.9, rng=stream)
    mem.T.copy_(torch.as_tensor(np.stack(Ts)))
    mem.update_sr()
    need = mem.compute_need(None).cpu().numpy()[:, :S]
    SR = mem.SR.cpu().numpy()
    for i in range(n):
        M = np.eye(S) - gam[i] * Ts[i]
        if gam[i] == 0.0:
            assert np.array_equal(SR[i], np.eye(S)), 'S=%d %s: gamma = 0 must give SR = I exactly' % (S, names[i])
        check_sr(SR[i], ref_inverse(M), M, 'S=%d %s' % (S, names[i]), key='dense sr')
        check_stationary(need[i], Ts[i], 'S=%d %s' % (S, names[i]), key='dense need')
    print('\n[dense S=%d] %s' % (S, report()))


# ---- shared set-up of the train() cases ---------------------------------------------------------------------------
def _world(h, w, goal, start):
    from cobel_rl_b200.misc import gridworld_tools as mg
    return mg.make_gridworld(h, w, terminals=[goal], rewards=np.array([[goal, 1.0]]), goals=[goal], starting_states=[start])


def _masks(h, w, goal, n_reach, n_out):
    """Per-agent action masks ([N, S, A]) that fix how a trial ends: the first n_reach agents can only step from the
    start state (the cell next to the goal) onto the goal, the other n_out agents only shuttle between the start
    state and the cell on its far side, so their trials time out.  Actions: 0 left, 1 up, 2 right, 3 down."""
    S = h * w
    toward, away = (1, 3) if goal < w else (3, 1)       # goal in the top row: the start is below it
    start = goal + w if goal < w else goal - w
    far = start + w if goal < w else start - w
    assert 0 <= far < S and far != goal
    m = np.ones((n_reach + n_out, S, 4), dtype=bool)
    m[:n_reach, start] = False
    m[:n_reach, start, toward] = True
    m[n_reach:, start] = False
    m[n_reach:, start, away] = True
    m[n_reach:, far] = False
    m[n_reach:, far, toward] = True
    return start, m


def _train(h, w, goal, Ts, gam, n_reach, sr_band_max, lr_T=0.0, trials=2, steps=4, seed=0, sr_init=None):
    """PMA.train() on an h x w gridworld with one start state next to `goal`, each agent's T written as given.
    Returns (agent, memory, result, start)."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import PMA
    from cobel_rl_b200.memory import PMAMemory
    from cobel_rl_b200.policy import EpsilonGreedy
    n = len(Ts)
    start, mask = _masks(h, w, goal, n_reach, n - n_reach)
    world = _world(h, w, goal, start)
    stream = cb.BatchStream(n, seed=seed, device='cuda:0')
    env = Gridworld(world, rng=stream)
    mem = PMAMemory(world['sas'], EpsilonGreedy(0.1, rng=stream), 0.9, 0.9, list(gam), 0.9, rng=stream)
    ag = PMA(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream), mem)
    ag.mask_actions = True
    ag.action_mask = torch.as_tensor(mask)
    mem.sr_band_max = sr_band_max
    mem.learning_rate_T = lr_T
    mem.T.copy_(torch.as_tensor(np.stack(Ts)))
    if sr_init is not None:
        mem.SR.copy_(torch.as_tensor(np.stack(sr_init).astype(np.float64)))
    res = ag.train(env, trials, steps, 8)
    torch.cuda.synchronize()
    assert int(res['flags'].sum()) == 0
    return ag, mem, res, start


# ---- B. dense path inside train() ----------------------------------------------------------------------------------
@pytest.mark.parametrize('h, w', [(12, 12), (10, 16)])
def test_dense_update_sr_inside_train(h, w):
    """sr_band_max = -1: pma_sr_kernel<10> runs after every trial of a 144- / 160-state world, with a fixed random dense
    T (learning_rate_T = 0 keeps T exactly as written).  Final SR of every agent; the dense GTH need of the agents
    whose last trial timed out."""
    S = h * w
    goal = S - 1
    gam = list(GAMMAS) * 2
    Ts = [dense_T(S, 7000 + i) for i in range(len(gam))]
    ag, mem, res, start = _train(h, w, goal, Ts, gam, n_reach=5, sr_band_max=-1)
    assert mem.sr_band(0)[0] == -1
    carry = mem._carry[:, 0].cpu().numpy()
    assert list(carry) == [goal] * 5 + [-1] * 5
    SR, need = mem.SR.cpu().numpy(), mem._need_scratch[0].cpu().numpy()
    for i, g in enumerate(gam):
        M = np.eye(S) - g * Ts[i]
        if g == 0.0:
            assert np.array_equal(SR[i], np.eye(S))
        check_sr(SR[i], ref_inverse(M), M, '%dx%d agent %d gamma=%g' % (h, w, i, g), key='dense train sr')
        if carry[i] < 0:
            check_stationary(need[i], Ts[i], '%dx%d agent %d' % (h, w, i), key='dense train need')
    print('\n[dense train %dx%d] %s' % (h, w, report()))


# ---- C. banded path inside train(), every half band ---------------------------------------------------------------
def _height(bw):
    return {1: 5, 2: 4}.get(bw, 3)       # the goal S-3 and the cell two rows above it must exist; 2 bw + 1 < S


def _band_case(h, bw, goal, seed, lr_T=0.0, shared=False):
    """`shared`: the reaching and the timed-out agent of a gamma share one T (halves the reference's work)."""
    S = h * bw
    gam = list(GAMMAS) * 2
    Ts = [band_T(S, bw, seed + i) for i in range(len(GAMMAS) if shared else len(gam))]
    Ms = [np.eye(S) - g * T for g, T in zip(gam, Ts)]
    Rs = [ref_inverse(M) for M in Ms]
    if shared:
        Ts, Ms, Rs = Ts * 2, Ms * 2, Rs * 2
    ag, mem, res, start = _train(h, bw, goal, Ts, gam, n_reach=5, sr_band_max=31, lr_T=lr_T, sr_init=Rs, seed=seed)
    return S, gam, Ts, Ms, Rs, ag, mem, start


@pytest.mark.parametrize('bw', range(1, 32))
def test_band_update_sr_inside_train(bw):
    """Half band bw on an h x bw gridworld with a fixed T whose every band offset is non-zero: band_lu, band_solve_row
    (rows 0, S-3, S-2, S-1 of the goals and the start row of the next trial), band_gth (timed-out trials) and the final
    refresh pma_sr_band_kernel<BW> of the narrowest rung BW >= bw, each against one reference."""
    h = _height(bw)
    S = h * bw
    assert 2 * bw + 1 < S
    for goal in (0, S - 1, S - 2, S - 3):
        S, gam, Ts, Ms, Rs, ag, mem, start = _band_case(h, bw, goal, 100 * bw + goal)
        assert mem.sr_band(bw)[0] == bw
        carry = mem._carry[:, 0].cpu().numpy()
        assert list(carry) == [goal] * 5 + [-1] * 5
        SR, need = mem.SR.cpu().numpy(), mem._need_scratch.cpu().numpy()
        for i, g in enumerate(gam):
            what = 'bw=%d goal=%d agent %d gamma=%g' % (bw, goal, i, g)
            if g == 0.0:
                assert np.array_equal(SR[i], np.eye(S)), what
                assert np.array_equal(need[1, i], np.eye(S)[start]), what
                if carry[i] >= 0:
                    assert np.array_equal(need[0, i], np.eye(S)[goal]), what
            check_sr(SR[i], Rs[i], Ms[i], what + ' SR', key='band sr')
            check_sr(need[1, i], Rs[i], Ms[i], what + ' row %d (start)' % start, rows=start, key='band row')
            if carry[i] >= 0:
                check_sr(need[0, i], Rs[i], Ms[i], what + ' row %d' % goal, rows=goal, key='band row')
            else:
                check_stationary(need[0, i], Ts[i], what, key='band need')
    print('\n[band bw=%d] %s' % (bw, report()))


@pytest.mark.parametrize('bw', range(1, 32))
def test_band_update_sr_learned_T(bw):
    """The same with the default learning_rate_T: T changes with every step, the final SR and the first need plane
    belong to the T the run leaves behind."""
    h = _height(bw)
    S = h * bw
    S, gam, Ts, Ms, Rs, ag, mem, start = _band_case(h, bw, S - 1, 5000 + bw, lr_T=0.9)
    T = mem.T.cpu().numpy()
    carry = mem._carry[:, 0].cpu().numpy()
    SR, need = mem.SR.cpu().numpy(), mem._need_scratch[0].cpu().numpy()
    assert not np.array_equal(T[0], Ts[0])
    for i, g in enumerate(gam):
        M = np.eye(S) - g * T[i]
        R = ref_inverse(M)
        what = 'learned bw=%d agent %d gamma=%g' % (bw, i, g)
        check_sr(SR[i], R, M, what, key='band learned sr')
        if carry[i] >= 0:
            check_sr(need[i], R, M, what + ' row %d' % carry[i], rows=int(carry[i]), key='band learned row')
        else:
            check_stationary(need[i], T[i], what, key='band learned need')
    print('\n[band learned bw=%d] %s' % (bw, report()))


@pytest.mark.parametrize('h, bw', [(28, 16), (18, 24)])
def test_band_update_sr_big_worlds(h, bw):
    """More than 160 states (pma_main_kernel<A, false, BIG>, no dense fallback): 448 states with the <16> refresh and
    432 with <24>.  (512 and 504 states at 4 actions exceed the main kernel's shared memory.)"""
    S = h * bw
    S, gam, Ts, Ms, Rs, ag, mem, start = _band_case(h, bw, S - 2, 9000 + bw, shared=True)
    carry = mem._carry[:, 0].cpu().numpy()
    assert list(carry) == [S - 2] * 5 + [-1] * 5
    SR, need = mem.SR.cpu().numpy(), mem._need_scratch.cpu().numpy()
    for i, g in enumerate(gam):
        what = '%dx%d agent %d gamma=%g' % (h, bw, i, g)
        check_sr(SR[i], Rs[i], Ms[i], what, key='big sr')
        check_sr(need[1, i], Rs[i], Ms[i], what + ' start row', rows=start, key='big row')
        if carry[i] >= 0:
            check_sr(need[0, i], Rs[i], Ms[i], what + ' goal row', rows=S - 2, key='big row')
        else:
            check_stationary(need[0, i], Ts[i], what, key='big need')
    print('\n[big %dx%d] %s' % (h, bw, report()))


def test_band_refresh_too_large_fails_before_running():
    """18 x 25 (450 states, half band 25): the final refresh would need pma_sr_band_kernel<32> with 450 * 66 doubles
    of shared memory, and 450 states have no dense update_sr.  train() raises before anything runs."""
    import cobel_rl_b200 as cb
    from cobel_rl_b200.interface import Gridworld
    from cobel_rl_b200.agent import PMA
    from cobel_rl_b200.memory import PMAMemory
    from cobel_rl_b200.policy import EpsilonGreedy
    h, w = 18, 25
    world = _world(h, w, h * w - 1, 0)
    stream = cb.BatchStream(2, seed=3, device='cuda:0')
    env = Gridworld(world, rng=stream)
    mem = PMAMemory(world['sas'], EpsilonGreedy(0.1, rng=stream), rng=stream)
    ag = PMA(env.observation_space, env.action_space, EpsilonGreedy(0.1, rng=stream), mem)
    mem.sr_band_max = 31
    assert mem.sr_band(env.transition_band)[0] == 25
    before = dict(Q=ag.Q.clone(), T=mem.T.clone(), dc=stream.draw_count.clone())
    with pytest.raises(NotImplementedError, match='half band 25'):
        ag.train(env, 2, 10, 4)
    torch.cuda.synchronize()
    assert torch.equal(ag.Q, before['Q']) and torch.equal(mem.T, before['T']) and torch.equal(stream.draw_count, before['dc'])


# ---- D. singular T ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('path', ['dense', 'band'])
def test_reducible_T_raises(path):
    """A T with two closed classes has no unique stationary distribution: a timed-out trial must raise CobelError
    (COBEL_FLAG_SINGULAR from the dense or the banded GTH), and so must the stand-alone compute_need(None)."""
    from cobel_rl_b200 import _lib
    if path == 'dense':
        h, w, bw = 12, 12, None
    else:
        h, w, bw = 6, 8, 8
    S = h * w
    Ts = [reducible_T(S, 40 + i, bw=bw) for i in range(len(GAMMAS))]
    with pytest.raises(_lib.CobelError, match='singular'):
        _train(h, w, S - 1, Ts, GAMMAS, n_reach=0, sr_band_max=-1 if bw is None else 31)
    import cobel_rl_b200 as cb
    from cobel_rl_b200.memory import PMAMemory
    from cobel_rl_b200.policy import EpsilonGreedy
    stream = cb.BatchStream(len(Ts), seed=1, device='cuda:0')
    mem = PMAMemory(np.tile(np.arange(S)[:, None], (1, 4)), EpsilonGreedy(0.1, rng=stream), 0.9, 0.9, list(GAMMAS), 0.9,
                    rng=stream)
    mem.T.copy_(torch.as_tensor(np.stack(Ts)))
    with pytest.raises(_lib.CobelError, match='singular'):
        mem.compute_need(None)
