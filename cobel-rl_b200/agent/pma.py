"""PMA agent (reference: agent/pma.py:26-369): Dyna-Q whose replays are chosen by prioritized
memory access (gain x need) at the start and at the end of every trial.

``train()`` / ``test()`` run the whole loop for all N agents in one launch of ``cobel_pma_run``
(csrc/pma.cu).
"""
import numpy as np
import torch

from .. import _lib
from ..experience import Experience, ExperienceBatch  # noqa: F401
from ..spaces import Discrete
from .agent import Agent, launch_stream


class PMA(Agent):
    def __init__(self, observation_space, action_space, policy, memory, policy_test=None, learning_rate=0.9,
                 gamma=0.99, custom_callbacks=None):
        assert type(observation_space) is Discrete, 'PMA requires a discrete observation space!'
        assert type(action_space) is Discrete, 'PMA requires a discrete action space!'
        super().__init__(observation_space, action_space, custom_callbacks)
        self.policy = policy
        self.policy_test = policy if policy_test is None else policy_test
        self.learning_rate = learning_rate
        self.gamma = gamma
        self.M = memory
        self.mask_actions = False
        stream = self._find_stream(self.policy, self.policy_test, self.M, self.M.policy)
        if stream is not None:
            self._bind(stream)

    def _allocate(self, stream):
        S, A = int(self.observation_space.n), int(self.action_space.n)
        self._Q = torch.zeros((stream.n_agents, S, A), dtype=torch.float64, device=stream.device)
        self._action_mask = torch.ones((S, A), dtype=torch.bool, device=stream.device)
        self.M._allocate(stream)

    @property
    def Q(self):
        return self._view(self._Q)

    @Q.setter
    def Q(self, value):
        self._assign(self._Q, value)

    @property
    def action_mask(self):
        return self._action_mask

    @action_mask.setter
    def action_mask(self, value):
        self._action_mask = torch.as_tensor(value, device=self._stream.device).bool().contiguous()

    def _params(self, world, pol, tr, n_tr, steps, batch_size, no_replay, learn, band, bscratch, keep, agent_pow=False):
        """``CobelPMAParams`` of a call.  ``agent_pow``: the power table slot holds ``agent.gamma ** k`` (the stand-alone
        ``PMA.update_q``) instead of ``M.gamma_q ** k``."""
        st, M = self._stream, self.M
        A = self._Q.shape[2]
        par = {k: st.param(v, k) for k, v in dict(lr=self.learning_rate, gamma=self.gamma, mem_lr=M.learning_rate,
                                                  lr_q=M.learning_rate_q, gamma_q=M.gamma_q, gamma_sr=M.gamma).items()}
        psr, pq, pstride = M.power_tables(st, keep, q_gamma=self.gamma if agent_pow else None)
        mptr, mstride = self._mask_args(keep)
        n_tab, tkind, tpar, tof, tscr = M.policy_tables(st, pol, A, keep)
        keep.append(par)
        return _lib.PMAParams(
            st.n_agents, world, st.c_struct(), pol.c_struct(st, keep), M.policy.c_struct(st, keep), tr,
            self._Q.data_ptr(), M._rewards.data_ptr(), M._states.data_ptr(), M._terminals.data_ptr(),
            M._T.data_ptr(), M._SR.data_ptr(), M._update_mask.data_ptr(), mptr, mstride,
            par['lr'].data_ptr(), par['gamma'].data_ptr(), par['mem_lr'].data_ptr(), par['lr_q'].data_ptr(),
            par['gamma_q'].data_ptr(), par['gamma_sr'].data_ptr(), psr.data_ptr(), pq.data_ptr(), pstride,
            M._min_gap.data_ptr(), M._carry.data_ptr(), M._need_scratch.data_ptr(),
            float(M.learning_rate_T), float(M.min_gain),
            1 if M.min_gain_mode == 'original' else 0, n_tr, steps, batch_size, 1 if no_replay else 0,
            1 if learn else 0, band, M.options(), _lib.ptr(bscratch),
            n_tab, 0, _lib.ptr(tkind), _lib.ptr(tpar), _lib.ptr(tof), _lib.ptr(tscr))

    def _run(self, interface, trials, steps, batch_size, no_replay, learn):
        if self._stream is None:
            self._bind(interface.rng)
        st, M = self._stream, self.M
        assert interface.rng is st, 'environment and agent must share one BatchStream'
        M.check_supported()
        S, A = self._Q.shape[1], self._Q.shape[2]
        assert interface.n_states == S and interface.n_actions == A
        # the reference's PMA.test() also acts with `policy` (agent/pma.py:287)
        pol = self.policy
        results = []
        for t0, n_tr in self._chunks(trials):
            keep = []
            tr, res = self._make_trace(n_tr, steps, 0, 2 if (learn and not no_replay) else 0, batch_size, keep, td=learn)
            band, bscratch, trusted = M.sr_band(interface.transition_band) if (learn and not no_replay) else (-1, None, False)
            p = self._params(interface.c_world(), pol, tr, n_tr, steps, batch_size, no_replay, learn, band, bscratch, keep)
            p.band_trusted = 1 if trusted else 0
            _lib.call('cobel_pma_run', st.device, p, launch_stream(st))
            self._check_flags(res)                                 # incl. COBEL_FLAG_BAND_VIOLATION (one sync per launch)
            self._fire_trial_callbacks(res, self.current_trial, (1, 1) if (learn and not no_replay) else (0, 0), session_first=t0)
            self.current_trial += n_tr
            results.append(res)
        self.last_run = self._merge(results)
        return self.last_run

    def train(self, interface, trials, steps, batch_size=32, no_replay=False):
        """agent/pma.py:167-258 for all agents."""
        return self._run(interface, trials, steps, batch_size, no_replay, learn=True)

    def test(self, interface, trials, steps):
        """agent/pma.py:260-317 for all agents."""
        return self._run(interface, trials, steps, 0, True, learn=False)

    # ---- stand-alone methods -----------------------------------------------------------------------------------
    def _table_world(self):
        return _lib.World(self._Q.shape[1], self._Q.shape[2], 0, 0, None, None, None, None, None, None, None)

    def update_q(self, update):
        """agent/pma.py:319-353: ONE n-step update over the list of experiences (a one-element list inside the
        reference's step loop), with the agent's learning rate and ``agent.gamma ** k``."""
        st = self._stream
        if isinstance(update, dict):
            update = [update]
        batch = ExperienceBatch.from_dicts(st, update)
        self.M._check_experience(batch)
        keep = []
        p = self._params(self._table_world(), self.policy, _lib.Trace(), 0, 1, 0, False, True, -1, None, keep, agent_pow=True)
        e = batch.c_struct()
        _lib.call('cobel_pma_op', st.device, p, _lib.OP_UPDATE_Q, e, None, None, launch_stream(st))

    def replay(self, replay_length, current_state=None, update_sr=False):
        """The replay call of the reference's train loop (agent/pma.py:206-213, 248-256):
        ``updates, self.Q = M.replay(self.Q, mask, replay_length, current_state)``; returns the performed updates as a
        padded ``[N, L]`` tensor of flat indices ``a*S + s`` (-1 = none).  Same sizes and rules as ``PMAMemory.replay``
        (banded eliminations beyond 160 states or 1024 one-step backups)."""
        mask = self._action_mask if self.mask_actions else None
        updates, _ = self.M.replay(self, mask, replay_length, current_state, update_sr=update_sr)
        return updates

    def predict_on_batch(self, batch):
        idx = torch.as_tensor(np.array(batch).astype(int), device=self._Q.device).reshape(-1)
        out = self._Q[:, idx]
        return out[0].cpu().numpy() if self._stream.single else out
