"""Dyna-Q agent (reference: agent/dyna_q.py:17-330).

``train()`` / ``test()`` run the reference's whole trial x step loop -- action
selection, environment step, memory store, online TD update and the replay of
``batch_size`` uniformly drawn experiences after every step -- for all N agents
in one launch of ``cobel_dynaq_run`` (csrc/dynaq.cu).
"""
import numpy as np
import torch

from .. import _lib
from ..experience import Experience, ExperienceBatch  # noqa: F401
from ..memory.dyna_q import DynaQMemory
from ..spaces import Discrete
from .agent import Agent, launch_stream


class DynaQ(Agent):
    def __init__(self, observation_space, action_space, policy, policy_test=None, learning_rate=0.99,
                 gamma=0.99, memory=None, custom_callbacks=None):
        assert type(observation_space) is Discrete, 'DynaQ requires a discrete observation space!'
        assert type(action_space) is Discrete, 'DynaQ requires a discrete action space!'
        super().__init__(observation_space, action_space, custom_callbacks)
        self.policy = policy
        self.policy_test = policy if policy_test is None else policy_test
        self.learning_rate = learning_rate
        self.gamma = gamma
        S, A = int(observation_space.n), int(action_space.n)
        self.M = DynaQMemory(S, A) if memory is None else memory
        self.mask_actions = False
        self.episodic_replay = False
        stream = self._find_stream(self.policy, self.policy_test, self.M)
        if stream is not None:
            self._bind(stream)

    def _allocate(self, stream):
        S, A = int(self.observation_space.n), int(self.action_space.n)
        self._Q = torch.zeros((stream.n_agents, S, A), dtype=torch.float64, device=stream.device)
        self._action_mask = torch.ones((S, A), dtype=torch.bool, device=stream.device)
        self.M._allocate(stream)

    # reference attribute names
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
        m = torch.as_tensor(value, device=self._stream.device).bool()
        assert m.shape[-2:] == self._Q.shape[-2:]
        self._action_mask = m.contiguous()

    def _run(self, interface, trials, steps, batch_size, no_replay, learn):
        if self._stream is None:
            self._bind(interface.rng)
        st = self._stream
        assert interface.rng is st, 'environment and agent must share one BatchStream'
        S, A = self._Q.shape[1], self._Q.shape[2]
        assert interface.n_states == S and interface.n_actions == A
        pol = self.policy if learn else self.policy_test
        results = []
        for t0, n_tr in self._chunks(trials):
            keep = []
            tr, res = self._make_trace(n_tr, steps, 0 if (no_replay or self.episodic_replay or not learn) else 1,
                                       1 if (learn and not no_replay and self.episodic_replay) else 0,
                                       batch_size, keep, td=learn, replay_td=learn and not no_replay)
            lr, gm, mlr = (st.param(self.learning_rate, 'learning_rate'), st.param(self.gamma, 'gamma'),
                           st.param(self.M.learning_rate, 'memory learning_rate'))
            mptr, mstride = self._mask_args(keep)
            p = _lib.DynaQParams(st.n_agents, interface.c_world(), st.c_struct(), pol.c_struct(st, keep), tr,
                                 self._Q.data_ptr(), self.M._rewards.data_ptr(), self.M._states.data_ptr(),
                                 self.M._terminals.data_ptr(), mptr, mstride, lr.data_ptr(), gm.data_ptr(),
                                 mlr.data_ptr(), n_tr, steps, batch_size, 1 if learn else 0,
                                 1 if no_replay else 0, 1 if self.episodic_replay else 0)
            _lib.call('cobel_dynaq_run', st.device, p, launch_stream(st))
            self._check_flags(res)
            self._fire_trial_callbacks(res, self.current_trial, session_first=t0)
            self.current_trial += n_tr
            results.append(res)
            if self.stop:
                break
        self.last_run = self._merge(results)
        return self.last_run

    def train(self, interface, trials, steps, batch_size=32, no_replay=False):
        """agent/dyna_q.py:140-215 for all agents."""
        return self._run(interface, trials, steps, batch_size, no_replay, learn=True)

    def test(self, interface, trials, steps):
        """agent/dyna_q.py:217-273 for all agents (``policy_test``; nothing is learned)."""
        return self._run(interface, trials, steps, 0, True, learn=False)

    # ---- stand-alone methods: for callers that drive the loop themselves (agent/dyna_q.py:176-203) -------------
    def _op(self, op, batch):
        st = self._stream
        keep = []
        lr, gm = st.param(self.learning_rate, 'learning_rate'), st.param(self.gamma, 'gamma')
        p, e = self.M._table_params(keep, self._Q, lr, gm), batch.c_struct()
        _lib.call('cobel_dynaq_op', st.device, p, op, e, launch_stream(st))
        return batch

    def update_q(self, experience):
        """agent/dyna_q.py:275-301 for all agents; returns the experience with its TD error (``'td'``)."""
        batch = ExperienceBatch.from_dicts(self._stream, experience, with_td=True)
        self.M._check_experience(batch)
        self._op(_lib.OP_UPDATE_Q, batch)
        out = dict(experience)
        out['td'] = batch.td[0, 0].item() if self._stream.single else batch.td[:, 0]
        return out

    def replay(self, batch_size):
        """agent/dyna_q.py:319-330: ``M.retrieve_batch(batch_size)``, then ``update_q`` for each experience in order."""
        if batch_size > 0:
            self._op(_lib.OP_REPLAY, ExperienceBatch(self._stream, batch_size))

    def predict_on_batch(self, batch):
        """agent/dyna_q.py:303-317: Q-values of a batch of states (``[N, B, A]``, or ``[B, A]`` for one agent)."""
        idx = torch.as_tensor(np.array(batch).astype(int), device=self._Q.device).reshape(-1)
        out = self._Q[:, idx]
        return out[0].cpu().numpy() if self._stream.single else out
