"""Tabular Q-learning agent (reference: agent/q.py:26-354).

The reference keeps ``Q`` as a dict keyed by the observation tuple and ``M`` as a growing
list of experience dicts.  Here ``Q`` is a ``[N, n_keys, A]`` table whose rows are the
distinct observations of the environment (gridworld states, or Topology node poses) and
``M`` is a per-agent append-only log in HBM; ``train()`` / ``test()`` run the whole loop of
all N agents in one launch of ``cobel_q_run`` (csrc/qagent.cu).
"""
import numpy as np
import torch

from .. import _lib
from ..experience import Experience, ExperienceBatch  # noqa: F401  (Experience: agent/q.py:17-23)
from ..spaces import Box, Discrete
from ..stream import BatchStream
from .agent import Agent, launch_stream


class QAgent(Agent):
    def __init__(self, observation_space, action_space, policy, policy_test=None, learning_rate=0.9,
                 gamma=0.8, custom_callbacks=None, rng=None):
        assert type(observation_space) in (Discrete, Box), 'Wrong observation space!'
        assert type(action_space) is Discrete, 'Wrong action space!'
        super().__init__(observation_space, action_space, custom_callbacks)
        self.policy = policy
        self.policy_test = policy if policy_test is None else policy_test
        assert rng is None or isinstance(rng, BatchStream), 'rng must be a cobel_rl_b200.BatchStream'
        self.rng = rng
        self.gamma = gamma
        self.learning_rate = learning_rate
        self.nb_actions = int(action_space.n)
        self._Q = None
        self._log = None
        self._log_len = None
        stream = self._find_stream(rng, self.policy, self.policy_test)
        if stream is not None:
            self._bind(stream)

    def _allocate(self, stream):
        self.rng = stream
        self._log_len = torch.zeros(stream.n_agents, dtype=torch.int64, device=stream.device)
        if type(self.observation_space) is Discrete:
            self._alloc_q(int(self.observation_space.n))

    def _alloc_q(self, n_keys):
        if self._Q is None:
            st = self._stream
            self._Q = torch.zeros((st.n_agents, n_keys, self.nb_actions), dtype=torch.float64, device=st.device)
        assert self._Q.shape[1] == n_keys, 'environment has a different number of observations'

    @property
    def Q(self):
        """``[N, n_keys, A]`` table (``[n_keys, A]`` for a single-agent stream); row k belongs to
        observation key k (state index, or node index of the first node with that pose)."""
        return self._view(self._Q)

    @property
    def M(self):
        """The experience log as a dict of ``[N, L]`` tensors (L = longest log; see ``log_len``)."""
        if self._log is None:
            return {}
        L = int(self._log_len.max())
        raw = self._log[:, :L]
        meta = raw[:, :, 1]
        return {'reward': raw[:, :, 0].view(torch.float64), 'state': meta & 0xFFFF,
                'next_state': (meta >> 16) & 0xFFFF, 'action': (meta >> 32) & 0xFF,
                'terminal': (meta >> 40) & 0xFF, 'log_len': self._log_len}

    def _ensure_log(self, extra):
        st = self._stream
        need = int(self._log_len.max()) + extra
        if self._log is None or self._log.shape[1] < need:
            new = torch.zeros((st.n_agents, need, 2), dtype=torch.int64, device=st.device)
            if self._log is not None:
                new[:, :self._log.shape[1]] = self._log
            self._log = new

    def _run(self, interface, trials, steps, batch_size, learn):
        if self._stream is None:
            self._bind(interface.rng)
        st = self._stream
        assert interface.rng is st, 'environment and agent must share one BatchStream'
        obs_key = getattr(interface, '_obs_key', None)
        self._alloc_q(interface.n_states)
        assert interface.n_actions == self.nb_actions
        pol = self.policy if learn else self.policy_test
        results = []
        for t0, n_tr in self._chunks(trials):
            keep = []
            if learn:
                self._ensure_log(n_tr * steps)
            tr, res = self._make_trace(n_tr, steps, 1 if learn else 0, 0, batch_size, keep, td=learn, replay_td=learn)
            lr, gm = st.param(self.learning_rate, 'learning_rate'), st.param(self.gamma, 'gamma')
            key_t = None
            if obs_key is not None:
                key_t = torch.as_tensor(obs_key, dtype=torch.int32, device=st.device).contiguous()
                keep.append(key_t)
            p = _lib.QParams(st.n_agents, interface.c_world(), st.c_struct(), pol.c_struct(st, keep), tr,
                             self._Q.data_ptr(), _lib.ptr(key_t), self._Q.shape[1], 0,
                             _lib.ptr(self._log) if learn else None, self._log.shape[1] if learn else 0,
                             self._log_len.data_ptr(), lr.data_ptr(), gm.data_ptr(), n_tr, steps,
                             batch_size if learn else 0, 1 if learn else 0)
            _lib.call('cobel_q_run', st.device, p, launch_stream(st))
            self._check_flags(res)
            self._fire_trial_callbacks(res, self.current_trial, session_first=t0)
            self.current_trial += n_tr
            results.append(res)
            if self.stop:
                break
        self.last_run = self._merge(results)
        return self.last_run

    def train(self, interface, trials, steps=32, batch_size=32):
        """agent/q.py:160-228 for all agents."""
        return self._run(interface, trials, steps, batch_size, learn=True)

    def test(self, interface, trials, steps=32):
        """agent/q.py:230-295 for all agents."""
        return self._run(interface, trials, steps, 0, learn=False)

    # ---- stand-alone methods (agent/q.py:196-216: the body of the reference's step loop) ------------------------
    def _op(self, op, batch, interface=None):
        st = self._stream
        obs_key = getattr(interface, '_obs_key', None) if interface is not None else getattr(self, '_op_obs_key', None)
        self._op_obs_key = obs_key
        keep = []
        key_t = None
        if obs_key is not None:
            key_t = torch.as_tensor(obs_key, dtype=torch.int32, device=st.device).contiguous()
            keep.append(key_t)
        n_keys = self._Q.shape[1]
        lr, gm = st.param(self.learning_rate, 'learning_rate'), st.param(self.gamma, 'gamma')
        world = _lib.World(n_keys if key_t is None else key_t.numel(), self.nb_actions, 0, 0, None, None, None, None, None, None, None)
        flags = torch.zeros(st.n_agents, dtype=torch.int32, device=st.device)
        tr = _lib.Trace(None, None, None, None, None, 0, None, 0, None, 0, flags.data_ptr(), None)
        p = _lib.QParams(st.n_agents, world, st.c_struct(), _lib.Policy(0, 0, None), tr, self._Q.data_ptr(),
                         _lib.ptr(key_t), n_keys, 0, _lib.ptr(self._log), 0 if self._log is None else self._log.shape[1],
                         self._log_len.data_ptr(), lr.data_ptr(), gm.data_ptr(), 0, 0, 0, 1)
        e = batch.c_struct()
        _lib.call('cobel_q_op', st.device, p, op, e, launch_stream(st))
        return batch

    def bind_interface(self, interface):
        """Allocate the Q rows for the observations of ``interface`` (the reference's dict grows on demand,
        agent/q.py:152-158) before the agent is driven step by step."""
        if self._stream is None:
            self._bind(interface.rng)
        self._alloc_q(interface.n_states)
        self._op_obs_key = getattr(interface, '_obs_key', None)

    def append(self, experience):
        """``self.M.append(experience)`` of the reference's step loop (agent/q.py:213)."""
        self._ensure_log(1)
        self._op(_lib.OP_STORE, ExperienceBatch.from_dicts(self._stream, experience))

    def update_q(self, experience):
        """agent/q.py:297-322 for all agents; returns the experience with its TD error."""
        batch = ExperienceBatch.from_dicts(self._stream, experience, with_td=True)
        self._op(_lib.OP_UPDATE_Q, batch)
        out = dict(experience)
        out['td'] = batch.td[0, 0].item() if self._stream.single else batch.td[:, 0]
        return out

    def replay(self, batch_size=32):
        """agent/q.py:344-354: ``for i in rng.choice(len(M), batch_size): update_q(M[i])``."""
        if batch_size > 0:
            assert bool((self._log_len > 0).all()), 'replay from an empty memory'
            self._op(_lib.OP_REPLAY, ExperienceBatch(self._stream, batch_size))

    def predict_on_batch(self, batch):
        """agent/q.py:324-342 for Discrete observations (state indices)."""
        idx = torch.as_tensor(np.array(batch).astype(int), device=self._Q.device).reshape(-1)
        out = self._Q[:, idx]
        return out[0].cpu().numpy() if self._stream.single else out
