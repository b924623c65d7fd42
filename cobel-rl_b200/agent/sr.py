"""Successor-representation agent (reference: agent/sr.py:25-324).

``train()`` / ``test()`` run the reference's loop (Q from the SR and the learned reward
vector, action selection, environment step, reward / transition-model / SR row update) for all
N agents in one launch of ``cobel_sr_run`` (csrc/sr.cu).  The reference's dense one-hot
transition model ``transitions[S,A,S]`` is held as its arg-max ``model[S,A]``.

``SR(..., compact=True, max_visited=V)`` selects the visited-set compaction for very large
state spaces (100x100 and beyond, csrc/sr_compact.cu): per agent only the V x V block of the
SR over the states it has touched is stored, everything else is implied (identity rows,
self-loop model, zero reward); results are bit-identical to the dense agent.
Memory (``N·V²·8`` bytes of ``SRc``) is the only limit on ``max_visited``.  The stand-alone methods
``update``, ``retrieve_q`` and ``predict_on_batch`` act on the compact tables too (``cobel_sr_compact_op``, one
launch per call): ``update`` inserts ``state``, then ``next_state``, into the visited set exactly as a learning
step of ``train()`` does, so hand-written loops and fused training interleave freely; ``retrieve_q`` /
``predict_on_batch`` insert nothing and return the dense agent's values (an unvisited state's row is ``e_s``).
"""
import numpy as np
import torch

from .. import _lib
from ..experience import Experience, ExperienceBatch  # noqa: F401  (Experience: agent/sr.py:16-22)
from ..spaces import Discrete
from .agent import Agent, launch_stream

_VISITED_OVERFLOW = ('an agent visited more than max_visited=%d distinct states; raise max_visited or shorten the '
                     'horizon')


class SR(Agent):
    def __init__(self, observation_space, action_space, policy, policy_test=None, learning_rate=0.1,
                 gamma=0.99, custom_callbacks=None, compact=False, max_visited=128):
        assert type(observation_space) is Discrete, 'SR requires a discrete observation space!'
        assert type(action_space) is Discrete, 'SR requires a discrete action space!'
        super().__init__(observation_space, action_space, custom_callbacks)
        self.policy = policy
        self.policy_test = policy if policy_test is None else policy_test
        self.learning_rate = learning_rate
        self.gamma = gamma
        self.mask_actions = False
        self.compact = bool(compact)
        self.max_visited = int(max_visited)
        stream = self._find_stream(self.policy, self.policy_test)
        if stream is not None:
            self._bind(stream)

    def _allocate(self, stream):
        S, A, n, dev = int(self.observation_space.n), int(self.action_space.n), stream.n_agents, stream.device
        self._action_mask = torch.ones((S, A), dtype=torch.bool, device=dev)
        if self.compact:
            V = self.max_visited
            self._SRc = torch.zeros((n, V, V), dtype=torch.float64, device=dev)
            self._visited = torch.full((n, V), -1, dtype=torch.int32, device=dev)
            self._n_visited = torch.zeros(n, dtype=torch.int32, device=dev)
            self._rewards = torch.zeros((n, V), dtype=torch.float64, device=dev)
            self._model = torch.zeros((n, V, A), dtype=torch.int32, device=dev)
            return
        self._SR = torch.eye(S, dtype=torch.float64, device=dev).repeat(n, 1, 1).contiguous()     # sr.py:130
        self._model = torch.arange(S, dtype=torch.int32, device=dev).reshape(1, S, 1).repeat(n, 1, A).contiguous()
        self._rewards = torch.zeros((n, S), dtype=torch.float64, device=dev)                       # sr.py:136
        self._action_mask = torch.ones((S, A), dtype=torch.bool, device=dev)

    @property
    def SR(self):
        if self.compact:
            raise AttributeError('compact SR agent: use SR_compact / visited / n_visited, or dense_sr(agent)')
        return self._view(self._SR)

    rewards = property(lambda self: self._view(self._rewards))
    model = property(lambda self: self._view(self._model))
    SR_compact = property(lambda self: self._view(self._SRc))
    visited = property(lambda self: self._view(self._visited))
    n_visited = property(lambda self: self._view(self._n_visited))

    def dense_sr(self, agent=0):
        """Materialise the dense ``[S,S]`` SR of one agent of a compact run (checking / analysis)."""
        S = int(self.observation_space.n)
        v = int(self._n_visited[agent])
        idx = self._visited[agent, :v].long()
        out = torch.eye(S, dtype=torch.float64, device=self._SRc.device)
        out[idx.unsqueeze(1), idx.unsqueeze(0)] = self._SRc[agent, :v, :v]
        return out

    def dense_rewards(self, agent=0):
        S = int(self.observation_space.n)
        v = int(self._n_visited[agent])
        out = torch.zeros(S, dtype=torch.float64, device=self._SRc.device)
        out[self._visited[agent, :v].long()] = self._rewards[agent, :v]
        return out

    @property
    def transitions(self):
        """The reference's one-hot ``(S, A, S)`` model (sr.py:131-135), materialised on demand."""
        S = self._SR.shape[1]
        return self._view(torch.nn.functional.one_hot(self._model.long(), S).to(torch.float64))

    @property
    def action_mask(self):
        return self._action_mask

    @action_mask.setter
    def action_mask(self, value):
        self._action_mask = torch.as_tensor(value, device=self._stream.device).bool().contiguous()

    def _run(self, interface, trials, steps, learn):
        if self._stream is None:
            self._bind(interface.rng)
        st = self._stream
        assert interface.rng is st, 'environment and agent must share one BatchStream'
        assert interface.n_states == int(self.observation_space.n) and interface.n_actions == self._model.shape[2]
        pol = self.policy if learn else self.policy_test
        results = []
        for t0, n_tr in self._chunks(trials):
            keep = []
            tr, res = self._make_trace(n_tr, steps, 0, 0, 0, keep)
            lr, gm = st.param(self.learning_rate, 'learning_rate'), st.param(self.gamma, 'gamma')
            mptr, mstride = self._mask_args(keep)
            if self.compact:
                assert mstride == 0, 'compact SR supports one action mask shared by all agents'
                p = _lib.SRCompactParams(st.n_agents, interface.c_world(), st.c_struct(), pol.c_struct(st, keep), tr,
                                         self._SRc.data_ptr(), self._rewards.data_ptr(), self._model.data_ptr(),
                                         self._visited.data_ptr(), self._n_visited.data_ptr(), mptr, lr.data_ptr(),
                                         gm.data_ptr(), self.max_visited, n_tr, steps, 1 if learn else 0)
                _lib.call('cobel_sr_compact_run', st.device, p, launch_stream(st))
                if bool((res['flags'] & 16).any()):
                    raise _lib.CobelError(_VISITED_OVERFLOW % self.max_visited)
            else:
                p = _lib.SRParams(st.n_agents, interface.c_world(), st.c_struct(), pol.c_struct(st, keep), tr,
                                  self._SR.data_ptr(), self._rewards.data_ptr(), self._model.data_ptr(), mptr, mstride,
                                  lr.data_ptr(), gm.data_ptr(), n_tr, steps, 1 if learn else 0, 0)
                _lib.call('cobel_sr_run', st.device, p, launch_stream(st))
            self._check_flags(res)
            self._fire_trial_callbacks(res, self.current_trial, session_first=t0)
            self.current_trial += n_tr
            results.append(res)
            if self.stop:
                break
        self.last_run = self._merge(results)
        return self.last_run

    def train(self, interface, trials, steps):
        """agent/sr.py:142-197 for all agents."""
        return self._run(interface, trials, steps, learn=True)

    def test(self, interface, trials, steps):
        """agent/sr.py:199-253 for all agents."""
        return self._run(interface, trials, steps, learn=False)

    # ---- stand-alone methods -----------------------------------------------------------------------------------
    def _op_params(self):
        st = self._stream
        S, A = self._SR.shape[1], self._model.shape[2]
        lr, gm = st.param(self.learning_rate, 'learning_rate'), st.param(self.gamma, 'gamma')
        world = _lib.World(S, A, 0, 0, None, None, None, None, None, None, None)
        p = _lib.SRParams(st.n_agents, world, st.c_struct(), _lib.Policy(0, 0, None), _lib.Trace(), self._SR.data_ptr(),
                          self._rewards.data_ptr(), self._model.data_ptr(), None, 0, lr.data_ptr(), gm.data_ptr(), 0, 0, 1, 0)
        return p, (lr, gm)

    def _compact_op(self, op, e=None, states=None, q=None, flags=None):
        """One launch of ``cobel_sr_compact_op`` (csrc/sr_compact.cu) on the compact tables."""
        st = self._stream
        S, A = int(self.observation_space.n), self._model.shape[2]
        lr, gm = st.param(self.learning_rate, 'learning_rate'), st.param(self.gamma, 'gamma')
        world = _lib.World(S, A, 0, 0, None, None, None, None, None, None, None)
        tr = _lib.Trace()
        tr.flags = _lib.ptr(flags)
        p = _lib.SRCompactParams(st.n_agents, world, st.c_struct(), _lib.Policy(0, 0, None), tr, self._SRc.data_ptr(),
                                 self._rewards.data_ptr(), self._model.data_ptr(), self._visited.data_ptr(),
                                 self._n_visited.data_ptr(), None, lr.data_ptr(), gm.data_ptr(), self.max_visited, 0, 0, 1)
        n_query = 0 if states is None else states.shape[1]
        _lib.call('cobel_sr_compact_op', st.device, p, op, e, _lib.ptr(states), n_query, _lib.ptr(q), launch_stream(st))

    def _compact_retrieve_q(self, states):
        """Q of the compact tables for ``states[N, B]`` -> ``[N, B, A]``, one launch."""
        st = self._stream
        S = int(self.observation_space.n)
        if bool(((states < 0) | (states >= S)).any()):
            raise IndexError('state outside the tables')
        states = states.to(torch.int32).contiguous()
        q = torch.empty((st.n_agents, states.shape[1], self._model.shape[2]), dtype=torch.float64, device=st.device)
        self._compact_op(_lib.OP_RETRIEVE_Q, states=states, q=q)
        return q

    def update(self, experience):
        """agent/sr.py:255-286 for all agents: learned reward, transition model and the SR row of ``state``."""
        st = self._stream
        batch = ExperienceBatch.from_dicts(st, experience)
        S = int(self.observation_space.n)
        if bool(((batch.state < 0) | (batch.state >= S) | (batch.next_state < 0) | (batch.next_state >= S)).any()):
            raise IndexError('experience with a state outside the tables')
        if self.compact:
            flags = torch.zeros(st.n_agents, dtype=torch.int32, device=st.device)
            self._compact_op(_lib.OP_STORE, e=batch.c_struct(), flags=flags)
            if bool((flags & 16).any()):           # COBEL_FLAG_VISITED_OVERFLOW
                raise _lib.CobelError(_VISITED_OVERFLOW % self.max_visited)
            return experience
        p, keep = self._op_params()
        e = batch.c_struct()
        _lib.call('cobel_sr_op', st.device, p, _lib.OP_STORE, e, None, None, launch_stream(st))
        return experience

    def retrieve_q(self, state):
        """agent/sr.py:288-308: ``Q[a] = np.sum(SR[m(s, a)] * rewards)`` in NumPy's pairwise order (csrc/ops.cu;
        compact agents: csrc/sr_compact.cu).  ``state`` is a scalar or ``[N]``; returns ``[N, A]`` (``[A]`` single)."""
        st = self._stream
        if self.compact:
            s = torch.as_tensor(state, device=st.device).reshape(-1, 1)
            return self._view(self._compact_retrieve_q(s.expand(st.n_agents, 1))[:, 0])
        s = torch.as_tensor(state, device=st.device).reshape(-1).to(torch.int32)
        s = (s.expand(st.n_agents) if s.numel() == 1 else s).contiguous()
        q = torch.empty((st.n_agents, self._model.shape[2]), dtype=torch.float64, device=st.device)
        p, keep = self._op_params()
        _lib.call('cobel_sr_op', st.device, p, _lib.OP_RETRIEVE_Q, None, s.data_ptr(), q.data_ptr(), launch_stream(st))
        return self._view(q)

    def predict_on_batch(self, batch):
        """Q of every state of ``batch`` for all agents: ``[N, B, A]``, or a NumPy ``[B, A]`` for a single-agent stream.
        Compact agents evaluate the whole batch in one launch."""
        idx = np.array(batch).astype(int).reshape(-1)
        if self.compact:
            st = self._stream
            s = torch.as_tensor(idx, device=st.device).reshape(1, -1)
            out = self._compact_retrieve_q(s.expand(st.n_agents, -1))
            return out[0].cpu().numpy() if st.single else out
        out = torch.stack([self.retrieve_q(int(s)) for s in idx], dim=-2)
        return out.cpu().numpy() if self._stream.single else out
