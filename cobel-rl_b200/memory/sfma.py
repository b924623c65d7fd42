"""SFMA memory (reference: memory/sfma.py:21-416).

Per-agent experience tables plus the replay-relevant structures: strengths ``C`` and recency
``T`` (flat index ``a*S + s``) and inhibition ``I``.  The replay itself
(priority = C * D * (1 - I), softmax sampling, inhibition) runs inside ``SFMA.train()``
(csrc/sfma.cu); this object owns the tensors and the tunables, with the reference's names.
"""
import torch

from .. import _lib
from ..experience import Experience, ExperienceBatch  # noqa: F401  (Experience: memory/sfma.py:12-18)
from ..stream import cuda_stream
from .dyna_q import TableMemory

MODES = ('default', 'forward', 'reverse', 'blend_forward', 'blend_reverse', 'interpolate', 'sweeping')


class SFMAMemory(TableMemory):
    def __init__(self, metric, nb_states, nb_actions, decay_inhibition=0.9, decay_strength=1.0,
                 learning_rate=0.9, rng=None):
        self.metric = metric
        self.nb_states, self.nb_actions = int(nb_states), int(nb_actions)
        self.decay_inhibition = decay_inhibition
        self.decay_strength = decay_strength
        self.decay_recency = 0.9
        self.beta = 20
        self.C_step = 1.0
        self.I_step = 1.0
        self.R_threshold = 10.0 ** -6
        self.deterministic = False
        self.recency = False
        self.mode = 'default'
        self.blend = 0.1
        self.interpolation_fwd, self.interpolation_rev = 0.5, 0.5
        # strength-modulation and normalisation switches (memory/sfma.py:216-236, 283-288, 319-320): implemented in-kernel
        # (COBEL_SFMA_MOD_*), except error_mod / error_mod_local (see check_supported)
        self.C_normalize = False
        self.D_normalize = False
        self.R_normalize = True
        self.reward_mod_local = self.error_mod_local = self.reward_mod = self.error_mod = False
        self.policy_mod = self.state_mod = False
        self.reward_modulation = 1.0
        self._D_dev = None
        super().__init__(nb_states, nb_actions, learning_rate, rng, init_self_loops=True)

    def _allocate_extra(self, stream):
        n, S, A, dev = stream.n_agents, self.nb_states, self.nb_actions, stream.device
        self._C = torch.zeros((n, S * A), dtype=torch.float64, device=dev)
        self._T = torch.zeros((n, S * A), dtype=torch.float64, device=dev)
        self._I = torch.zeros((n, S), dtype=torch.float64, device=dev)
        self._carry = torch.zeros((n, 4), dtype=torch.int64, device=dev)            # kernel scratch

    C = property(lambda self: self._view(self._C))
    T = property(lambda self: self._view(self._T))
    I = property(lambda self: self._view(self._I))      # noqa: E741

    def similarity(self):
        """``metric.D`` as a device tensor (re-uploaded when the metric object changed it)."""
        D = self.metric.D
        if self._D_dev is None or self._D_src is not D:
            self._D_dev = torch.as_tensor(D, dtype=torch.float64).contiguous().to(self._alloc_for.device)
            self._D_src = D
        assert self._D_dev.shape == (self.nb_states, self.nb_states)
        return self._D_dev

    def check_supported(self):
        # error_mod / error_mod_local read experience['td'], which the reference's SFMA.train() has not computed
        # when it calls store() (agent/sfma.py:289-291) -- they cannot run there either
        unsupported = [k for k in ('error_mod_local', 'error_mod') if getattr(self, k)]
        if unsupported:
            raise NotImplementedError('SFMAMemory options not implemented by the B200 path: %s' % unsupported)

    def mod_flags(self):
        """COBEL_SFMA_MOD_* / *_NORMALIZE bits (include/cobel_b200.h), memory/sfma.py:216-236, 283-288, 319-320."""
        return ((1 if self.reward_mod_local else 0) | (2 if self.reward_mod else 0) | (4 if self.state_mod else 0) |
                (8 if self.C_normalize else 0) | (16 if self.D_normalize else 0) | (0 if self.R_normalize else 32))

    def mode_id(self):
        # an unknown mode string behaves like 'default' in the reference (memory/sfma.py:289-306)
        return MODES.index(self.mode) if self.mode in MODES else 0

    # ---- C ABI parameters ------------------------------------------------------------------------------------------
    def _params(self, st, world, pol, tr, keep, agent=None, n_tr=0, steps=1, batch=0, no_replay=False, learn=True,
                dynamic=False, trial_mode=None, nb_replays=None, random=None):
        """``CobelSFMAParams`` around the memory's tables; ``agent`` (an SFMA agent) adds Q, the action mask, the agent's
        hyper-parameters and replay switches."""
        mlr = st.param(self.learning_rate, 'memory learning_rate')
        keep.append(mlr)
        Q = lr = gm = td = mptr = None
        mstride = 0
        nbr, start_replay, rnd = 1, False, False
        if agent is not None:
            lr, gm = st.param(agent.learning_rate, 'learning_rate'), st.param(agent.gamma, 'gamma')
            keep += [lr, gm]
            mptr, mstride = agent._mask_args(keep)
            Q, td = agent._Q, agent._td
            nbr, start_replay, rnd = agent.nb_replays, agent.start_replay, agent.random
        if nb_replays is not None:
            nbr = nb_replays
        if random is not None:
            rnd = random
        polc = pol.c_struct(st, keep) if pol is not None else _lib.Policy(0, 0, None)
        return _lib.SFMAParams(
            st.n_agents, world, st.c_struct(), polc, tr,
            _lib.ptr(Q), self._rewards.data_ptr(), self._states.data_ptr(), self._terminals.data_ptr(),
            self._C.data_ptr(), self._T.data_ptr(), self._I.data_ptr(), self.similarity().data_ptr(), mptr, mstride,
            _lib.ptr(lr), _lib.ptr(gm), mlr.data_ptr(), float(self.beta), float(self.R_threshold),
            float(self.decay_inhibition), float(self.decay_strength), float(self.decay_recency), float(self.C_step),
            float(self.I_step), float(self.blend), float(self.interpolation_fwd), float(self.interpolation_rev),
            self.mode_id(), 1 if self.recency else 0, 1 if self.deterministic else 0, n_tr, steps, batch,
            nbr, 1 if start_replay else 0, 1 if rnd else 0, 1 if dynamic else 0,
            1 if no_replay else 0, 1 if learn else 0, _lib.ptr(td), _lib.ptr(trial_mode),
            float(self.reward_modulation), self.mod_flags(), 0, self._carry.data_ptr())

    def _table_world(self):
        return _lib.World(self.nb_states, self.nb_actions, 0, 0, None, None, None, None, None, None, None)

    # ---- stand-alone methods -----------------------------------------------------------------------------------
    def store(self, experience):
        """memory/sfma.py:195-236 for all agents: the table entry, strength ``C`` (decay, step, modulation) and
        recency ``T``."""
        self.check_supported()
        st = self._alloc_for
        batch = ExperienceBatch.from_dicts(st, experience)
        self._check_experience(batch)
        keep = []
        p, e = self._params(st, self._table_world(), None, _lib.Trace(), keep), batch.c_struct()
        _lib.call('cobel_sfma_op', st.device, p, _lib.OP_STORE, e, cuda_stream(st.device))

    def _gather(self, idx):
        """Experience dicts behind a padded ``[N, L]`` tensor of flat indices ``a*S + s``."""
        st = self._alloc_for
        batch = ExperienceBatch(st, idx.shape[1])
        batch.state.copy_(idx)
        keep = []
        p, e = self._params(st, self._table_world(), None, _lib.Trace(), keep), batch.c_struct()
        _lib.call('cobel_sfma_op', st.device, p, _lib.OP_GATHER, e, cuda_stream(st.device))
        return batch.to_dicts()

    def _replay(self, replay_length, current_state, agent=None, random=False, mask=None):
        assert not self.recency, 'the recency option runs inside SFMA.train() only'
        st = self._alloc_for
        n, dev = st.n_agents, st.device
        L = max(int(replay_length), 1)
        idx = torch.full((n, L), -1, dtype=torch.int32, device=dev)
        ln = torch.zeros((n, 1), dtype=torch.int32, device=dev)
        cnt = torch.zeros((2, n), dtype=torch.int64, device=dev)
        flags = torch.zeros(n, dtype=torch.int32, device=dev)
        tr = _lib.Trace(None, None, cnt[0].data_ptr(), cnt[1].data_ptr(), None, 0, idx.data_ptr(), L, ln.data_ptr(), 1,
                        flags.data_ptr(), None)
        keep = []
        p = self._params(st, self._table_world(), None if agent is None else agent.policy, tr, keep, agent=agent,
                         batch=int(replay_length), nb_replays=1, random=(random or (agent is not None and agent.random)))
        if mask is not None:        # retrieve_random_batch(n, mask): the caller's mask instead of the agent's
            m = torch.as_tensor(mask, device=dev).to(torch.uint8).contiguous()
            keep.append(m)
            p.action_mask, p.mask_agent_stride = m.data_ptr(), (m.shape[-2] * m.shape[-1] if m.dim() == 3 else 0)
        if current_state is None:
            state = torch.full((n,), -1, dtype=torch.int32, device=dev)
        else:
            state = torch.as_tensor(current_state, device=dev).reshape(-1).to(torch.int32)
            state = (state.expand(n) if state.numel() == 1 else state).contiguous()
        apply = agent is not None
        _lib.call('cobel_sfma_replay', dev, p, state.data_ptr(), 1 if apply else (2 if random else 0), cuda_stream(dev))
        if bool((flags & 2).any()):
            import warnings
            warnings.warn('SFMA replay: a draw fell within 1e-12 of a CDF bin edge (COBEL_FLAG_CDF_NEAR_TIE)')
        return self._gather(idx)

    def replay(self, replay_length, current_state=None, current_action=None):
        """memory/sfma.py:238-347 for all agents: the reactivated experiences as a list of Experience dicts (fields
        ``[N]`` tensors, -1 where an agent's replay ended early).  ``current_state``: one state per agent or None
        (start drawn from the strengths)."""
        assert current_action is None, 'current_action is drawn (memory/sfma.py:264); fixing it is not implemented'
        return self._replay(replay_length, current_state)

    def retrieve_random_batch(self, number_of_experiences, mask):
        """memory/sfma.py:375-416: ``number_of_experiences`` draws, uniform over the experiences the mask allows
        (``mask``: ``[S, A]`` or ``[N, S, A]`` booleans, or the reference's flat F-order ``[S*A]`` vector)."""
        S, A = self.nb_states, self.nb_actions
        m = torch.as_tensor(mask, device=self._alloc_for.device)
        if m.dim() == 1:
            m = m.reshape(A, S).t()
        return self._replay(number_of_experiences, None, random=True, mask=m.bool())
