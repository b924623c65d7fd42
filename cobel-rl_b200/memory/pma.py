"""PMA memory (reference: memory/pma.py:20-496): prioritized memory access after Mattar & Daw (2018).

Holds, per agent, the experience tables, the learned state-state transition matrix ``T``, the
successor representation ``SR = inv(I - gamma T)`` and ``update_mask``; the replay
(gain x need arg-max with n-step sequences) runs inside ``PMA.train()`` (csrc/pma.cu).

The stand-alone ``replay()`` and ``compute_need(None)`` run on worlds of up to 512 states and 2048 one-step backups.
Beyond 160 states or 1024 backups they take the banded eliminations of ``train()``, so T must keep the band of the
world (``sr_band()`` >= 0); otherwise they raise ``NotImplementedError`` before anything runs.
"""
import numpy as np
import torch

from .. import _lib
from ..experience import Experience, ExperienceBatch  # noqa: F401  (Experience: memory/pma.py:11-17)
from ..stream import cuda_stream
from .dyna_q import TableMemory


def _check_flags(flags):
    """COBEL_FLAG_BAND_VIOLATION and COBEL_FLAG_SINGULAR of a stand-alone call: raise instead of returning a vector
    that means nothing."""
    if bool((flags & 32).any()):
        raise _lib.CobelError('PMA: T lies outside the band assumed by the banded update_sr')
    if bool((flags & 8).any()):
        raise _lib.CobelError('PMA: singular elimination (T has a closed class without a unique stationary distribution)')


class PMAMemory(TableMemory):
    def __init__(self, sas, policy, learning_rate=0.9, learning_rate_q=0.9, gamma=0.9, gamma_q=0.9, rng=None):
        sas = np.asarray(sas)
        if sas.ndim == 3:                       # dense one-hot sas[S,A,S] (memory/pma.py:139)
            self.nb_states, self.nb_actions = sas.shape[0], sas.shape[1]
            self._T0 = np.sum(sas, axis=1) / self.nb_actions
        else:                                   # extension: successor table succ[S,A]
            self.nb_states, self.nb_actions = sas.shape
            T0 = np.zeros((self.nb_states, self.nb_states))
            np.add.at(T0, (np.repeat(np.arange(self.nb_states), self.nb_actions), sas.reshape(-1)), 1.0)
            self._T0 = T0 / self.nb_actions
        self.sas = sas
        self.policy = policy
        self.learning_rate_q = learning_rate_q
        self.learning_rate_T = 0.9
        self.gamma = gamma
        self.gamma_q = gamma_q
        self.min_gain = 10 ** -6
        self.min_gain_mode = 'original'
        self.equal_need = False
        self.equal_gain = False
        self.ignore_barriers = True
        self.allow_loops = False
        if rng is None and getattr(policy, 'rng', None) is not None:
            rng = policy.rng
        super().__init__(self.nb_states, self.nb_actions, learning_rate, rng, init_self_loops=False)

    def _allocate_extra(self, stream):
        n, S, dev = stream.n_agents, self.nb_states, stream.device
        self._T = torch.as_tensor(self._T0, dtype=torch.float64).to(dev).repeat(n, 1, 1).contiguous()
        g = stream.param(self.gamma, 'gamma').cpu().numpy()
        eye = np.eye(S)
        cache = {}
        SR = np.empty((n, S, S))
        for i, gi in enumerate(g):              # memory/pma.py:141, same LAPACK call as the reference
            if gi not in cache:
                cache[gi] = np.linalg.inv(eye - gi * self._T0)
            SR[i] = cache[gi]
        self._SR = torch.as_tensor(SR).to(dev).contiguous()
        self._update_mask = torch.zeros((n, S * self.nb_actions), dtype=torch.uint8, device=dev)
        self._min_gap = torch.full((n,), float('inf'), dtype=torch.float64, device=dev)
        self._carry = torch.zeros((n, 8), dtype=torch.int64, device=dev)            # kernel scratch
        self._need_scratch = torch.zeros((2, n, S), dtype=torch.float64, device=dev)   # kernel scratch
        self._world_band = self._matrix_band(self._T0)  # half bandwidth of the initial T
        self._band_T = self._world_band                # half bandwidth of T; None = must be re-measured
        self._band_scratch = None
        self.sr_band_max = 24                          # wider T: dense update_sr every trial (csrc/pma.cu); at most 31
        self.compute_update_mask()

    @staticmethod
    def _matrix_band(T):
        i, j = np.nonzero(np.asarray(T))
        return int(np.abs(i - j).max()) if i.size else 0

    @property
    def T(self):
        self._band_T = None                            # the caller may write through the view
        return self._view(self._T)

    def sr_band(self, world_band):
        """``(band, scratch, trusted)``: the half bandwidth that T keeps during a run (its own and the world's
        transitions), or -1 for the dense update_sr; allocates the factorisation scratch.  ``trusted``: T has not been
        handed out since this object last measured it or a kernel last enforced the band on it, so the library's
        streaming check of T (``pma_band_check_kernel``) can be skipped."""
        trusted = self._band_T is not None
        if self._band_T is None:
            nz = (self._T != 0).any(dim=0).nonzero()
            self._band_T = int((nz[:, 0] - nz[:, 1]).abs().max().item()) if nz.numel() else 0
        bw = max(self._band_T, int(world_band))
        S = self.nb_states
        if bw > self.sr_band_max or 2 * bw + 1 >= S:
            return -1, None, False
        self._band_T = bw                              # experienced transitions stay inside the world's band
        n = self._T.shape[0] * S * (2 * bw + 1)
        if self._band_scratch is None or self._band_scratch.numel() < n:
            self._band_scratch = torch.empty(n, dtype=torch.float64, device=self._T.device)
        return bw, self._band_scratch, trusted

    SR = property(lambda self: self._view(self._SR))
    update_mask = property(lambda self: self._view(self._update_mask).bool())
    min_gap = property(lambda self: self._view(self._min_gap))

    def compute_update_mask(self):
        """memory/pma.py:417-421: backups that lead into their own state are ignored."""
        S, A = self.nb_states, self.nb_actions
        flatF = self._states.permute(0, 2, 1).reshape(-1, S * A)          # states.flatten(order='F')
        own = torch.arange(S, device=flatF.device, dtype=flatF.dtype).repeat(A).unsqueeze(0)
        self._update_mask.copy_((flatF != own).to(torch.uint8))

    def update_sr(self):
        """memory/pma.py:413-415 as a stand-alone call: ``SR = inv(I - gamma T)`` for all agents by the register-tiled
        Gauss-Jordan kernel of csrc/pma.cu (a replay call of length 0 with ``update_sr`` set); more than 160 states:
        ``torch.linalg.inv`` (``train()`` and ``replay(..., update_sr=True)`` refresh SR on the device from the band
        factors instead)."""
        st = self._alloc_for
        S, A = self.nb_states, self.nb_actions
        if S > 160 or S * A > 1024:
            g = st.param(self.gamma, 'gamma').reshape(-1, 1, 1)
            eye = torch.eye(S, dtype=torch.float64, device=self._T.device)
            self._SR.copy_(torch.linalg.inv(eye - g * self._T))
            return
        keep = []
        p = self._mem_params(keep)
        n, dev = st.n_agents, st.device
        tmp = {'Q': torch.zeros((n, S, A), dtype=torch.float64, device=dev), 'one': torch.ones(n, dtype=torch.float64, device=dev),
               'cnt': torch.zeros((2, n), dtype=torch.int64, device=dev), 'state': torch.zeros(n, dtype=torch.int32, device=dev),
               'flags': torch.zeros(n, dtype=torch.int32, device=dev)}
        keep.append(tmp)
        p.Q, p.lr, p.gamma = tmp['Q'].data_ptr(), tmp['one'].data_ptr(), tmp['one'].data_ptr()
        p.policy = self.policy.c_struct(st, keep)
        p.trace.n_steps, p.trace.n_replay = tmp['cnt'][0].data_ptr(), tmp['cnt'][1].data_ptr()
        p.trace.flags = tmp['flags'].data_ptr()
        p.batch = 0
        dc = st.draw_count.clone()
        _lib.call('cobel_pma_replay', dev, p, tmp['state'].data_ptr(), 1, cuda_stream(dev))
        st.draw_count.copy_(dc)                      # a replay of length 0 draws nothing; keep the stream untouched either way
        _check_flags(tmp['flags'])

    def check_supported(self):
        pass        # every replay switch of the reference's PMAMemory is implemented

    def options(self):
        """COBEL_PMA_OPT_* bits (include/cobel_b200.h) of the reference's replay switches, memory/pma.py:238-249."""
        return ((1 if self.equal_need else 0) | (2 if self.equal_gain else 0) | (0 if self.ignore_barriers else 4) |
                (8 if self.allow_loops else 0))

    def policy_tables(self, stream, agent_policy, n_actions, keep):
        """Tie-pattern policy tables of a call (include/cobel_b200.h: CobelPMAParams.tab_*): one table per distinct
        (kind, parameter) among the agents' online policy and the memory's policy.  Returns
        ``(n_tab, kinds, params, table-of-agent [N,2] or None, scratch)``; ``n_tab = 0`` when the kernels
        evaluate the policies per row instead (more than 4 actions, or no epsilon-greedy policy at all)."""
        pols = (agent_policy, self.policy)
        if n_actions > 4 or all(pl.kind == 2 for pl in pols):
            return 0, None, None, None, None
        dev = stream.device
        kinds, params, cols = [], [], []
        for pl in pols:
            par = pl._param()
            if not torch.is_tensor(par) and np.ndim(par) == 0:
                key = (pl.kind, float(par))
                if key not in list(zip(kinds, params)):
                    kinds.append(key[0]); params.append(key[1])
                cols.append(list(zip(kinds, params)).index(key))
            else:
                uniq, inv = torch.unique(stream.param(par, pl.param_name), return_inverse=True)
                base = len(kinds)
                kinds += [pl.kind] * uniq.numel()
                params += uniq.cpu().tolist()
                cols.append(inv.to(torch.int32) + base)
        n_tab = len(kinds)
        tof = None
        if not (all(isinstance(c, int) for c in cols) and cols == [0, n_tab - 1]):
            # not the kernel's default assignment (agent: table 0, memory: the last one)
            tof = torch.stack([c if torch.is_tensor(c) else torch.full((stream.n_agents,), c, dtype=torch.int32, device=dev)
                               for c in cols], dim=1).contiguous()
        tcache = self.__dict__.setdefault('_tab_cache', {})
        tkey = (tuple(kinds), tuple(params), str(dev))
        if tkey not in tcache:
            if len(tcache) >= 16:
                tcache.clear()
            tcache[tkey] = (torch.tensor(kinds, dtype=torch.int32, device=dev), torch.tensor(params, dtype=torch.float64, device=dev))
        tkind, tpar = tcache[tkey]
        n = n_tab * _lib.pma_tab_doubles(n_actions) + 1024      # + COBEL_PMA_TIE_DOUBLES
        if getattr(self, '_tab_scratch', None) is None or self._tab_scratch.numel() < n:
            self._tab_scratch = torch.empty(n, dtype=torch.float64, device=dev)
        keep += [tkind, tpar, tof]
        return n_tab, tkind, tpar, tof, self._tab_scratch

    # ---- stand-alone methods -----------------------------------------------------------------------------------
    def _mem_params(self, keep, agent=None, batch=0, tr=None):
        """``CobelPMAParams`` around the memory's tables; ``agent`` (a PMA agent) adds Q, the action mask and the
        agent's hyper-parameters."""
        st = self._alloc_for
        S, A = self.nb_states, self.nb_actions
        if agent is not None:
            world = _lib.World(S, A, 0, 0, None, None, None, None, None, None, None)
            return agent._params(world, agent.policy, tr if tr is not None else _lib.Trace(), 0, 1, batch, False, True, -1, None, keep)
        par = {k: st.param(v, k) for k, v in dict(mem_lr=self.learning_rate, lr_q=self.learning_rate_q,
                                                  gamma_q=self.gamma_q, gamma_sr=self.gamma).items()}
        psr, pq, pstride = self.power_tables(st, keep)
        keep.append(par)
        world = _lib.World(S, A, 0, 0, None, None, None, None, None, None, None)
        return _lib.PMAParams(
            st.n_agents, world, st.c_struct(), _lib.Policy(0, 0, None), self.policy.c_struct(st, keep), _lib.Trace(),
            None, self._rewards.data_ptr(), self._states.data_ptr(), self._terminals.data_ptr(),
            self._T.data_ptr(), self._SR.data_ptr(), self._update_mask.data_ptr(), None, 0,
            None, None, par['mem_lr'].data_ptr(), par['lr_q'].data_ptr(), par['gamma_q'].data_ptr(),
            par['gamma_sr'].data_ptr(), psr.data_ptr(), pq.data_ptr(), pstride, self._min_gap.data_ptr(),
            self._carry.data_ptr(), self._need_scratch.data_ptr(), float(self.learning_rate_T), float(self.min_gain),
            1 if self.min_gain_mode == 'original' else 0, 0, 1, batch, 0, 1, -1, self.options(), None,
            0, 0, None, None, None, None)

    def store(self, experience):
        """memory/pma.py:148-166 for all agents: the table entry and ``T[s] += lr_T * (onehot(s') - T[s])``."""
        st = self._alloc_for
        batch = ExperienceBatch.from_dicts(st, experience)
        self._check_experience(batch)
        keep = []
        p, e = self._mem_params(keep), batch.c_struct()
        _lib.call('cobel_pma_op', st.device, p, _lib.OP_STORE, e, None, None, cuda_stream(st.device))
        self._band_T = None

    def _states_arg(self, current_state):
        st = self._alloc_for
        if current_state is None:
            return torch.full((st.n_agents,), -1, dtype=torch.int32, device=st.device)
        s = torch.as_tensor(current_state, device=st.device).reshape(-1).to(torch.int32)
        if bool(((s < 0) | (s >= self.nb_states)).any()):
            raise IndexError('PMA: current_state must lie in 0..%d (None for the stationary need)' % (self.nb_states - 1))
        return (s.expand(st.n_agents) if s.numel() == 1 else s).contiguous()

    def _set_band(self, p):
        """The banded update_sr arguments of a stand-alone replay beyond 160 states or 1024 one-step backups, where the
        library has no dense eliminations: the band ``train()`` would use, or -1, which the library rejects
        (``NotImplementedError``) before it launches anything."""
        S, A = self.nb_states, self.nb_actions
        if S <= 160 and S * A <= 1024:
            return
        band, scratch, trusted = self.sr_band(self._world_band)
        p.sr_band, p.band_scratch, p.band_trusted = band, _lib.ptr(scratch), 1 if trusted else 0

    def replay(self, q_function, action_mask, replay_length, current_state, force_first=None, update_sr=False):
        """memory/pma.py:168-267 for all agents.  ``q_function`` is the PMA agent whose Q table the replay reads and
        updates IN PLACE (the reference copies Q and the agent rebinds ``self.Q``, agent/pma.py:207); ``current_state``
        a state per agent in 0..S-1 (else ``IndexError``), or None (need = stationary distribution of T).
        ``update_sr``: ``update_sr()`` first, then the need from the refreshed SR, as the reference's train loop does at
        the end of a trial.  Returns ``(performed, Q)``: the performed updates as a padded ``[N, L]`` tensor of flat
        indices ``a*S + s`` (-1 = none) and the agent's Q table.

        Beyond 160 states or 1024 one-step backups (at most 512 and 2048) the replay takes the banded eliminations of
        ``train()``: SR is refreshed from the band LU of ``I - gamma T`` and the stationary need comes from the banded
        GTH elimination.  T must then lie inside the band of the memory's initial T (``sr_band()`` >= 0), else
        ``NotImplementedError``; a T the library finds outside the band it was promised raises ``CobelError``."""
        assert force_first is None, 'force_first is not implemented by the B200 path'
        agent = q_function
        assert hasattr(agent, '_Q') and agent.M is self, 'pass the PMA agent that owns this memory as q_function'
        st = self._alloc_for
        n, dev = st.n_agents, st.device
        state = self._states_arg(current_state)
        saved_mask, saved_flag = agent._action_mask, agent.mask_actions
        if action_mask is not None:
            agent._action_mask, agent.mask_actions = torch.as_tensor(action_mask, device=dev).bool().contiguous(), True
        else:
            agent.mask_actions = False
        try:
            keep = []
            L = max(int(replay_length), 1)
            idx = torch.full((n, L), -1, dtype=torch.int32, device=dev)
            ln = torch.zeros((n, 1), dtype=torch.int32, device=dev)
            zeros = torch.zeros((2, n), dtype=torch.int64, device=dev)
            flags = torch.zeros(n, dtype=torch.int32, device=dev)
            tr = _lib.Trace(None, None, zeros[0].data_ptr(), zeros[1].data_ptr(), None, 0, idx.data_ptr(), L,
                            ln.data_ptr(), 1, flags.data_ptr(), None)
            p = self._mem_params(keep, agent, int(replay_length), tr)
            self._set_band(p)
            _lib.call('cobel_pma_replay', dev, p, state.data_ptr(), 1 if update_sr else 0, cuda_stream(dev))
        finally:
            agent._action_mask, agent.mask_actions = saved_mask, saved_flag
        _check_flags(flags)
        return self._view(idx), agent.Q

    def compute_gain_batch(self, q_function, action_mask=None):
        """memory/pma.py:333-386: the gain of every one-step backup, ``[N, S*A]`` in the reference's order ``a*S + s``.
        ``q_function`` is the PMA agent that owns this memory."""
        agent = q_function
        st = self._alloc_for
        saved_mask, saved_flag = agent._action_mask, agent.mask_actions
        if action_mask is not None:
            agent._action_mask, agent.mask_actions = torch.as_tensor(action_mask, device=st.device).bool().contiguous(), True
        else:
            agent.mask_actions = False
        try:
            keep = []
            p = self._mem_params(keep, agent)
            out = torch.empty((st.n_agents, self.nb_states * self.nb_actions), dtype=torch.float64, device=st.device)
            _lib.call('cobel_pma_op', st.device, p, _lib.OP_GAIN_BATCH, None, None, out.data_ptr(), cuda_stream(st.device))
        finally:
            agent._action_mask, agent.mask_actions = saved_mask, saved_flag
        return self._view(out)

    def compute_need(self, current_state=None):
        """memory/pma.py:388-411: ``tile(SR[current_state], A)``, or the stationary distribution of T (|left Perron
        vector|, unit 2-norm) tiled when ``current_state`` is None.  The latter comes from the dense GTH elimination up
        to 160 states and 1024 one-step backups and from the banded one beyond (T inside the band of the memory's
        initial T, else ``NotImplementedError``, as for ``replay``)."""
        st = self._alloc_for
        keep = []
        p = self._mem_params(keep)
        state = self._states_arg(current_state)
        if current_state is None:
            # the stationary distribution comes from the GTH elimination of the replay path: a replay of length 0 on a
            # scratch Q table leaves it in need_scratch
            n, dev = st.n_agents, st.device
            tmp = {'Q': torch.zeros((n, self.nb_states, self.nb_actions), dtype=torch.float64, device=dev),
                   'one': torch.ones(n, dtype=torch.float64, device=dev), 'cnt': torch.zeros((2, n), dtype=torch.int64, device=dev),
                   'dc': st.draw_count.clone(), 'flags': torch.zeros(n, dtype=torch.int32, device=dev)}
            keep.append(tmp)
            p.Q, p.lr, p.gamma = tmp['Q'].data_ptr(), tmp['one'].data_ptr(), tmp['one'].data_ptr()
            p.policy = self.policy.c_struct(st, keep)
            p.trace.n_steps, p.trace.n_replay = tmp['cnt'][0].data_ptr(), tmp['cnt'][1].data_ptr()
            p.trace.flags = tmp['flags'].data_ptr()
            p.batch = 0
            self._set_band(p)
            _lib.call('cobel_pma_replay', dev, p, state.data_ptr(), 0, cuda_stream(dev))
            _check_flags(tmp['flags'])
        out = torch.empty((st.n_agents, self.nb_states * self.nb_actions), dtype=torch.float64, device=st.device)
        _lib.call('cobel_pma_op', st.device, p, _lib.OP_NEED, None, state.data_ptr(), out.data_ptr(), cuda_stream(st.device))
        return self._view(out)

    def action_probs_batch(self, q_function, action_mask=None):
        """memory/pma.py:423-450: ``policy.get_action_probs`` for every row of a ``[N, S, A]`` (or ``[S, A]``) table,
        each row divided by its sum."""
        p = self.policy.get_action_probs(q_function, action_mask)
        cols = [p[..., a] for a in range(p.shape[-1])]
        if len(cols) == 8:      # np.sum over exactly 8 values is a tree, below that a plain loop (SURVEY.md App. A.3)
            tot = ((cols[0] + cols[1]) + (cols[2] + cols[3])) + ((cols[4] + cols[5]) + (cols[6] + cols[7]))
        else:
            tot = cols[0]
            for c in cols[1:]:
                tot = tot + c
        return p / tot.unsqueeze(-1)

    def power_tables(self, stream, keep, q_gamma=None):
        """``float(gamma) ** k`` for k = 0..MAX_SEQ+1 with Python's pow, like the reference
        (memory/pma.py:310,315,485,491).  Returns (sr table, q table, per-agent stride)."""
        L = _lib.PMA_MAX_SEQ + 2
        gq = self.gamma_q if q_gamma is None else q_gamma
        if isinstance(self.gamma, (int, float)) and isinstance(gq, (int, float)):      # scalars: built once per pair
            cache = self.__dict__.setdefault('_pow_cache', {})
            key = (float(self.gamma), float(gq), str(stream.device))
            if key not in cache:
                if len(cache) >= 16:
                    cache.clear()
                cache[key] = tuple(torch.tensor([[float(g) ** k for k in range(L)]], dtype=torch.float64, device=stream.device)
                                   for g in key[:2])
            ta, tb = cache[key]
            return ta, tb, 0

        def table(x):
            v = stream.param(x, 'gamma').cpu().numpy()
            if np.all(v == v[0]):
                rows = [[float(v[0]) ** k for k in range(L)]]
            else:
                cache = {}
                rows = [cache.setdefault(float(g), [float(g) ** k for k in range(L)]) for g in v]
            return np.array(rows, dtype=np.float64)
        a, b = table(self.gamma), table(self.gamma_q if q_gamma is None else q_gamma)
        if a.shape[0] != b.shape[0]:
            n = stream.n_agents
            a, b = np.broadcast_to(a, (n, L)).copy(), np.broadcast_to(b, (n, L)).copy()
        ta = torch.as_tensor(a).to(stream.device).contiguous()
        tb = torch.as_tensor(b).to(stream.device).contiguous()
        keep += [ta, tb]
        return ta, tb, (0 if a.shape[0] == 1 else L)
