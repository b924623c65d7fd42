"""Agent base class and callbacks (reference: agent/agent.py:14-243).

The reference runs ``for trial: for step:`` in Python and fires callbacks inline.
Here one call to ``train()`` / ``test()`` is one fused kernel launch for all N
agents, so per-step Python callbacks cannot run inside the loop.  What is kept:

* hook names and the ``logs`` keys; ``on_trial_begin`` / ``on_trial_end`` (and the
  replay hooks of PMA / SFMA) are fired after the launch, once per trial in
  order, with batched values (``[N]`` tensors; scalars for a single-agent stream);
* ``agent.stop`` is honoured between launches when ``trials_per_launch`` splits a
  session into several launches;
* per-step information is available from the recorded trajectory buffers
  (``agent.record = True`` -> ``agent.last_run``): ``step_sa``, ``step_next`` and, for the
  Q-learning agents when the call learns, ``step_td`` (the TD error of each step's online update).
This is the one intentional API deviation (SURVEY.md section 7.2).
"""
import abc

import torch

from .. import _lib
from ..stream import BatchStream, cuda_stream


class Callbacks:
    """Dispatcher with the reference's semantics (agent/agent.py:145-243): each hook
    receives a shallow copy of ``logs`` with ``logs['agent']`` injected and may return
    a dict that is merged back."""

    HOOKS = ('on_trial_begin', 'on_trial_end', 'on_step_begin', 'on_step_end', 'on_replay_begin', 'on_replay_end')

    def __init__(self, agent, custom_callbacks=None):
        self.agent = agent
        self.custom_callbacks = {} if custom_callbacks is None else custom_callbacks

    def _fire(self, name, logs):
        for cb in self.custom_callbacks.get(name, []):
            view = dict(logs)
            view['agent'] = self.agent
            out = cb(view)
            if isinstance(out, dict):
                logs.update(out)
        return logs

    def __getattr__(self, name):
        if name in Callbacks.HOOKS:
            return lambda logs: self._fire(name, logs)
        raise AttributeError(name)


class RunResult(dict):
    """Per-agent outputs of one ``train()`` / ``test()`` call (CobelTrace).

    Always: ``trial_steps``, ``trial_reward`` ``[N, trials]``; ``n_steps``, ``n_replay``, ``flags`` ``[N]``.
    With ``agent.record``: ``step_sa`` (``s*A + a``) and ``step_next`` (arrival state) ``[N, trials*steps]`` int32,
    -1 behind ``n_steps``; ``replay_idx`` and ``replay_len``.  With ``agent.record`` in a call that learns (Dyna-Q,
    QAgent, SFMA, PMA ``train()``, also with ``no_replay=True``): ``step_td`` ``[N, trials*steps]`` fp64, the TD error
    that each step's online update added to ``Q[s,a]`` (scaled by the learning rate), NaN behind ``n_steps``.
    Entry k of every per-step buffer belongs to the agent's k-th step.  Every buffer keeps its leading agent axis,
    also for a single-agent stream."""
    __getattr__ = dict.__getitem__


class Agent(abc.ABC):
    def __init__(self, observation_space, action_space, custom_callbacks=None):
        self.observation_space = observation_space
        self.action_space = action_space
        self.callbacks = Callbacks(self, custom_callbacks)
        self.current_trial = 0
        self.stop = False
        # batched-path extras
        self.record = False            # record per-step (s,a), next state, TD error and replay indices of each call
        self.trials_per_launch = None  # split a session into launches of this many trials
        self.last_run = None
        self._stream = None

    # ---- stream / allocation -------------------------------------------------
    def _find_stream(self, *candidates):
        for c in candidates:
            rng = getattr(c, 'rng', None) if not isinstance(c, BatchStream) else c
            if isinstance(rng, BatchStream):
                return rng
        return None

    def _bind(self, stream):
        """Attach the agent to a BatchStream (fixes N and the device) and allocate its tables."""
        if self._stream is stream:
            return
        assert self._stream is None, 'agent is already bound to another BatchStream'
        self._stream = stream
        self._allocate(stream)

    @abc.abstractmethod
    def _allocate(self, stream):
        ...

    def _view(self, t):
        return t[0] if self._stream.single else t

    def _assign(self, dst, value):
        v = torch.as_tensor(value, device=dst.device).to(dst.dtype)
        dst.copy_(v.reshape(dst.shape) if v.numel() == dst.numel() else v.expand_as(dst))

    # ---- trace plumbing --------------------------------------------------------
    def _make_trace(self, trials, steps, replay_per_step, replay_calls_per_trial, replay_len_max, keep, td=False):
        """CobelTrace of one launch and the RunResult that owns its buffers; ``td`` = the launch performs online
        Q updates whose TD errors are recorded (``step_td``) when ``agent.record`` is set."""
        st = self._stream
        n, dev = st.n_agents, st.device
        res = RunResult()
        res['trial_steps'] = torch.zeros((n, trials), dtype=torch.int32, device=dev)
        res['trial_reward'] = torch.zeros((n, trials), dtype=torch.float64, device=dev)
        res['n_steps'] = torch.zeros(n, dtype=torch.int64, device=dev)
        res['n_replay'] = torch.zeros(n, dtype=torch.int64, device=dev)
        res['flags'] = torch.zeros(n, dtype=torch.int32, device=dev)
        step_cap = replay_cap = calls_cap = 0
        if self.record:
            step_cap = trials * steps
            calls_cap = trials * (steps * replay_per_step + replay_calls_per_trial)
            replay_cap = calls_cap * replay_len_max
            res['step_sa'] = torch.full((n, max(step_cap, 1)), -1, dtype=torch.int32, device=dev)
            res['step_next'] = torch.full((n, max(step_cap, 1)), -1, dtype=torch.int32, device=dev)
            if td:
                res['step_td'] = torch.full((n, max(step_cap, 1)), float('nan'), dtype=torch.float64, device=dev)
            res['replay_idx'] = torch.full((n, max(replay_cap, 1)), -1, dtype=torch.int32, device=dev)
            res['replay_len'] = torch.full((n, max(calls_cap, 1)), -1, dtype=torch.int32, device=dev)
        keep.append(res)
        tr = _lib.Trace(res['trial_steps'].data_ptr(), res['trial_reward'].data_ptr(), res['n_steps'].data_ptr(),
                        res['n_replay'].data_ptr(), _lib.ptr(res.get('step_sa')), step_cap,
                        _lib.ptr(res.get('replay_idx')), replay_cap, _lib.ptr(res.get('replay_len')), calls_cap,
                        res['flags'].data_ptr(), _lib.ptr(res.get('step_next')), _lib.ptr(res.get('step_td')))
        return tr, res

    def _mask_args(self, keep):
        """(pointer, per-agent stride) of the action mask, or (NULL, 0) when mask_actions is False."""
        if not self.mask_actions:
            return None, 0
        m = self._action_mask.to(torch.uint8).contiguous()
        keep.append(m)
        S, A = m.shape[-2], m.shape[-1]
        return m.data_ptr(), (S * A if m.dim() == 3 else 0)

    def _fire_trial_callbacks(self, res, first_trial, replay_calls=(0, 0), flat_order='F', session_first=0):
        """Fire the per-trial hooks after a launch, once per trial in order, with batched values.
        ``replay_calls = (calls at trial start, calls at trial end)`` additionally fires
        ``on_replay_begin`` / ``on_replay_end`` (agent/pma.py:112-135, agent/sfma.py:139-187) with
        ``logs['replay']`` = dict of padded ``[N, L]`` tensors (flat index, state, action; -1 = no
        experience) when the run was recorded (``agent.record``), else ``None``."""
        cbs = self.callbacks.custom_callbacks
        if not any(k in cbs for k in Callbacks.HOOKS):
            return
        single = self._stream.single
        trials = res['trial_steps'].shape[1]
        per_trial = replay_calls[0] + replay_calls[1]
        offsets = None
        if per_trial and 'replay_len' in res and ('on_replay_end' in cbs or 'on_replay_begin' in cbs):
            lens = res['replay_len'][:, :trials * per_trial].clamp(min=0).long()
            offsets = torch.cumsum(lens, dim=1) - lens
        S = int(self.observation_space.n) if hasattr(self.observation_space, 'n') else 0

        def replay_logs(call):
            if offsets is None:
                return None
            ln, off = lens[:, call], offsets[:, call]
            L = int(ln.max()) if ln.numel() else 0
            pos = torch.arange(L, device=ln.device).unsqueeze(0)
            valid = pos < ln.unsqueeze(1)
            idx = torch.gather(res['replay_idx'].long(), 1, (off.unsqueeze(1) + pos).clamp(max=res['replay_idx'].shape[1] - 1))
            idx = torch.where(valid, idx, torch.full_like(idx, -1))
            A = int(self.action_space.n)
            state = torch.where(valid, idx % S if flat_order == 'F' else idx // A, idx)
            action = torch.where(valid, idx // S if flat_order == 'F' else idx % A, idx)
            return {'index': idx, 'state': state, 'action': action, 'length': ln}

        for t in range(trials):
            steps_t, rew_t = res['trial_steps'][:, t], res['trial_reward'][:, t]
            logs = {'trial_reward': 0.0, 'trial': first_trial + t, 'trial_session': session_first + t}
            logs = self.callbacks.on_trial_begin(logs)
            for c in range(per_trial):
                if c == replay_calls[0]:      # the online steps lie between the start and the end replays
                    logs['steps'] = int(steps_t[0]) if single else steps_t
                    logs['trial_reward'] = float(rew_t[0]) if single else rew_t
                logs = self.callbacks.on_replay_begin(logs)
                logs['replay'] = replay_logs(t * per_trial + c)
                logs = self.callbacks.on_replay_end(logs)
            logs['steps'] = int(steps_t[0]) if single else steps_t
            logs['trial_reward'] = float(rew_t[0]) if single else rew_t
            logs = self.callbacks.on_trial_end(logs)

    def _chunks(self, trials):
        c = trials if not self.trials_per_launch else int(self.trials_per_launch)
        if trials <= 0:          # a zero-trial session is a no-op that still returns empty statistics
            yield 0, 0
            return
        t = 0
        while t < trials:
            yield t, min(c, trials - t)
            t += c

    @staticmethod
    def _merge(results):
        """One RunResult for a session that ran as several launches (``trials_per_launch``).  Per-trial arrays are
        concatenated; the recorded per-step / per-replay buffers of a launch are padded (-1, NaN for ``step_td``)
        behind the data of each agent, so they are compacted per agent (the merged buffer is addressed by cumulative
        counts, exactly like the buffer of a single launch)."""
        if len(results) == 1:
            return results[0]

        def compact_cat(bufs, counts, pad=-1):
            n = bufs[0].shape[0]
            total = sum(c.long() for c in counts)
            out = torch.full((n, max(int(total.max()), 1)), pad, dtype=bufs[0].dtype, device=bufs[0].device)
            rows = torch.arange(n, device=out.device).unsqueeze(1)
            offset = torch.zeros(n, dtype=torch.long, device=out.device)
            for b, c in zip(bufs, counts):
                pos = torch.arange(b.shape[1], device=out.device).unsqueeze(0)
                valid = pos < c.long().unsqueeze(1)
                dst = (offset.unsqueeze(1) + pos)
                out[rows.expand_as(dst)[valid], dst[valid]] = b[valid]
                offset += c.long()
            return out

        out = RunResult()
        for k in results[0]:
            if k in ('n_steps', 'n_replay'):
                out[k] = sum(r[k] for r in results)
            elif k == 'flags':
                out[k] = results[0][k]
                for r in results[1:]:
                    out[k] = out[k] | r[k]
            elif k in ('step_sa', 'step_next'):
                out[k] = compact_cat([r[k] for r in results], [r['n_steps'] for r in results])
            elif k == 'step_td':
                out[k] = compact_cat([r[k] for r in results], [r['n_steps'] for r in results], float('nan'))
            elif k == 'replay_idx':
                out[k] = compact_cat([r[k] for r in results], [r['n_replay'] for r in results])
            elif k == 'replay_len':
                out[k] = compact_cat([r[k] for r in results], [(r[k] >= 0).sum(dim=1) for r in results])
            else:
                out[k] = torch.cat([r[k] for r in results], dim=1)
        return out

    def _check_flags(self, res):
        """Raise / warn on the COBEL_FLAG_* bits a launch left behind (include/cobel_b200.h)."""
        fl = res['flags']
        if not fl.numel() or int(fl.max().item()) == 0:
            return
        if bool((fl & 32).any()):      # COBEL_FLAG_BAND_VIOLATION (a violated band promise also derails the eliminations)
            raise _lib.CobelError('PMA: T or a transition left the band assumed by the banded update_sr')
        if bool((fl & 8).any()):       # COBEL_FLAG_SINGULAR
            raise _lib.CobelError('PMA: singular elimination -- T has no unique stationary distribution (unreachable cells '
                                  'form closed classes of their own) or a pivot of I - gamma T underflowed')
        if bool((fl & 64).any()):      # COBEL_FLAG_REPLAY_OVERFLOW
            raise _lib.CobelError('SFMA: an agent has experienced more (state, action) pairs than the replay kernel can '
                                  'stage in shared memory for this state space')
        if self.record and bool((fl & 1).any()):
            raise _lib.CobelError('trace buffer overflow (internal sizing error)')
        if bool((fl & 2).any()):       # COBEL_FLAG_CDF_NEAR_TIE: exp() / prefix sums are not bit-identical to NumPy's
            import warnings
            warnings.warn('SFMA replay: %d agent(s) drew within 1e-12 of a CDF bin edge; their sampled indices may '
                          'differ from the reference' % int((fl & 2).bool().sum()))

    @abc.abstractmethod
    def train(self, interface, trials, steps):
        ...

    @abc.abstractmethod
    def test(self, interface, trials, steps):
        ...

    @abc.abstractmethod
    def predict_on_batch(self, batch):
        ...


def launch_stream(stream):
    return cuda_stream(stream.device)
