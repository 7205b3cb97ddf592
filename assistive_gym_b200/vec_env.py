"""`AssistiveVecEnv` — the batched env as a learner sees it (SURVEY.md §8(b) "fused vector path", §8(f)2).

The reference trains one `gym.Env` per RLlib worker process (`learn.py:26,61-69`); here ONE object steps
`n_envs` environments on one GPU.  `step(actions)` takes and returns torch CUDA tensors: the action tensor's
`data_ptr()` goes straight into `ag_feeding_step_dev` / `ag_bathing_step_dev`, observations / rewards / dones are
written into pre-allocated device tensors on the simulation's own stream, and nothing crosses PCIe.  Episodes of
all envs have the same length (200 steps, feeding.py:37), so the batch resets together; `auto_reset` does it inside
`step` the way vector-env wrappers do (the terminal observation is kept in `info['terminal_observation']`).
With numpy inputs the host-buffer entry points are used instead (pinned staging inside the C ABI)."""
import numpy as np


class AssistiveVecEnv:
    def __init__(self, env_id='assistive_gym:FeedingJaco-v1', n_envs=4096, device=0, seed=1001, auto_reset=True, config=None, _lib=None,
                 double_buffer=False, **env_kw):
        """double_buffer: a second copy of the batch is re-randomised by a background thread (the C ABI releases the GIL; its
        kernels run on that copy's own stream) while the first one is stepped; at the end of an episode the two swap, so
        `step` never waits for the 0.5 s of reset orchestration (reference env.py:92-97 rebuilds the world at every reset)."""
        from . import envs
        self.env = envs.make(env_id, n_envs=n_envs, device=device, seed=seed, config=config, **env_kw)
        if _lib is not None:
            self.env._sim_lib = _lib
        self._standby = None
        if double_buffer:
            self._standby = envs.make(env_id, n_envs=n_envs, device=device, seed=seed + 7919, config=config, **env_kw)
            if _lib is not None:
                self._standby._sim_lib = _lib
        self._bg, self._bg_obs, self._bg_err = None, None, None
        self.n_envs, self.device, self.auto_reset = n_envs, device, auto_reset
        self.task = self.env.task
        self.observation_space, self.action_space = self.env.observation_space, self.env.action_space
        self.obs_dim, self.act_dim = self.observation_space.shape[0], self.action_space.shape[0]
        self._step_dev = None
        self._buf = None

    # ------------------------------------------------------------------ gym-style API
    def _reset_standby(self):
        try:
            self._bg_obs = np.atleast_2d(self._standby.reset())
        except Exception as ex:          # surfaced by the next reset()
            self._bg_err = ex

    def _start_standby(self):
        import threading
        self._bg_obs, self._bg_err = None, None
        self._bg = threading.Thread(target=self._reset_standby, daemon=True)
        self._bg.start()

    def reset(self):
        if self._standby is not None and self._bg is not None:
            self._bg.join()
            if self._bg_err is not None:
                raise self._bg_err
            self.env, self._standby = self._standby, self.env          # the freshly reset copy becomes the live one
            obs = self._bg_obs
            self._buf = None                                            # device tensors are bound to a sim's stream
        else:
            obs = np.atleast_2d(self.env.reset())
        if self._standby is not None:
            self._start_standby()
        sim = self.env.id
        prefix = {'feeding': 'feeding', 'bed_bathing': 'bathing', 'dressing': 'dressing', 'scratch_itch': 'scratch'}[self.task]
        self._step_dev, self._step_host = getattr(sim, prefix + '_step_dev'), getattr(sim, prefix + '_step_host')
        self._t = 0
        return obs

    def _tensors(self, like):
        import torch
        if self._buf is None or self._buf[0].device != like.device:
            n = self.n_envs
            mk = lambda *shape: torch.zeros(shape, device=like.device, dtype=torch.float32)
            self._buf = (mk(n, self.obs_dim), mk(n), mk(n), mk(n, 4))
            self._stream = torch.cuda.ExternalStream(self.env.id.stream_ptr(), device=like.device)
        return self._buf

    def step(self, actions):
        """actions: torch CUDA tensor [n_envs, act_dim] (float32, contiguous) -> device tensors, or numpy -> numpy."""
        if self._step_dev is None:
            raise RuntimeError('call reset() first')
        is_torch = hasattr(actions, 'data_ptr')
        if is_torch:
            import torch
            a = actions.to(dtype=torch.float32).contiguous()
            obs, rew, done, info = self._tensors(a)
            # the caller's stream produced `a`; the simulation runs on its own stream
            self._stream.wait_stream(torch.cuda.current_stream(a.device))
            self._step_dev(a.data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(), info.data_ptr())
            torch.cuda.current_stream(a.device).wait_stream(self._stream)
            out = (obs, rew, done > 0.5, {'total_force_on_human': info[:, 0], 'task_success': info[:, 1]})
            finished = None     # decided from the step counter: no device read-back
        else:
            obs, rew, done, info = self._step_host(np.asarray(actions, dtype=np.float32).reshape(self.n_envs, -1))
            out = (obs, rew, done > 0.5, {'total_force_on_human': info[:, 0], 'task_success': info[:, 1]})
        self._t += 1
        self.env.iteration = self._t
        if self.auto_reset and self._t >= 200:
            term = out[0].clone() if is_torch else out[0].copy()
            new_obs = self.reset()
            if is_torch:
                import torch
                new_obs = torch.as_tensor(new_obs, device=out[0].device, dtype=torch.float32)
            out = (new_obs, out[1], out[2], dict(out[3], terminal_observation=term))
        return out

    def close(self):
        if self._bg is not None:
            self._bg.join()
        self.env.close()
        if self._standby is not None:
            self._standby.close()


class AssistiveRLlibVectorEnv:
    """The batched backend behind the interface RLlib's `VectorEnv` asks of a vectorised env (`vector_reset`, `reset_at`,
    `vector_step`, `get_sub_environments`; reference learn.py:41,61-69 hands RLlib one `gym.Env` per worker -- with this
    adapter one worker owns `n_envs` lock-step envs on its GPU).  RLlib itself is not a dependency: the class is duck-typed,
    `ray.rllib.env.VectorEnv.register` / `to_base_env` accept it where RLlib is installed.

    Episodes of all envs end together (200 steps, feeding.py:37): the first `reset_at` after the batch is done re-randomises
    the whole batch, the following `reset_at(i)` calls of the same round read row i of that reset."""

    def __init__(self, env_id='assistive_gym:FeedingJaco-v1', n_envs=64, device=0, seed=1001, config=None, _lib=None, **env_kw):
        self.vec = AssistiveVecEnv(env_id, n_envs=n_envs, device=device, seed=seed, auto_reset=False, config=config, _lib=_lib, **env_kw)
        self.num_envs = n_envs
        self.observation_space, self.action_space = self.vec.observation_space, self.vec.action_space
        self._obs = None
        self._fresh = np.zeros(n_envs, dtype=bool)

    def vector_reset(self):
        self._obs = self.vec.reset()
        self._fresh[:] = False
        return [self._obs[i] for i in range(self.num_envs)]

    def reset_at(self, index=None):
        index = 0 if index is None else int(index)
        if self._obs is None or self._fresh[index] or self.vec._t >= 200:
            self._obs = self.vec.reset()
            self._fresh[:] = False
        self._fresh[index] = True
        return self._obs[index]

    def vector_step(self, actions):
        obs, rew, done, info = self.vec.step(np.asarray(actions, dtype=np.float32).reshape(self.num_envs, -1))
        self._obs = obs
        self._fresh[:] = False
        infos = [{k: (v[i].item() if hasattr(v[i], 'item') else v[i]) for k, v in info.items()} for i in range(self.num_envs)]
        over = self.vec._t >= 200               # the env's own counter says the same (feeding.py:37); this one survives a replayed state
        return [obs[i] for i in range(self.num_envs)], [float(r) for r in rew], [bool(d) or over for d in done], infos

    def get_sub_environments(self):
        return []        # there are no per-env Python objects: the sub-environments are lanes of one simulation

    def try_render_at(self, index=None):
        return None
