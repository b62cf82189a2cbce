"""``parl.utils.ReplayMemory`` with the storage in HBM — interface of parl/utils/replay_memory.py:21-199
(append / sample_batch / make_index / sample_batch_by_index / size / save / load with the same .npz
keys).  Rows are gathered on the device (rl_gather_rows); ``sample_batch`` hands back numpy arrays
like the reference unless ``as_tensor=True`` (device tensors for a device-resident learner)."""
import numpy as np
import torch

from .. import kernels

__all__ = ['ReplayMemory']


class ReplayMemory(object):
    def __init__(self, max_size, obs_dim, act_dim, device=None):
        self.max_size = int(max_size)
        self.obs_dim, self.act_dim = obs_dim, act_dim
        if device is None:
            if not torch.cuda.is_available():
                raise RuntimeError('parl_b200.ReplayMemory lives in HBM: no CUDA device visible (no CPU fallback)')
            device = torch.device('cuda', torch.cuda.current_device())
        self.device = torch.device(device)
        f32 = torch.float32
        self.obs = torch.zeros((self.max_size, obs_dim), dtype=f32, device=self.device)
        if act_dim == 0:
            self.action = torch.zeros((self.max_size, 1), dtype=torch.int32, device=self.device)
        else:
            self.action = torch.zeros((self.max_size, act_dim), dtype=f32, device=self.device)
        self.reward = torch.zeros((self.max_size, 1), dtype=f32, device=self.device)
        self.terminal = torch.zeros((self.max_size, 1), dtype=torch.int32, device=self.device)   # bool widened to 4 B rows
        self.next_obs = torch.zeros((self.max_size, obs_dim), dtype=f32, device=self.device)
        self._curr_size = 0
        self._curr_pos = 0

    # ---- writes -----------------------------------------------------------------------------------------
    def append(self, obs, act, reward, next_obs, terminal):
        p = self._curr_pos
        self.obs[p] = torch.as_tensor(np.asarray(obs, np.float32))
        self.action[p] = torch.as_tensor(np.asarray(act)).to(self.action.dtype).reshape(-1)
        self.reward[p, 0] = float(reward)
        self.next_obs[p] = torch.as_tensor(np.asarray(next_obs, np.float32))
        self.terminal[p, 0] = int(bool(terminal))
        self._curr_size = min(self._curr_size + 1, self.max_size)
        self._curr_pos = (p + 1) % self.max_size

    def append_batch(self, obs, act, reward, next_obs, terminal):
        """Vectorised append of n transitions already on the device (the on-device actor pool path)."""
        n = obs.shape[0]
        idx = (torch.arange(n, device=self.device) + self._curr_pos) % self.max_size
        self.obs[idx] = obs.to(torch.float32)
        self.action[idx] = act.reshape(n, -1).to(self.action.dtype)
        self.reward[idx] = reward.reshape(n, 1).to(torch.float32)
        self.next_obs[idx] = next_obs.to(torch.float32)
        self.terminal[idx] = terminal.reshape(n, 1).to(torch.int32)
        self._curr_size = min(self._curr_size + n, self.max_size)
        self._curr_pos = (self._curr_pos + n) % self.max_size

    def commit(self, n):
        """Account for n rows a device kernel wrote in place from the current position on (rl_explore_mlp): the same
        bookkeeping as ``append_batch`` of n transitions."""
        n = int(n)
        if n < 0 or n > self.max_size:
            raise ValueError('ReplayMemory.commit: n=%d outside 0..%d' % (n, self.max_size))
        self._curr_size = min(self._curr_size + n, self.max_size)
        self._curr_pos = (self._curr_pos + n) % self.max_size

    # ---- reads ------------------------------------------------------------------------------------------
    def make_index(self, batch_size):
        return np.random.randint(self._curr_size, size=batch_size)

    def sample_batch_by_index(self, batch_idx, as_tensor=False):
        idx = torch.as_tensor(np.asarray(batch_idx), dtype=torch.int32).to(self.device)
        obs = kernels.gather_rows(self.obs, idx)
        action = kernels.gather_rows(self.action, idx)
        reward = kernels.gather_rows(self.reward, idx).reshape(-1)
        next_obs = kernels.gather_rows(self.next_obs, idx)
        terminal = kernels.gather_rows(self.terminal, idx).reshape(-1) != 0
        if self.act_dim == 0:
            action = action.reshape(-1)
        if as_tensor:
            return obs, action, reward, next_obs, terminal
        return tuple(t.cpu().numpy() for t in (obs, action, reward, next_obs, terminal))

    def sample_batch(self, batch_size, as_tensor=False):
        return self.sample_batch_by_index(self.make_index(batch_size), as_tensor=as_tensor)

    def size(self):
        return self._curr_size

    def __len__(self):
        return self._curr_size

    # ---- persistence (same keys as replay_memory.py:119-147) ----------------------------------------------
    def save(self, pathname):
        n = self._curr_size
        other = np.array([self._curr_size, self._curr_pos], dtype=np.int32)
        act = self.action[:n].cpu().numpy()
        np.savez(pathname, obs=self.obs[:n].cpu().numpy(), action=act.reshape(-1) if self.act_dim == 0 else act,
                 reward=self.reward[:n, 0].cpu().numpy(), terminal=self.terminal[:n, 0].cpu().numpy().astype(bool),
                 next_obs=self.next_obs[:n].cpu().numpy(), other=other)

    def load(self, pathname):
        data = np.load(pathname)
        other = data['other']
        n = min(int(other[0]), self.max_size)
        self._curr_size = n
        self._curr_pos = min(int(other[1]), self.max_size - 1)
        self.obs[:n] = torch.as_tensor(data['obs'][:n])
        self.action[:n] = torch.as_tensor(data['action'][:n]).reshape(n, -1).to(self.action.dtype)
        self.reward[:n, 0] = torch.as_tensor(data['reward'][:n])
        self.terminal[:n, 0] = torch.as_tensor(data['terminal'][:n].astype(np.int32))
        self.next_obs[:n] = torch.as_tensor(data['next_obs'][:n])
