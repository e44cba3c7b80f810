"""Forking envs of a vector env: copy the whole state of chosen envs onto other envs (sampling-based planning,
population-based restarts, evaluation from a common state)."""
from .. import _native as nat


class ForkableVectorEnv:
    """Base of the vector envs: `copy_envs` over the handle's sr_copy_envs and the class's per-env host state, the
    tensors named in PER_ENV (dim 0 = env)."""

    PER_ENV = ()

    def copy_envs(self, dst_idx, src_idx, src=None):
        """Env dst_idx[i] takes the whole state of env src_idx[i] of `src` (a vector env of the same class and
        configuration; default: this one): the handle's per-env device buffers (Handle.copy_envs) and the host-side
        episode bookkeeping (step counts, previous actions and observations, targets).  Every source is read before
        any destination is written, so permutations and swaps work; destinations must be distinct.  The destination
        then continues bit for bit like its source under the same actions.

        A fork copies an env's physical state and episode, not its seed identity: what a later autoreset draws for a
        destination is what this vector env draws for that index, not what the source's would.

        Indices: ints, sequences, NumPy arrays or torch tensors.  ValueError on unequal lengths, out-of-range indices,
        duplicate destinations, a `src` of another class or shape, or a vector env that has not been reset yet (some
        keep per-env state from their first reset on)."""
        import torch
        src = self if src is None else src
        if type(src) is not type(self):
            raise ValueError(f"copy_envs: src is a {type(src).__name__}, not a {type(self).__name__}")
        missing = [n for n in self.PER_ENV if not (hasattr(self, n) and hasattr(src, n))]
        if missing:
            raise ValueError(f"copy_envs: {', '.join(missing)} not set yet: reset() both vector envs first")
        for name in self.PER_ENV:
            a, b = getattr(self, name), getattr(src, name)
            if a.shape[1:] != b.shape[1:] or a.dtype != b.dtype:
                raise ValueError(f"copy_envs: {name} is {tuple(b.shape[1:])} {b.dtype} per env in src, "
                                 f"{tuple(a.shape[1:])} {a.dtype} here")
        self._check_copy_source(src)
        d, s = nat.copy_env_indices(dst_idx, src_idx, self.n_env, src.n_env)
        self.handle.copy_envs(d, s, src.handle)
        if d.size == 0:
            return
        di, si = torch.as_tensor(d, device=self.device), torch.as_tensor(s, device=src.device)
        for name in self.PER_ENV:
            # a new tensor rather than an update in place: a previous action may be the caller's own action tensor
            t = getattr(self, name).clone()
            t[di] = getattr(src, name)[si].to(t.device)
            setattr(self, name, t)

    def _check_copy_source(self, src):
        """Raise ValueError when envs of `src` cannot continue in this vector env (class-specific)."""
