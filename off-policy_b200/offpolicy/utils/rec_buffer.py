"""Drop-in `offpolicy.utils.rec_buffer` backed by the HBM-resident replay of libmarl_b200.

Same public surface as /root/reference/offpolicy/utils/rec_buffer.py (constructor arguments,
`insert`, `sample`, `update_priorities`, `__len__`, `policy_buffers[p_id].filled_i/current_i`),
so `offpolicy/runner/rnn/base_runner.py:7,162-178,266-275` runs unchanged.  What differs is where
the data lives: every field is an episode-major SoA in device memory; `sample` launches the index
draw + 128-bit gather kernels and returns a 9-tuple whose entries are *lazy* views -- the B200
trainers consume the device-side batch directly, while indexing an entry (`obs['policy_0']`)
materialises the reference's NumPy layout on demand.

Index streams (SURVEY.md App. C):
  * default `rng="numpy"`: indices / PER masses are drawn on the host from NumPy's process-global
    legacy stream with the reference's own calls (np.random.choice / np.random.random), so a run
    seeded like the reference stays bit-identical even though the env shares the stream;
  * `rng="device"`: a device-resident copy of the MT19937 state (seed_device_rng / adopt_numpy_rng)
    is advanced by the sample kernel itself -- no host work per step (used by the CUDA-graph loop).
"""
import ctypes as C

import numpy as np
import torch

from offpolicy._b200 import capi

FIELDS = ("obs", "share_obs", "acts", "rewards", "dones", "dones_env", "avail_acts")


def _space_dim(space):
    """obs/share/act space -> flat width; accepts gym Box/Discrete look-alikes and SMAC's `[dim]` lists
    (reference: utils/util.py:230-243, rec_buffer.py:111-118)."""
    if isinstance(space, (list, tuple)):
        return int(space[0])
    name = space.__class__.__name__
    if name == "Box":
        return int(space.shape[0])
    if name == "Discrete":
        return int(space.n)
    if "MultiDiscrete" in name:
        return int(np.sum(np.asarray(space.high) - np.asarray(space.low) + 1))
    raise NotImplementedError("Unrecognized space: %r" % (space,))


class DeviceArray(object):
    """A small device-resident result (indices, priorities, importance weights) that behaves like an
    ndarray when the caller insists (`np.asarray`, len, indexing) but stays on the GPU between the trainer
    and the buffer."""

    def __init__(self, tensor):
        self.tensor = tensor

    def __array__(self, dtype=None, copy=None):
        a = self.tensor.detach().cpu().numpy()
        return a.astype(dtype) if dtype is not None else a

    def __len__(self):
        return int(self.tensor.shape[0])

    def __getitem__(self, i):
        return np.asarray(self)[i]

    def numpy(self):
        return np.asarray(self)


class _LazyField(dict):
    """dict {p_id: ndarray} that materialises the reference layout from the device batch on first access."""

    def __init__(self, owner, field, p_ids):
        super().__init__()
        self._owner, self._field, self._p_ids = owner, field, tuple(p_ids)

    def __missing__(self, p_id):
        if p_id not in self._p_ids:
            raise KeyError(p_id)
        val = self._owner.materialize(p_id, self._field)
        self[p_id] = val
        return val

    def keys(self):
        return self._p_ids

    def __iter__(self):
        return iter(self._p_ids)

    def __len__(self):
        return len(self._p_ids)

    def __contains__(self, k):
        return k in self._p_ids


class SampledBatch(object):
    """The reference's 9-tuple (rec_buffer.py:82,304) + a handle on the device-side batch.  Behaves like the tuple (len 9,
    indexing, unpacking); the seven field entries are created on first access (a B200 trainer never touches them)."""

    __slots__ = ("buffers", "B", "serial", "_p_ids", "_items")

    def __init__(self, buffers, B, weights, idxes, p_ids):
        self.buffers = buffers
        self.B = B
        self._p_ids = p_ids
        self.serial = {p: buffers[p].sample_serial for p in p_ids}
        self._items = [None] * 7 + [weights, idxes]

    def __len__(self):
        return 9

    def __getitem__(self, i):
        if isinstance(i, slice):
            return tuple(self[k] for k in range(*i.indices(9)))
        if i < 0:
            i += 9
        v = self._items[i]
        if v is None and i < 7:
            v = self._items[i] = _LazyField(self, FIELDS[i], self._p_ids)
        return v

    def __iter__(self):
        return (self[k] for k in range(9))

    def materialize(self, p_id, field):
        buf = self.buffers[p_id]
        if buf.sample_serial != self.serial[p_id]:
            raise RuntimeError("this sample was overwritten by a later sample() call (the device batch region is reused)")
        return buf.materialize(field, self.B)


class RecPolicyBuffer(object):
    """One policy's episode store (rec_buffer.py:85-240) in device memory."""

    DEFAULT_MAX_BATCH = 128

    def __init__(self, buffer_size, episode_length, num_agents, obs_space, share_obs_space, act_space,
                 use_same_share_obs, use_avail_acts, use_reward_normalization=False, use_per=False, per_alpha=0.0,
                 max_batch=None):
        if not use_same_share_obs:
            raise NotImplementedError("B200 replay stores one centralised observation per step (use_same_share_obs=True)")
        self.buffer_size = int(buffer_size)
        self.episode_length = int(episode_length)
        self.num_agents = int(num_agents)
        self.use_same_share_obs = use_same_share_obs
        self.use_avail_acts = bool(use_avail_acts)
        self.use_reward_normalization = bool(use_reward_normalization)
        self.obs_dim = _space_dim(obs_space)
        self.share_dim = _space_dim(share_obs_space)
        self.act_dim = _space_dim(act_space)
        self.max_batch = int(max_batch or self.DEFAULT_MAX_BATCH)
        self.sample_serial = 0

        lib = capi.lib()
        self.dev = capi.device()
        cfg = capi.ReplayCfg(self.buffer_size, self.episode_length, self.num_agents, self.obs_dim, self.share_dim, self.act_dim,
                             int(self.use_avail_acts), int(bool(use_per)), int(self.use_reward_normalization), self.max_batch,
                             float(per_alpha))
        self.cfg = cfg
        self.L = capi.ReplayLayout()
        capi.check(lib.mx_replay_layout_query(C.byref(cfg), C.byref(self.L)))
        self.blob = torch.zeros(int(self.L.total_bytes), dtype=torch.uint8, device=self.dev)
        h = C.c_void_p()
        capi.check(lib.mx_replay_create(C.byref(cfg), capi.ptr(self.blob), capi.stream_ptr(), C.byref(h)))
        self.handle = h
        self._lib = lib         # the library that made the handle frees it, even if another build is bound by the time this is collected
        self._stage = [None, None]
        self._stage_evt = [None, None]
        self._stage_i = 0
        self._pack_cache = {}
        self._view_cache = {}
        self._first_slot = C.c_int32()
        self._idx_dev = torch.zeros(self.max_batch, dtype=torch.int64, device=self.dev)
        self._idx_pin = None
        self._idx_ring, self._idx_k = None, 0

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self._lib.mx_replay_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # -- reference attributes -------------------------------------------------------------------
    @property
    def filled_i(self):
        return int(capi.lib().mx_replay_len(self.handle))

    @property
    def current_i(self):
        return int(capi.lib().mx_replay_cursor(self.handle))

    def __len__(self):
        return self.filled_i

    # -- views into the blob ----------------------------------------------------------------------
    def _view(self, off, count, dtype):
        nbytes = count * torch.empty((), dtype=dtype).element_size()
        return self.blob[off:off + nbytes].view(dtype)

    def _field_view(self, field, batch, n):
        L, T, N = self.L, self.episode_length, self.num_agents
        pre = "off_b_" if batch else "off_"
        spec = {
            "obs": (pre + "obs", L.ep_obs, (T + 1, N, L.obs_ld), self.obs_dim),
            "share_obs": (pre + "share", L.ep_share, (T + 1, L.share_ld), self.share_dim),
            "acts": (pre + "acts", L.ep_acts, (T, N, L.act_ld), self.act_dim),
            "avail_acts": (pre + "avail", L.ep_avail, (T + 1, N, L.act_ld), self.act_dim),
            "rewards": (pre + "rew", L.ep_rew, None, T * N),
            "dones": (pre + "dones", L.ep_dones, None, T * N),
            "dones_env": (pre + "dones_env", L.ep_dones_env, None, T),
        }[field]
        off, ep, shape, width = getattr(L, spec[0]), spec[1], spec[2], spec[3]
        flat = self._view(off, n * ep, torch.float32).view(n, ep)
        if shape is None:
            return flat[:, :width]
        return flat.view((n,) + shape)[..., :width]

    def materialize(self, field, B):
        """Reference layout of one sampled field (rec_buffer.py:192-240): agent-major (N, T[+1], B, D)."""
        T, N = self.episode_length, self.num_agents
        if field == "avail_acts" and not self.use_avail_acts:
            return None
        v = self._field_view(field, True, B)
        if field in ("obs", "acts", "avail_acts"):
            out = v.permute(2, 1, 0, 3)
        elif field == "share_obs":
            out = v.permute(1, 0, 2)
        elif field in ("rewards", "dones"):
            out = v.reshape(B, T, N).permute(2, 1, 0).unsqueeze(-1)
        else:
            out = v.reshape(B, T).permute(1, 0).unsqueeze(-1)
        return out.contiguous().cpu().numpy()

    # -- insert -----------------------------------------------------------------------------------
    def _staging(self, nbytes):
        i = self._stage_i
        self._stage_i ^= 1
        if self._stage_evt[i] is not None:
            capi.check(capi.lib().mx_host_fence_wait(self._stage_evt[i]))
        if self._stage[i] is None or self._stage[i].numel() < nbytes:
            pin = self.dev.type == "cuda"
            self._stage[i] = torch.empty(int(nbytes * 1.25) + 1024, dtype=torch.uint8, pin_memory=pin)
        return i, self._stage[i]

    def _packed_layout(self, n_ep):
        lay = self._pack_cache.get(n_ep)
        if lay is None:
            offs, cnts = (C.c_int64 * 7)(), (C.c_int64 * 7)()
            total = int(capi.lib().mx_replay_insert_packed_layout(self.handle, n_ep, offs, cnts))
            lay = (list(offs), list(cnts), total)
            self._pack_cache[n_ep] = lay
        return lay

    def _stage_views(self, si, stage, n_ep):
        """float32 views of staging buffer `si`, one per field of an n_ep-episode insert (cached: the pinned buffers are reused)."""
        key = (si, n_ep, stage.data_ptr())
        v = self._view_cache.get(key)
        if v is None:
            offs, cnts, total = self._packed_layout(n_ep)
            host = stage.numpy()
            T, N = self.episode_length, self.num_agents
            shapes = [(T + 1, n_ep, N, self.obs_dim), (T + 1, n_ep, self.share_dim), (T, n_ep, N, self.act_dim), (T, n_ep, N, 1),
                      (T, n_ep, N, 1), (T, n_ep, 1), (T + 1, n_ep, N, self.act_dim)]
            v = [host[o:o + 4 * n].view(np.float32).reshape(sh) if n else None for o, n, sh in zip(offs, cnts, shapes)]
            self._view_cache = {k: w for k, w in self._view_cache.items() if k[0] != si or k[2] == stage.data_ptr()}
            self._view_cache[key] = v
        return v

    def insert(self, num_insert_episodes, obs, share_obs, acts, rewards, dones, dones_env, avail_acts=None):
        n_ep = int(num_insert_episodes)
        acts = np.asarray(acts)
        assert acts.shape[0] == self.episode_length, ("different dimension!")            # rec_buffer.py:165
        if n_ep > self.max_batch:
            raise ValueError("insert of %d episodes exceeds max_batch=%d" % (n_ep, self.max_batch))
        share_obs = np.asarray(share_obs)
        if share_obs.ndim == 4:
            share_obs = share_obs[:, :, 0]                                               # rec_buffer.py:173-175
        arrs = (obs, share_obs, acts, rewards, dones, dones_env, avail_acts if self.use_avail_acts else None)
        total = self._packed_layout(n_ep)[2]
        si, stage = self._staging(total)
        for a, view in zip(arrs, self._stage_views(si, stage, n_ep)):
            if view is not None:
                a = np.asarray(a)
                if a.size != view.size:
                    raise ValueError("insert: a field has %d elements, expected %d" % (a.size, view.size))
                np.copyto(view, a.reshape(view.shape), casting="same_kind")      # one (possibly strided) pass into pinned memory
        first = self._first_slot
        capi.check(capi.lib().mx_replay_insert_packed_async(self.handle, C.c_void_p(stage.data_ptr()), total, n_ep, C.byref(first),
                                                            capi.stream_ptr()))
        if self.dev.type == "cuda":           # the staging block may be rewritten once this copy has been consumed (library-side event: ~1 us)
            if self._stage_evt[si] is None:
                self._stage_evt[si] = capi.lib().mx_host_fence_alloc()
            capi.check(capi.lib().mx_host_fence_record(self._stage_evt[si], capi.stream_ptr()))
        return (first.value + np.arange(n_ep)) % self.buffer_size

    # -- sampling -----------------------------------------------------------------------------------
    def upload_indices(self, inds):
        inds = np.ascontiguousarray(inds, dtype=np.int64)
        B = inds.shape[0]
        if self.dev.type == "cuda":
            if self._idx_pin is None:
                self._idx_pin = torch.empty(self.max_batch, dtype=torch.int64, pin_memory=True)
            self._idx_pin[:B].numpy()[:] = inds
            self._idx_dev[:B].copy_(self._idx_pin[:B], non_blocking=True)
        else:
            self._idx_dev[:B] = torch.from_numpy(inds)
        return self._idx_dev

    def gather(self, inds):
        B = len(inds)
        if B > self.max_batch:
            raise ValueError("batch_size %d exceeds max_batch=%d (pass max_batch= to the buffer)" % (B, self.max_batch))
        if self.dev.type == "cuda":
            # indices go through a small pinned ring; a slot is rewritten only after the H2D copy that read it has completed
            if self._idx_ring is None:
                self._idx_ring = [torch.empty(self.max_batch, dtype=torch.int64, pin_memory=True) for _ in range(4)]
                self._idx_ring_np = [t.numpy() for t in self._idx_ring]
                self._idx_ring_ptr = [C.c_void_p(t.data_ptr()) for t in self._idx_ring]
                self._idx_ring_evt = [None] * 4
            k = self._idx_k
            self._idx_k = (k + 1) & 3
            lib, sp = capi.lib(), capi.stream_ptr()
            if self._idx_ring_evt[k] is not None:
                capi.check(lib.mx_host_fence_wait(self._idx_ring_evt[k]))
            else:
                self._idx_ring_evt[k] = lib.mx_host_fence_alloc()
            self._idx_ring_np[k][:B] = inds
            capi.check(lib.mx_replay_gather_host(self.handle, self._idx_ring_ptr[k], B, sp))
            capi.check(lib.mx_host_fence_record(self._idx_ring_evt[k], sp))
        else:
            dev = self.upload_indices(inds)
            capi.check(capi.lib().mx_replay_gather(self.handle, capi.ptr(dev), B, capi.stream_ptr()))
        self.sample_serial += 1

    def sample_device_uniform(self, B):
        capi.check(capi.lib().mx_replay_sample_uniform(self.handle, int(B), capi.stream_ptr()))
        self.sample_serial += 1

    def sample_device_per(self, B, beta):
        capi.check(capi.lib().mx_replay_sample_per(self.handle, int(B), float(beta), capi.stream_ptr()))
        self.sample_serial += 1

    def gather_device(self, idx_dev, B):
        """Gather the episodes whose indices another policy's buffer has just drawn (device int64 tensor): with several policies the
        reference draws ONE index set and applies it to every policy's store (rec_buffer.py:76-80, 291-299)."""
        capi.check(capi.lib().mx_replay_gather(self.handle, capi.ptr(idx_dev), int(B), capi.stream_ptr()))
        self.sample_serial += 1

    def batch_struct(self, B):
        b = capi.Batch()
        capi.check(capi.lib().mx_replay_batch(self.handle, int(B), C.byref(b)))
        return b

    def sampled_indices(self, B):
        return DeviceArray(self._view(self.L.off_b_idx, B, torch.int64))

    def sampled_weights(self, B):
        return DeviceArray(self._view(self.L.off_b_weights, B, torch.float64))

    # -- device RNG -----------------------------------------------------------------------------------
    def seed_device_rng(self, seed):
        capi.check(capi.lib().mx_replay_seed(self.handle, int(seed) & 0xFFFFFFFF, capi.stream_ptr()))

    def adopt_numpy_rng(self):
        st = np.random.get_state()
        key = (C.c_uint32 * 624)(*[int(v) for v in st[1]])
        self._np_gauss = (int(st[3]), float(st[4]))       # NumPy's cached second Gaussian of a pair: not part of the MT19937 key, handed back on export
        capi.check(capi.lib().mx_replay_set_rng_state(self.handle, key, int(st[2]), capi.stream_ptr()))

    def export_rng_to_numpy(self):
        key = (C.c_uint32 * 624)()
        pos = C.c_int32()
        capi.check(capi.lib().mx_replay_get_rng_state(self.handle, key, C.byref(pos), capi.stream_ptr()))
        has_gauss, cached = getattr(self, "_np_gauss", (0, 0.0))
        np.random.set_state(("MT19937", np.array(list(key), dtype=np.uint32), int(pos.value), has_gauss, cached))

    # -- checkpoint / resume (SURVEY.md 8(f).3: the reference checkpoints network weights only) -------------
    def state_dict(self):
        """Everything the replay is: the device blob holds the episodes, the PER trees, the device MT19937 key and the ring
        position and the running reward statistics.  Only that persistent part is saved (the sampled-batch region and the insert
        staging area behind it are scratch)."""
        if self.dev.type == "cuda":
            torch.cuda.current_stream(self.dev).synchronize()
        n = int(self.L.off_b_obs)
        return {"blob": self.blob[:n].cpu().clone(), "shape": self._shape_key()}

    def _shape_key(self):
        c = self.cfg
        return [int(getattr(c, f)) for f in ("capacity", "episode_len", "n_agents", "obs_dim", "share_dim", "act_dim", "use_avail", "use_per",
                                             "reward_norm")]

    def load_state_dict(self, sd):
        if list(sd["shape"]) != self._shape_key():
            raise ValueError("replay checkpoint has shape %s, this buffer %s" % (list(sd["shape"]), self._shape_key()))
        blob = torch.as_tensor(sd["blob"])
        n = int(self.L.off_b_obs)
        if blob.numel() != n:
            raise ValueError("replay checkpoint holds %d bytes, expected %d" % (blob.numel(), n))
        self.blob[:n].copy_(blob.to(self.dev))
        capi.check(capi.lib().mx_replay_restore(self.handle, capi.stream_ptr()))
        self.sample_serial += 1          # any batch sampled before the restore is stale

    # -- PER --------------------------------------------------------------------------------------------
    def tree_values(self):
        n = 2 * int(self.L.tree_cap)
        return (self._view(self.L.off_sum_tree, n, torch.float64).cpu().numpy(),
                self._view(self.L.off_min_tree, n, torch.float64).cpu().numpy())

    def update_priorities(self, idxes, priorities=None, leaves=None):
        dev = self.dev
        if isinstance(idxes, DeviceArray):
            idx_t = idxes.tensor
        else:
            idx_np = np.ascontiguousarray(idxes, dtype=np.int64)
            assert np.min(idx_np) >= 0                                                       # rec_buffer.py:317
            assert np.max(idx_np) < len(self)                                                # rec_buffer.py:318
            idx_t = torch.from_numpy(idx_np).to(dev)
        B = int(idx_t.shape[0])
        pr_t = lv_t = None
        if leaves is not None:
            lv_t = torch.as_tensor(np.ascontiguousarray(leaves, dtype=np.float64)).to(dev)
        elif isinstance(priorities, DeviceArray):
            pr_t = priorities.tensor
        else:
            pr_np = np.ascontiguousarray(priorities, dtype=np.float32)
            assert len(pr_np) == B                                                           # rec_buffer.py:315
            assert np.min(pr_np) > 0                                                         # rec_buffer.py:316
            pr_t = torch.from_numpy(pr_np).to(dev)
        capi.check(capi.lib().mx_replay_update_priorities(self.handle, capi.ptr(idx_t), capi.ptr(pr_t), capi.ptr(lv_t), None, B,
                                                          capi.stream_ptr()))
        self._keep = (idx_t, pr_t, lv_t)   # keep alive until the stream has consumed them


class RecReplayBuffer(object):
    """Uniform episode replay (rec_buffer.py:10-82)."""

    def __init__(self, policy_info, policy_agents, buffer_size, episode_length, use_same_share_obs, use_avail_acts,
                 use_reward_normalization=False, rng="numpy", max_batch=None, _per_alpha=None):
        self.policy_info = policy_info
        self.rng = rng
        self.policy_buffers = {
            p_id: RecPolicyBuffer(buffer_size, episode_length, len(policy_agents[p_id]), policy_info[p_id]["obs_space"],
                                  policy_info[p_id]["share_obs_space"], policy_info[p_id]["act_space"], use_same_share_obs,
                                  use_avail_acts, use_reward_normalization, use_per=_per_alpha is not None,
                                  per_alpha=_per_alpha or 0.0, max_batch=max_batch)
            for p_id in self.policy_info.keys()}

    def _first(self):
        return self.policy_buffers["policy_0"] if "policy_0" in self.policy_buffers else next(iter(self.policy_buffers.values()))

    def __len__(self):
        return self._first().filled_i                  # rec_buffer.py:54-55 (every policy's store holds the same episodes)

    def insert(self, num_insert_episodes, obs, share_obs, acts, rewards, dones, dones_env, avail_acts):
        idx_range = None
        for p_id in self.policy_info.keys():
            av = None if avail_acts is None or avail_acts[p_id] is None else avail_acts[p_id]
            idx_range = self.policy_buffers[p_id].insert(num_insert_episodes, obs[p_id], share_obs[p_id], acts[p_id],
                                                         rewards[p_id], dones[p_id], dones_env[p_id], av)
        return idx_range

    def seed_device_rng(self, seed):
        self.rng = "device"
        for b in self.policy_buffers.values():
            b.seed_device_rng(seed)

    def state_dict(self):
        return {"rng": self.rng, "policy_buffers": {p: b.state_dict() for p, b in self.policy_buffers.items()}}

    def load_state_dict(self, sd):
        self.rng = sd["rng"]
        for p, b in self.policy_buffers.items():
            b.load_state_dict(sd["policy_buffers"][p])

    def adopt_numpy_rng(self):
        self.rng = "device"
        for b in self.policy_buffers.values():
            b.adopt_numpy_rng()

    def sample(self, batch_size):
        p_ids = list(self.policy_info.keys())
        buf = self._first()
        if self.rng == "device":
            buf.sample_device_uniform(batch_size)
            for other in self.policy_buffers.values():      # several policies: ONE index set for every policy's store (rec_buffer.py:76-80)
                if other is not buf:
                    other.gather_device(buf.sampled_indices(batch_size).tensor, batch_size)
        else:
            # rec_buffer.py:76 draws np.random.choice(len, B); randint(0, len, B) is the same call underneath (same masked-rejection
            # draws from the global MT19937 stream, same int64 result: tests/test_oracle_rng.py) without choice()'s argument checks
            inds = np.random.randint(0, self.__len__(), batch_size)
            for b in self.policy_buffers.values():
                b.gather(inds)
        return SampledBatch(self.policy_buffers, batch_size, None, None, p_ids)


class PrioritizedRecReplayBuffer(RecReplayBuffer):
    """Proportional prioritised episode replay (rec_buffer.py:243-324); fp64 trees live on the device."""

    def __init__(self, alpha, policy_info, policy_agents, buffer_size, episode_length, use_same_share_obs, use_avail_acts,
                 use_reward_normalization=False, rng="numpy", max_batch=None):
        super().__init__(policy_info, policy_agents, buffer_size, episode_length, use_same_share_obs, use_avail_acts,
                         use_reward_normalization, rng=rng, max_batch=max_batch, _per_alpha=float(alpha))
        self.alpha = alpha

    def sample(self, batch_size, beta=0, p_id=None):
        assert len(self) > batch_size, "Cannot sample with no completed episodes in the buffer!"   # rec_buffer.py:287
        assert beta > 0                                                                              # rec_buffer.py:289
        buf = self.policy_buffers[p_id] if p_id else self._first()
        if self.rng != "device":
            # host draw keeps the process-global NumPy stream shared with the env (np.random.random, rec_buffer.py:274)
            buf.adopt_numpy_rng()
            buf.sample_device_per(batch_size, beta)
            buf.export_rng_to_numpy()
        else:
            buf.sample_device_per(batch_size, beta)
        for other in self.policy_buffers.values():          # the indices drawn from p_id's tree select the episodes of EVERY policy (rec_buffer.py:291-299)
            if other is not buf:
                other.gather_device(buf.sampled_indices(batch_size).tensor, batch_size)
        return SampledBatch(self.policy_buffers, batch_size, buf.sampled_weights(batch_size), buf.sampled_indices(batch_size),
                            list(self.policy_info.keys()))

    def update_priorities(self, idxes, priorities, p_id=None):
        (self.policy_buffers[p_id] if p_id else self._first()).update_priorities(idxes, priorities)
