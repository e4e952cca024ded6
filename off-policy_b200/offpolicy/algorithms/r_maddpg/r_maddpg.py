"""Drop-in `R_MADDPG` trainer (reference: offpolicy/algorithms/r_maddpg/r_maddpg.py) on the sm_100a learner.

`shared_train_policy_on_batch(p_id, batch)` = one `mx_maddpg_step`: target-actor next actions, critic sequence + target
branch steps, TD target, critic loss/backward/Adam, then (every `actor_update_interval`-th call) the actor update through
the updated critic -- all on the device.  MATD3's Gaussian target-action noise is drawn on the host with the reference's
own call (`torch.empty(shape).normal_`, utils/util.py:217-218) so a seeded run consumes torch's CPU RNG identically; for
Discrete actors the Gumbel draws of the target actions (MATD3) and of the actor update (`use_gumbel=True`, r_maddpg.py:277) are
drawn the same way (utils/util.py:127-130), in the reference's order.
`cent_train_policy_on_batch` (per-agent centralised observations) is unusable in the reference (SURVEY.md App. D-7) and is not built."""
import ctypes as C

import numpy as np
import torch

from offpolicy._b200 import capi
from offpolicy.algorithms.r_maddpg.algorithm.rMADDPGPolicy import maddpg_cfg_struct, sample_gumbel
from offpolicy.utils.rec_buffer import SampledBatch, DeviceArray


class _HostBatchC(object):
    """Device copy of a reference-layout NumPy batch."""

    def __init__(self, cfg, dev):
        B, T, N = cfg.max_batch, cfg.episode_len, cfg.n_agents
        r4 = lambda v: (v + 3) // 4 * 4
        self.cfg = cfg
        self.obs_ld, self.share_ld, self.act_ld = r4(cfg.obs_dim), r4(cfg.state_dim), r4(cfg.act_dim)
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)
        self.obs, self.share, self.acts = z(B, T + 1, N, self.obs_ld), z(B, T + 1, self.share_ld), z(B, T, N, self.act_ld)
        self.rew, self.dones, self.dones_env, self.weights = z(B, T, N), z(B, T, N), z(B, T), z(B)
        self.avail = None
        self.dev = dev

    def pack(self, batch, p_id, use_per):
        obs, share, acts, rew, dones, dones_env, _avail, weights, _idx = batch
        c = self.cfg
        t = lambda x: torch.as_tensor(np.asarray(x), dtype=torch.float32).to(self.dev)
        o = t(obs[p_id])
        B = o.shape[2]
        self.obs[:B, :, :, :c.obs_dim] = o.permute(2, 1, 0, 3)
        self.share[:B, :, :c.state_dim] = t(share[p_id]).permute(1, 0, 2)
        self.acts[:B, :, :, :c.act_dim] = t(acts[p_id]).permute(2, 1, 0, 3)
        self.rew[:B] = t(rew[p_id])[..., 0].permute(2, 1, 0)
        self.dones[:B] = t(dones[p_id])[..., 0].permute(2, 1, 0)
        self.dones_env[:B] = t(dones_env[p_id])[..., 0].permute(1, 0)
        if use_per:
            self.weights[:B] = t(weights)
        has_avail = _avail is not None and _avail.get(p_id) is not None
        if has_avail:
            if self.avail is None:
                self.avail = torch.ones(c.max_batch, c.episode_len + 1, c.n_agents, self.act_ld, dtype=torch.float32, device=self.dev)
            self.avail[:B, :, :, :c.act_dim] = t(_avail[p_id]).permute(2, 1, 0, 3)
        b = capi.Batch()
        b.B, b.obs_ld, b.share_ld, b.act_ld = B, self.obs_ld, self.share_ld, self.act_ld
        b.obs, b.share, b.acts = self.obs.data_ptr(), self.share.data_ptr(), self.acts.data_ptr()
        b.rewards, b.dones, b.dones_env = self.rew.data_ptr(), self.dones.data_ptr(), self.dones_env.data_ptr()
        b.weights = self.weights.data_ptr() if use_per else None
        b.avail = self.avail.data_ptr() if has_avail else None
        return b


class _Engine(object):
    """One policy's learner: its mx_maddpg handle + workspace views."""

    def __init__(self, args, pol, n_agents, episode_length, max_batch, actor_update_interval, cent_act_dim, act_offset):
        lib = capi.lib()
        self.dev = capi.device()
        self.pol, self.n_agents = pol, n_agents
        self.cfg = maddpg_cfg_struct(args, n_agents, pol.obs_dim, pol.act_dim, pol.central_obs_dim, episode_length, max_batch,
                                     pol.td3, pol.target_noise if pol.td3 else 0.0, actor_update_interval, pol.discrete,
                                     cent_act_dim=cent_act_dim, act_offset=act_offset)
        nbytes = int(lib.mx_maddpg_workspace_bytes(C.byref(self.cfg)))
        if nbytes < 0:
            raise capi.MxError(lib.mx_last_error().decode())
        self.workspace = torch.zeros(nbytes, dtype=torch.uint8, device=self.dev)
        av = (C.c_void_p * 4)(*[v.data_ptr() for v in pol.actor_vecs])
        cv = (C.c_void_p * 4)(*[v.data_ptr() for v in pol.critic_vecs])
        h = C.c_void_p()
        capi.check(lib.mx_maddpg_create(C.byref(self.cfg), av, cv, capi.ptr(self.workspace), nbytes, C.byref(h)))
        self.handle = h
        self._lib = lib         # the library that made the handle frees it, whichever build is bound later
        ip = lib.mx_maddpg_info(self.handle) - self.workspace.data_ptr()
        self.info = self.workspace[ip:ip + 32].view(torch.float32)
        pp = lib.mx_maddpg_priorities(self.handle) - self.workspace.data_ptr()
        self.prio = self.workspace[pp:pp + 4 * max_batch].view(torch.float32)
        self.host_batch = None
        self.noise_dev = None
        self.actor_noise_dev = None

    def close(self):
        if self.handle:
            self._lib.mx_maddpg_destroy(self.handle)
            self.handle = None


class R_MADDPG(object):
    def __init__(self, args, num_agents, policies, policy_mapping_fn, device=None, episode_length=None, actor_update_interval=1):
        self.args = args
        self.use_per = args.use_per
        if getattr(args, "use_popart", False):
            raise NotImplementedError("B200 R-MADDPG path: --use_popart is not implemented (the reference's PopArt target is used only there)")
        self.num_agents = num_agents
        self.policies = policies
        self.policy_mapping_fn = policy_mapping_fn
        self.policy_ids = sorted(list(self.policies.keys()))
        self.policy_agents = {p: sorted(a for a in range(num_agents) if policy_mapping_fn(a) == p) for p in self.policies}
        self.episode_length = args.episode_length if episode_length is None else episode_length
        self.actor_update_interval = actor_update_interval
        self.num_updates = {p: 0 for p in self.policy_ids}
        self.use_same_share_obs = getattr(args, "use_same_share_obs", True)
        self.max_batch = int(getattr(args, "batch_size", 32))
        self.dev = capi.device()
        # one shared policy ('policy_0' for every agent): the single-learner layout; several policies (config.py:61 share_policy False,
        # train/train_mpe.py:139-150): one learner per policy, the centralised action vector is ordered like r_maddpg.py:62-105 walks
        # the policies (sorted ids, each policy's agents in order)
        self.multi = len(self.policy_ids) > 1
        self._eng = {}
        off = 0
        total = sum(len(self.policy_agents[p]) * self.policies[p].act_dim for p in self.policy_ids)
        for p in self.policy_ids:
            pol, n_p = self.policies[p], len(self.policy_agents[p])
            if self.multi and pol.central_act_dim != total:
                raise ValueError("policy %s: cent_act_dim %d != total action width %d of all agents" % (p, pol.central_act_dim, total))
            self._eng[p] = _Engine(args, pol, n_p, self.episode_length, self.max_batch, actor_update_interval,
                                   total if self.multi else 0, off if self.multi else 0)
            pol._trainer, pol._handle = self, self._eng[p].handle
            off += n_p * pol.act_dim
        first = self._eng[self.policy_ids[0]]
        # single-policy attributes kept for the graph helpers / tests
        self.cfg, self.workspace, self.handle, self._info, self._prio = first.cfg, first.workspace, first.handle, first.info, first.prio

    def __del__(self):
        try:
            for e in getattr(self, "_eng", {}).values():
                e.close()
            self.handle = None
        except Exception:
            pass

    def grad_views(self, p_id=None):
        """Numerator gradients (actor, critic) as flat views, for the parity tests."""
        e = self._eng[p_id or self.policy_ids[0]]
        a, c = C.c_int64(), C.c_int64()
        capi.lib().mx_maddpg_grad_views(e.handle, C.byref(a), C.byref(c))
        return (e.workspace[a.value:a.value + 4 * (e.pol.Pa + 4)].view(torch.float32),
                e.workspace[c.value:c.value + 4 * (e.pol.Pc + 4)].view(torch.float32))

    def _device_batch(self, batch, p_id="policy_0"):
        if isinstance(batch, SampledBatch):
            buf = batch.buffers[p_id]
            if buf.sample_serial != batch.serial[p_id]:
                raise RuntimeError("stale sample: the buffer has been sampled again since this batch was drawn")
            return buf.batch_struct(batch.B)
        e = self._eng[p_id]
        if e.host_batch is None:
            e.host_batch = _HostBatchC(e.cfg, self.dev)
        return e.host_batch.pack(batch, p_id, self.use_per)

    def draw_target_noise(self, B, p_id=None):
        """The draw the reference makes for the target actions of one policy in one update: (T+1, N_p*B, Ac), agent-major rows, CPU RNG."""
        e = self._eng[p_id or self.policy_ids[0]]
        pol = e.pol
        T, N, Ac = self.episode_length, e.n_agents, pol.act_dim
        if pol.discrete:
            return sample_gumbel((T + 1, N * B, Ac))                                               # util.py:137 via rMADDPGPolicy.py:105-106
        return torch.empty(T + 1, N * B, Ac).normal_(mean=0, std=float(pol.target_noise))          # util.py:217-218

    def draw_actor_noise(self, B, p_id=None):
        """Gumbel draws of the actor update's `get_actions(..., use_gumbel=True)` over obs[:-1] (r_maddpg.py:277): (T, N_p*B, Ac)."""
        e = self._eng[p_id or self.policy_ids[0]]
        return sample_gumbel((self.episode_length, e.n_agents * B, e.pol.act_dim))

    def _target_noise(self, B, p_id=None):
        """N(0, target_noise) / Gumbel draws for every target action, in batch row order on the device."""
        e = self._eng[p_id or self.policy_ids[0]]
        if not e.pol.td3:
            return None
        T, N, Ac = self.episode_length, e.n_agents, e.pol.act_dim
        noise = self.draw_target_noise(B, p_id)
        ours = noise.view(T + 1, N, B, Ac).permute(2, 0, 1, 3).contiguous()                      # -> [b][t][n][Ac]
        e.noise_dev = ours.to(self.dev, non_blocking=True)
        self._noise_dev = e.noise_dev
        return e.noise_dev

    def _actor_noise(self, B, p_id=None):
        """Gumbel draws of the actor update's `get_actions(..., use_gumbel=True)` over obs[:-1] (r_maddpg.py:277), padded to T+1 steps."""
        e = self._eng[p_id or self.policy_ids[0]]
        T, N, Ac = self.episode_length, e.n_agents, e.pol.act_dim
        g = self.draw_actor_noise(B, p_id)
        ours = torch.zeros(B, T + 1, N, Ac)
        ours[:, :T] = g.view(T, N, B, Ac).permute(2, 0, 1, 3)
        e.actor_noise_dev = ours.to(self.dev, non_blocking=True)
        self._actor_noise_dev = e.actor_noise_dev
        return e.actor_noise_dev

    def train_policy_on_batch(self, update_policy_id, batch):
        if self.use_same_share_obs:
            return self.shared_train_policy_on_batch(update_policy_id, batch)
        return self.cent_train_policy_on_batch(update_policy_id, batch)

    def cent_train_policy_on_batch(self, update_policy_id, batch):
        raise NotImplementedError("cent_train_policy_on_batch is unusable in the reference (missing train_info['update_actor']) and is not built")

    def shared_train_policy_on_batch(self, update_policy_id, batch):
        lib, stream = capi.lib(), capi.stream_ptr()
        e = self._eng[update_policy_id]
        b = self._device_batch(batch, update_policy_id)
        if self.multi:
            # r_maddpg.py:40-105 (get_update_info): every policy's buffer actions and TARGET-actor next actions, policy by policy in
            # id order -- the target-noise draws (MATD3) consume torch's CPU generator in that same order
            noise = None
            keep = []
            for q in self.policy_ids:
                bq = b if q == update_policy_id else self._device_batch(batch, q)
                nq = self._target_noise(b.B, q)
                keep.append((bq, nq))
                if q == update_policy_id:
                    noise = nq
                capi.check(lib.mx_maddpg_cent_contribute(self._eng[q].handle, C.byref(bq), capi.ptr(nq), e.handle, stream))
            self._keep = keep
        else:
            noise = self._target_noise(b.B, update_policy_id)
        will_update_actor = self.num_updates[update_policy_id] % self.actor_update_interval == 0
        actor_noise = self._actor_noise(b.B, update_policy_id) if (e.pol.discrete and will_update_actor) else None
        upd = C.c_int32()
        capi.check(lib.mx_maddpg_step_ex(e.handle, C.byref(b), capi.ptr(noise), capi.ptr(actor_noise), C.byref(upd), stream))
        info = e.info
        train_info = {"critic_loss": info[0], "critic_grad_norm": info[1]}
        if upd.value:
            train_info["actor_loss"], train_info["actor_grad_norm"] = info[4], info[5]
        train_info["update_actor"] = bool(upd.value)
        self.num_updates[update_policy_id] += 1
        new_priorities = DeviceArray(e.prio[:b.B]) if self.use_per else None
        return train_info, new_priorities, batch[8]

    def prep_training(self):
        pass

    def prep_rollout(self):
        pass
