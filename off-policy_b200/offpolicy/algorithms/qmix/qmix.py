"""Drop-in `QMix` trainer (reference: offpolicy/algorithms/qmix/qmix.py) on the fused sm_100a learner.

Same constructor and methods as the reference class -- `train_policy_on_batch`, `soft_target_updates`,
`hard_target_updates`, `prep_training`, `prep_rollout`, attribute `mixer` -- so
offpolicy/runner/rnn/base_runner.py:143,259-284,314,337 drives it unchanged.  One call of
`train_policy_on_batch` = one `mx_qmix_step` (csrc/qmix.cu): live + target agent nets over the T+1 steps,
mixers, TD target, masked MSE/Huber, BPTT, global-norm clip and Adam, all on the device.  Live/target
parameters and Adam moments are four flat fp32 vectors; `policies[p].q_network` and `self.mixer` are named
views of the live vector with the reference's state_dict keys.

Data-parallel use (`torch.distributed` initialised, world size G > 1): each rank owns a replay shard and
samples its own batch; the per-rank gradient NUMERATORS plus the loss denominators are summed with a
single all-reduce of one flat buffer, after which every rank applies the identical clip + Adam update
(the reference has no distributed path: utils/util.py:148-153 is dead code).
"""
import ctypes as C
import os
import sys

import numpy as np
import torch

from offpolicy._b200 import capi
from offpolicy._b200.flat import FlatModule, reference_style_init
from offpolicy.algorithms.qmix.algorithm.QMixPolicy import qmix_cfg_struct, param_entries
from offpolicy.utils.rec_buffer import SampledBatch, DeviceArray


class _HostBatch(object):
    """Device copy of a batch handed over in the reference's NumPy layout (rec_buffer.py:82): the compatibility
    path for callers that sample elsewhere.  Layout conversion is torch plumbing, not a hot path."""

    def __init__(self, cfg, dev):
        self.cfg, self.dev = cfg, dev
        B, T, N = cfg.max_batch, cfg.episode_len, cfg.n_agents
        r4 = lambda v: (v + 3) // 4 * 4
        self.obs_ld, self.share_ld, self.act_ld = r4(cfg.obs_dim), r4(cfg.state_dim), r4(cfg.act_dim)
        z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=dev)
        self.obs = z(B, T + 1, N, self.obs_ld)
        self.share = z(B, T + 1, self.share_ld)
        self.acts = z(B, T, N, self.act_ld)
        self.act_idx = z(B, T, N, dt=torch.int32)
        self.avail = z(B, T + 1, N, self.act_ld)
        self.rew = z(B, T, N)
        self.dones = z(B, T, N)
        self.dones_env = z(B, T)
        self.weights = z(B)

    def pack(self, batch, p_id, use_avail, use_per):
        obs, share, acts, rew, dones, dones_env, avail, weights, idx = batch
        c, dev = self.cfg, self.dev
        t = lambda x: torch.as_tensor(np.asarray(x), dtype=torch.float32).to(dev)
        o = t(obs[p_id])                                   # (N, T+1, B, O)
        B = o.shape[2]
        self.obs[:B, :, :, :c.obs_dim] = o.permute(2, 1, 0, 3)
        self.share[:B, :, :c.state_dim] = t(share[p_id]).permute(1, 0, 2)
        a = t(acts[p_id]).permute(2, 1, 0, 3)              # (B, T, N, A)
        self.acts[:B, :, :, :c.act_dim] = a
        self.act_idx[:B] = a.max(dim=-1)[1].to(torch.int32)
        if use_avail:
            self.avail[:B, :, :, :c.act_dim] = t(avail[p_id]).permute(2, 1, 0, 3)
        self.rew[:B] = t(rew[p_id])[..., 0].permute(2, 1, 0)
        self.dones[:B] = t(dones[p_id])[..., 0].permute(2, 1, 0)
        self.dones_env[:B] = t(dones_env[p_id])[..., 0].permute(1, 0)
        if use_per:
            self.weights[:B] = t(weights)
        b = capi.Batch()
        b.B = B
        b.obs_ld, b.share_ld, b.act_ld = self.obs_ld, self.share_ld, self.act_ld
        b.obs, b.share, b.acts, b.act_idx = self.obs.data_ptr(), self.share.data_ptr(), self.acts.data_ptr(), self.act_idx.data_ptr()
        b.avail = self.avail.data_ptr() if use_avail else None
        b.rewards, b.dones, b.dones_env = self.rew.data_ptr(), self.dones.data_ptr(), self.dones_env.data_ptr()
        b.weights = self.weights.data_ptr() if use_per else None
        b.idx = None
        return b


class QMix(object):
    def __init__(self, args, num_agents, policies, policy_mapping_fn, device=None, episode_length=None, vdn=False):
        self.args = args
        self.use_per = args.use_per
        self.device = device
        self.num_agents = num_agents
        self.policies = policies
        self.policy_mapping_fn = policy_mapping_fn
        self.policy_ids = sorted(list(self.policies.keys()))
        self.policy_agents = {p: sorted(a for a in range(num_agents) if policy_mapping_fn(a) == p) for p in self.policies}
        if self.policy_ids != ["policy_0"]:
            raise NotImplementedError("B200 QMIX path: only the shared-policy configuration ('policy_0') is implemented")
        if getattr(args, "use_popart", False) and getattr(self, "_mlp", False):
            # mqmix.py:184-187 normalises the TD target with PopArt; the recurrent qmix.py:44-45 only constructs the normaliser and
            # never applies it, so the flag is a no-op there and needs no check
            raise NotImplementedError("B200 M_QMix path: --use_popart is not implemented")
        self.episode_length = args.episode_length if episode_length is None else episode_length
        self.use_same_share_obs = getattr(args, "use_same_share_obs", True)
        self.vdn = bool(vdn)
        pol = self.policies["policy_0"]
        self.use_avail = bool(getattr(args, "use_available_actions", True))
        self.max_batch = int(getattr(args, "batch_size", 32))

        lib = capi.lib()
        self.dev = capi.device()
        self.world_size = torch.distributed.get_world_size() if torch.distributed.is_available() and torch.distributed.is_initialized() else 1
        self.world_size = int(getattr(args, "dp_world_size", None) or self.world_size)     # (tests drive several "ranks" from one process)
        self._p2p = False
        self.cfg = self._cfg_struct(args, num_agents, pol)
        entries, total = param_entries(self.cfg)
        self.entries, self.P = entries, total
        z = lambda: torch.zeros(total, dtype=torch.float32, device=self.dev)
        self.theta, self.theta_tgt, self.adam_m, self.adam_v = z(), z(), z(), z()
        # adopt the policy's agent weights, initialise the mixer like the reference, then re-bind the views
        src = pol.q_network.state_dict()
        pol.q_network.bind(self.theta)
        pol.q_network.load_state_dict(src)
        self.mixer = FlatModule(self.theta, entries, "mixer.")
        if not self.vdn:
            init = reference_style_init([e for e in entries if e[0].startswith("mixer.")],
                                        dict(state_dim=pol.central_obs_dim, n_agents=num_agents, mixer_hidden=args.mixer_hidden_dim,
                                             hyper_hidden=args.hypernet_hidden_dim, hidden=args.hidden_size, obs_dim=getattr(pol, "q_network_input_dim", pol.obs_dim),
                                             act_dim=pol.act_dim), gain=1.0, use_orthogonal=args.use_orthogonal,
                                        hyper_layers=args.hypernet_layers)
            self.mixer.load_state_dict({k[len("mixer."):]: v for k, v in init.items()})
        self.theta_tgt.copy_(self.theta)                                               # qmix.py:63-64 (deepcopy)
        self.target_q_network = FlatModule(self.theta_tgt, entries, "agent.")
        self.target_mixer = FlatModule(self.theta_tgt, entries, "mixer.")
        self.parameters = pol.q_network.parameters() + self.mixer.parameters()          # qmix.py:66-70 (order kept)

        nbytes = int(lib.mx_qmix_workspace_bytes(C.byref(self.cfg)))
        if nbytes < 0:
            raise capi.MxError(lib.mx_last_error().decode())
        self.workspace = torch.zeros(nbytes, dtype=torch.uint8, device=self.dev)
        h = C.c_void_p()
        capi.check(lib.mx_qmix_create(C.byref(self.cfg), capi.ptr(self.theta), capi.ptr(self.theta_tgt), capi.ptr(self.adam_m),
                                      capi.ptr(self.adam_v), capi.ptr(self.workspace), nbytes, C.byref(h)))
        self.handle = h
        self._lib = lib         # the library that made the handle (and the step graphs) frees them, whichever build is bound later
        self._host_batch = None
        self.use_step_graph = True          # replay the captured launch sequence for batches that live in a replay's batch region
        self._graphs, self._graph_keep, self._cap_stream = {}, [], None
        self._info = self.ws_view("info")
        self._info_views = (self._info[0], self._info[1], self._info[2])       # 0-dim views, created once (they alias the workspace)
        self._prio_view = self.ws_view("prio")
        n = C.c_int64()
        gptr = lib.mx_qmix_grad_buffer(self.handle, C.byref(n))
        off = gptr - self.workspace.data_ptr()
        self._grad_buf = self.workspace[off:off + 4 * int(n.value)].view(torch.float32)
        if self.world_size > 1 and self.dev.type == "cuda" and os.environ.get("MARL_B200_P2P", "1") != "0" and \
                torch.distributed.is_available() and torch.distributed.is_initialized():
            try:
                self._setup_p2p()
            except Exception as ex:       # no peer access / symmetric memory on this box: the NCCL all-reduce path stays in use
                sys.stderr.write("marl_b200: peer-memory gradient exchange unavailable (%s); using the NCCL all-reduce\n" % (ex,))
            # every rank must use the same exchange: fall back everywhere if any rank could not map its peers
            agree = torch.tensor([1 if self._p2p else 0], dtype=torch.int32, device=self.dev)
            torch.distributed.all_reduce(agree, op=torch.distributed.ReduceOp.MIN)
            if int(agree) == 0:
                self._p2p = False
        if getattr(args, "use_double_q", True):
            print("double Q learning will be used")

    def _cfg_struct(self, args, num_agents, pol):
        return qmix_cfg_struct(args, num_agents, pol.obs_dim, pol.act_dim, pol.central_obs_dim, self.episode_length, self.max_batch,
                               vdn=self.vdn, use_avail=True, world_size=self.world_size)

    # -- data-parallel gradient exchange over NVLink peer memory (csrc/p2p.cu) ----------------------------------------
    def _setup_p2p(self):
        """One symmetric block per rank (torch.distributed._symmetric_memory: allocation + exchange of the peer mappings is
        plumbing), handed to the library; from then on `mx_qmix_step` contains the whole exchange and NCCL is not called."""
        import torch.distributed._symmetric_memory as symm
        dist = torch.distributed
        n = int(capi.lib().mx_qmix_p2p_block_bytes(self.handle)) // 4
        block = symm.empty(n, dtype=torch.float32, device=self.dev)
        block.zero_()
        hdl = symm.rendezvous(block, dist.group.WORLD.group_name)
        torch.cuda.synchronize(self.dev)
        dist.barrier()
        self.attach_peer_blocks(dist.get_rank(), [int(p) for p in hdl.buffer_ptrs], keep=(block, hdl))
        self._p2p = self._p2p_selftest(block)

    def _p2p_selftest(self, block):
        """One exchange of a known pattern before the first real step: rank r publishes r + 1 in every element, the reduce must
        return G (G + 1) / 2 everywhere without a time-out.  Every rank always reaches both barriers (local failures are only
        recorded), and the caller combines the verdicts with an all-reduce, so a box on which peer loads misbehave falls back to
        the NCCL exchange on ALL ranks instead of training on garbage."""
        dist = torch.distributed
        lib, stream = capi.lib(), capi.stream_ptr()
        rank, world = dist.get_rank(), dist.get_world_size()
        ok = True
        adam_t = self.ws_view("adam_t", torch.float64)
        saved = adam_t.clone()
        try:
            self._grad_buf.fill_(float(rank + 1))
            self._info[7] = 0.0
            adam_t[0] = 1.0                                   # the kernels take the step number (slot parity, flag value) from here
            capi.check(lib.mx_qmix_p2p_publish(self.handle, stream))
            capi.check(lib.mx_qmix_p2p_reduce(self.handle, stream))
            torch.cuda.synchronize(self.dev)
            want = world * (world + 1) / 2.0
            ok = bool((self._grad_buf == want).all().item()) and float(self._info[7]) == 0.0
        except Exception as ex:
            sys.stderr.write("marl_b200: peer-memory self-test raised %s\n" % (ex,))
            ok = False
        adam_t.copy_(saved)
        self._grad_buf.zero_()
        self._info[7] = 0.0
        torch.cuda.synchronize(self.dev)
        dist.barrier()                                        # nobody is reading a slot any more
        block.zero_()                                         # flags back to 0: the first real step is step 1 again
        torch.cuda.synchronize(self.dev)
        dist.barrier()
        return ok

    def attach_peer_blocks(self, rank, block_ptrs, keep=None):
        ptrs = (C.c_void_p * len(block_ptrs))(*block_ptrs)
        self._p2p_counter = torch.zeros(4, dtype=torch.int32, device=self.dev)
        capi.check(capi.lib().mx_qmix_set_peers(self.handle, int(rank), len(block_ptrs), ptrs, capi.ptr(self._p2p_counter)))
        self._p2p_keep = keep
        self._p2p = True

    def __del__(self):
        try:
            self.drop_step_graphs()
            if getattr(self, "handle", None):
                self._lib.mx_qmix_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # -- introspection used by the parity tests ------------------------------------------------------------
    def ws_view(self, name, dtype=torch.float32):
        off, n = C.c_int64(), C.c_int64()
        capi.check(capi.lib().mx_qmix_ws_lookup(self.handle, name.encode(), C.byref(off), C.byref(n)))
        return self.workspace[off.value:off.value + 4 * n.value].view(dtype)

    def grad_views(self):
        """Unclipped mean gradients d(loss)/d(param) by reference name (numerators / sum(1-bad))."""
        g = self.ws_view("grad")
        denom = g[self.P]
        out = {}
        for name, off, rows, cols in self.entries:
            n = rows * (cols if cols else 1)
            v = g[off:off + n] / denom
            out[name] = v.view(rows, cols) if cols else v
        return out

    # -- the update ----------------------------------------------------------------------------------------------
    def _device_batch(self, batch):
        if isinstance(batch, SampledBatch):
            buf = batch.buffers["policy_0"]
            if buf.sample_serial != batch.serial["policy_0"]:
                raise RuntimeError("stale sample: the buffer has been sampled again since this batch was drawn")
            return buf.batch_struct(batch.B)
        if self._host_batch is None:
            self._host_batch = _HostBatch(self.cfg, self.dev)
        avail = batch[6]["policy_0"] if batch[6] is not None else None
        return self._host_batch.pack(batch, "policy_0", avail is not None, self.use_per)      # MPE: no masks (mpe_runner.py:62)

    def train_policy_on_batch(self, batch, update_policy_id=None):
        lib = capi.lib()
        stream = capi.stream_ptr()
        sampled = isinstance(batch, SampledBatch)
        if sampled and self.use_step_graph and self.dev.type == "cuda" and (self.world_size == 1 or self._p2p):
            # fast path: the batch lives in a replay's batch region -> replay the captured launch sequence (one cudaGraphLaunch)
            buf = batch.buffers["policy_0"]
            if buf.sample_serial != batch.serial["policy_0"]:
                raise RuntimeError("stale sample: the buffer has been sampled again since this batch was drawn")
            B = batch.B
            capi.check(lib.mx_graph_launch(self._step_graph(batch, B), stream))
        else:
            b = self._device_batch(batch)
            B = b.B
            if self.world_size > 1 and not self._p2p:
                capi.check(lib.mx_qmix_backward_only(self.handle, C.byref(b), stream))
                torch.distributed.all_reduce(self._grad_buf)
                capi.check(lib.mx_qmix_apply(self.handle, stream))
            else:
                capi.check(lib.mx_qmix_step(self.handle, C.byref(b), stream))
        self._check_exchange()
        v = self._info_views
        train_info = {"loss": v[0], "grad_norm": v[1], "Q_tot": v[2]}                   # qmix.py:195-198 (0-dim device tensors)
        new_priorities = DeviceArray(self._prio_view[:B]) if self.use_per else None
        return train_info, new_priorities, batch[8]

    def _check_exchange(self):
        """Peer-memory exchange watchdog.  A rank that waits more than 10 s for a peer sets info[7] = -1 on the device and applies NO
        update from then on (csrc/optim.cu, csrc/p2p.cu).  The flag is mirrored to pinned host memory after every step without a
        synchronisation; the copy of the PREVIOUS step is inspected here, so a dead peer turns into an exception one step later
        instead of silently diverging replicas."""
        if not self._p2p or self.dev.type != "cuda":
            return
        if getattr(self, "_xchg_host", None) is None:
            self._xchg_host = torch.zeros(1, dtype=torch.float32).pin_memory()
            self._xchg_ev = torch.cuda.Event()
            self._xchg_pending = False
        if self._xchg_pending and self._xchg_ev.query():
            self._xchg_pending = False
            if float(self._xchg_host[0]) < 0.0:
                raise RuntimeError("marl_b200: a data-parallel peer did not deliver its gradient within 10 s; no update was applied "
                                   "(replicas are still identical). Restart the job or set MARL_B200_P2P=0 for the NCCL exchange.")
        if not self._xchg_pending:
            self._xchg_host.copy_(self._info[7:8], non_blocking=True)
            self._xchg_ev.record(torch.cuda.current_stream(self.dev))
            self._xchg_pending = True

    def _step_graph(self, batch, B):
        """The learner step on a sampled batch always reads the replay's batch region, so its launch sequence is captured once
        per (buffer, B) into a CUDA graph (on a private stream; the legacy default stream cannot capture) and replayed on the
        caller's stream: one cudaGraphLaunch instead of 13 kernel launches per `train_policy_on_batch`."""
        buf = batch.buffers["policy_0"]
        key = (id(buf), int(B))
        g = self._graphs.get(key)
        if g is None:
            if self._cap_stream is None:
                self._cap_stream = torch.cuda.Stream(device=self.dev)
            torch.cuda.synchronize(self.dev)
            h = C.c_void_p()
            capi.check(capi.lib().mx_graph_capture(buf.handle, self.handle, int(B), 0.0, 0, C.c_void_p(self._cap_stream.cuda_stream), C.byref(h)))
            self._graphs[key] = g = h
            self._graph_keep.append(buf)
        return g

    def drop_step_graphs(self):
        for g in self._graphs.values():
            self._lib.mx_graph_destroy(g)
        self._graphs = {}

    # -- checkpoint / resume (SURVEY.md 8(f).3) ------------------------------------------------------------------------
    def state_dict(self):
        """The whole learner: live + target parameters, Adam moments and step count.  (`policies[p].q_network.state_dict()` /
        `mixer.state_dict()` remain the reference's per-network checkpoints, base_runner.py:286-337.)"""
        return {"theta": self.theta.cpu().clone(), "theta_tgt": self.theta_tgt.cpu().clone(), "adam_m": self.adam_m.cpu().clone(),
                "adam_v": self.adam_v.cpu().clone(), "adam_t": self.ws_view("adam_t", torch.float64).cpu().clone(),
                "layout": [(n, int(o), int(r), int(c)) for n, o, r, c in self.entries]}

    def load_state_dict(self, sd):
        if [tuple(e) for e in sd["layout"]] != [(n, int(o), int(r), int(c)) for n, o, r, c in self.entries]:
            raise ValueError("learner checkpoint was written for a different network configuration")
        for name in ("theta", "theta_tgt", "adam_m", "adam_v"):
            getattr(self, name).copy_(torch.as_tensor(sd[name]).to(self.dev))
        self.ws_view("adam_t", torch.float64).copy_(torch.as_tensor(sd["adam_t"]).to(self.dev))
        if self._p2p and self._p2p_keep is not None and torch.distributed.is_initialized():
            # the peers' "step reached" flags in the symmetric block belong to the run that wrote them: start over (every rank
            # restores the same step count, so the exchange resumes in lock-step)
            torch.cuda.synchronize(self.dev)
            torch.distributed.barrier()
            self._p2p_keep[0].zero_()
            torch.cuda.synchronize(self.dev)
            torch.distributed.barrier()

    def hard_target_updates(self):
        print("hard update targets")
        capi.check(capi.lib().mx_qmix_hard_update(self.handle, capi.stream_ptr()))

    def soft_target_updates(self):
        capi.check(capi.lib().mx_qmix_soft_update(self.handle, capi.stream_ptr()))

    def prep_training(self):
        pass            # no dropout / batch-norm in these nets: train()/eval() are numerical no-ops (qmix.py:218-232)

    def prep_rollout(self):
        pass
