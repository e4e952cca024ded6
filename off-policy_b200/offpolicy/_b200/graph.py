"""Whole-step CUDA graph: [sample ->] QMIX step [-> PER write-back] [-> soft update] captured once, replayed per step.

`mx_graph_capture` records the library's own launch sequence on a dedicated (non-default) stream; after that a learner
step costs one `cudaGraphLaunch` and no host work at all (indices come from the device-resident MT19937 stream).
"""
import ctypes as C

import torch

from offpolicy._b200 import capi

SAMPLE_UNIFORM, SAMPLE_PER, SOFT_UPDATE, PER_WRITEBACK = 1, 2, 4, 8


class StepGraph(object):
    """`buffer`: RecReplayBuffer / PrioritizedRecReplayBuffer with a recurrent trainer, or MlpReplayBuffer / PrioritizedMlpReplayBuffer with
    M_QMix / M_VDN (transitions are length-1 episodes of the same HBM replay, so the captured sequence is the same)."""

    def __init__(self, buffer, trainer, batch_size, beta=0.4, soft_update=True, p_id="policy_0"):
        lib = capi.lib()
        pb = buffer.policy_buffers[p_id]
        pb = getattr(pb, "rep", pb)               # MlpPolicyBuffer wraps the episode replay
        per = bool(getattr(trainer, "use_per", False))
        self.flags = (SAMPLE_PER | PER_WRITEBACK if per else SAMPLE_UNIFORM) | (SOFT_UPDATE if soft_update else 0)
        dev = capi.device()
        self.cuda = dev.type == "cuda"            # (the CPU-emulated unit-test build re-runs the sequence instead of a graph)
        self.stream = torch.cuda.Stream(device=dev) if self.cuda else None
        if self.cuda:
            self.stream.wait_stream(torch.cuda.current_stream(dev))
        self._sp = C.c_void_p(self.stream.cuda_stream if self.cuda else 0)
        g = C.c_void_p()
        capi.check(lib.mx_graph_capture(pb.handle, trainer.handle, int(batch_size), float(beta), self.flags, self._sp, C.byref(g)))
        self.handle = g
        self.lib = lib          # the library that made the graph frees it, whichever build is bound later
        self.num_kernels = int(lib.mx_graph_num_kernels(g))
        self._keep = (buffer, trainer)
        self._per, self._rep, self._beta = per, pb, float(beta)

    def launch(self, beta=None):
        """`beta`: PER importance-sampling exponent of this step (the runner anneals it every step, base_runner.py:159-160); it lives
        in a device scalar the captured draw reads, so changing it costs one tiny launch and no re-capture."""
        if beta is not None and self._per and float(beta) != self._beta:
            capi.check(capi.lib().mx_replay_set_beta(self._rep.handle, float(beta), self._sp))
            self._beta = float(beta)
        capi.check(capi.lib().mx_graph_launch(self.handle, self._sp))

    def synchronize(self):
        if self.cuda:
            self.stream.synchronize()

    def close(self):
        if self.handle:
            self.lib.mx_graph_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MaddpgStepGraph(object):
    """[sample ->] R_MADDPG.shared_train_policy_on_batch [-> soft update] as CUDA graphs (one per update_actor variant).

    Per `launch()` the host only draws the noise the reference would draw (MATD3 target noise / Gumbel draws, torch CPU RNG,
    same order as r_maddpg.py) into pinned buffers, enqueues their H2D copies on the graph's stream and replays the graph."""

    def __init__(self, buffer, trainer, batch_size, beta=0.4, soft_update=True, p_id="policy_0"):
        lib = capi.lib()
        self.lib = lib
        pb = buffer.policy_buffers[p_id]
        per = bool(getattr(trainer, "use_per", False))
        self.flags = (SAMPLE_PER | PER_WRITEBACK if per else SAMPLE_UNIFORM) | (SOFT_UPDATE if soft_update else 0)
        self.trainer, self.B, self.p_id = trainer, int(batch_size), p_id
        pol = trainer.policies[p_id]
        self.pol = pol
        T, N, Ac = trainer.episode_length, trainer.num_agents, pol.act_dim
        dev = capi.device()
        self.cuda = dev.type == "cuda"            # (the CPU-emulated unit-test build re-runs the sequence instead of a graph)
        self.stream = torch.cuda.Stream(device=dev) if self.cuda else None
        if self.cuda:
            self.stream.wait_stream(torch.cuda.current_stream(dev))
        self._sp = C.c_void_p(self.stream.cuda_stream if self.cuda else 0)
        shape = (self.B, T + 1, N, Ac)
        self.tnoise_dev = torch.zeros(shape, dtype=torch.float32, device=dev) if pol.td3 else None
        self.anoise_dev = torch.zeros(shape, dtype=torch.float32, device=dev) if pol.discrete else None
        # pinned staging ring: a slot is rewritten only after the H2D copy that last read it has completed (its event)
        self.RING = 4
        mk = lambda: [torch.zeros(shape, dtype=torch.float32).pin_memory() if self.cuda else torch.zeros(shape) for _ in range(self.RING)]
        self.tnoise_host = mk() if pol.td3 else None
        self.anoise_host = mk() if pol.discrete else None
        self._copied = [None] * self.RING
        self._slot = 0
        self.graphs = {}
        variants = (1, 0) if trainer.actor_update_interval > 1 else (1,)
        for upd in variants:
            g = C.c_void_p()
            capi.check(lib.mx_maddpg_graph_capture(pb.handle, trainer.handle, self.B, float(beta), self.flags, capi.ptr(self.tnoise_dev),
                                                   capi.ptr(self.anoise_dev), upd, self._sp, C.byref(g)))
            self.graphs[upd] = g
        self.num_kernels = {u: int(lib.mx_graph_num_kernels(g)) for u, g in self.graphs.items()}
        self._keep = (buffer, trainer)
        self._per, self._rep, self._beta = per, pb, float(beta)

    def launch(self, beta=None):
        tr, pol = self.trainer, self.pol
        if beta is not None and self._per and float(beta) != self._beta:       # annealed PER exponent: device scalar (see StepGraph.launch)
            capi.check(self.lib.mx_replay_set_beta(self._rep.handle, float(beta), self._sp))
            self._beta = float(beta)
        T, N, Ac, B = tr.episode_length, tr.num_agents, pol.act_dim, self.B
        upd = 1 if tr.num_updates[self.p_id] % tr.actor_update_interval == 0 else 0
        k = self._slot
        self._slot = (k + 1) % self.RING
        if self._copied[k] is not None:
            self._copied[k].synchronize()
        with torch.cuda.stream(self.stream) if self.cuda else _null():
            if pol.td3:
                n = tr.draw_target_noise(B)                                     # (T+1, N*B, Ac), reference row order
                self.tnoise_host[k].copy_(n.view(T + 1, N, B, Ac).permute(2, 0, 1, 3))
                self.tnoise_dev.copy_(self.tnoise_host[k], non_blocking=True)
            if pol.discrete and upd:
                g = tr.draw_actor_noise(B)                                      # (T, N*B, Ac)
                self.anoise_host[k][:, :T].copy_(g.view(T, N, B, Ac).permute(2, 0, 1, 3))
                self.anoise_dev.copy_(self.anoise_host[k], non_blocking=True)
            if self.cuda and (pol.td3 or pol.discrete):
                if self._copied[k] is None:
                    self._copied[k] = torch.cuda.Event()
                self._copied[k].record(self.stream)
        capi.check(self.lib.mx_graph_launch(self.graphs[upd], self._sp))
        tr.num_updates[self.p_id] += 1
        return bool(upd)

    def synchronize(self):
        if self.cuda:
            self.stream.synchronize()

    def close(self):
        for g in self.graphs.values():
            self.lib.mx_graph_destroy(g)
        self.graphs = {}

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _null(object):
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False
