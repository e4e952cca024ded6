"""Error behaviour of the drop-in classes (host logic; CPU): the reference signals misuse with Python asserts / exceptions
(rec_buffer.py:165, 287-289, 315-318), the C-ABI with non-zero status + mx_last_error(); unsupported configurations are rejected at
construction instead of being approximated."""
import ctypes as C
import types

import numpy as np
import pytest

import qmix_checks as qc
import replay_checks as rc
from oracle.qmix import QmixConfig


def _episodes(N, O, A, S, T, n, rs):
    return [rc.d(x.astype(np.float32)) for x in (rs.randn(T + 1, n, N, O), np.repeat(rs.randn(T + 1, n, 1, S), N, 2), np.eye(A)[rs.randint(0, A, (T, n, N))],
                                                rs.randn(T, n, N, 1), np.zeros((T, n, N, 1)), np.zeros((T, n, 1)), np.ones((T + 1, n, N, A)))]


def test_buffer_misuse(emu_engine):
    MxError = emu_engine.MxError
    N, O, A, S, T, E = 2, 4, 3, 5, 3, 6
    rs = np.random.RandomState(0)
    buf = rc.make_buffers(N, O, A, S, T, E, max_batch=4)
    with pytest.raises(ValueError):
        buf.sample(2)                                                      # empty buffer: NumPy refuses to draw from range(0), like the reference's np.random.choice(0, B)
    dbuf = rc.make_buffers(N, O, A, S, T, E, rng="device", max_batch=4)
    with pytest.raises(MxError):
        dbuf.sample(2)                                                     # same with the device-side index stream
    ep = _episodes(N, O, A, S, T, 2, rs)
    with pytest.raises(AssertionError):
        buf.insert(2, *_episodes(N, O, A, S, T + 1, 2, rs))                # rec_buffer.py:165 "different dimension!"
    bad = list(ep)
    bad[0] = rc.d(np.zeros((T + 1, 2, N, O + 1), np.float32))
    with pytest.raises(ValueError):
        buf.insert(2, *bad)                                                # a field of the wrong size
    with pytest.raises(ValueError):
        buf.insert(5, *_episodes(N, O, A, S, T, 5, rs))                    # more episodes than max_batch in one call
    r = buf.insert(2, *ep)
    assert list(r) == [0, 1] and len(buf) == 2
    with pytest.raises(ValueError):
        buf.sample(5)                                                      # batch_size > max_batch
    s1 = buf.sample(2)
    s2 = buf.sample(2)
    with pytest.raises(RuntimeError):
        s1[0]["policy_0"]                                                  # the device batch region was reused by the later sample
    assert s2[0]["policy_0"].shape == (N, T + 1, 2, O)
    with pytest.raises(KeyError):
        s2[0]["policy_7"]


def test_per_misuse(emu_engine):
    N, O, A, S, T, E = 2, 4, 3, 5, 3, 8
    rs = np.random.RandomState(1)
    buf = rc.make_buffers(N, O, A, S, T, E, per_alpha=0.6, max_batch=8)
    buf.insert(4, *_episodes(N, O, A, S, T, 4, rs))
    with pytest.raises(AssertionError):
        buf.sample(4, 0.4, "policy_0")                                     # rec_buffer.py:287: len(self) > batch_size
    with pytest.raises(AssertionError):
        buf.sample(2, 0.0, "policy_0")                                     # rec_buffer.py:289: beta > 0
    with pytest.raises(AssertionError):
        buf.update_priorities(np.array([0, 1]), np.array([1.0, -1.0], np.float32), "policy_0")     # :316 priorities > 0
    with pytest.raises(AssertionError):
        buf.update_priorities(np.array([0, 9]), np.array([1.0, 1.0], np.float32), "policy_0")      # :318 idx < len
    with pytest.raises(AssertionError):
        buf.update_priorities(np.array([0, 1]), np.array([1.0], np.float32), "policy_0")           # :315 same length


def test_trainer_rejects_what_it_does_not_implement(emu_engine):
    MxError = emu_engine.MxError
    with pytest.raises(MxError):
        qc.build_trainer(QmixConfig(hidden=128), 4, 4)                     # kernels are specialised for hidden_size 64
    from offpolicy.algorithms.qmix.algorithm.QMixPolicy import QMixPolicy
    from offpolicy.algorithms.qmix.qmix import QMix
    cfg = QmixConfig()
    args = qc.make_args(cfg, 4)
    info = dict(obs_space=[cfg.obs_dim], share_obs_space=[cfg.state_dim], act_space=rc.Discrete(cfg.act_dim), cent_obs_dim=cfg.state_dim,
                cent_act_dim=cfg.act_dim * cfg.n_agents)
    for flag, val in (("layer_N", 2), ("use_rnn_layer", False), ("use_conv1d", True)):
        a2 = types.SimpleNamespace(**vars(args))
        setattr(a2, flag, val)
        with pytest.raises(NotImplementedError):
            QMixPolicy({"args": a2, "device": emu_engine.device()}, info)
    # the recurrent MADDPG / MATD3 policies validate the same flags
    import maddpg_checks as mdc
    from oracle.maddpg import MaddpgConfig
    from offpolicy.algorithms.r_maddpg.algorithm.rMADDPGPolicy import R_MADDPGPolicy
    margs = mdc.make_args(MaddpgConfig(n_agents=2, obs_dim=5, act_dim=2, state_dim=6), 4)
    minfo = dict(obs_space=[5], share_obs_space=[6], act_space=mdc.Box(2), cent_obs_dim=6, cent_act_dim=4)
    R_MADDPGPolicy({"args": margs, "device": emu_engine.device()}, minfo)
    for flag, val in (("layer_N", 2), ("hidden_size", 128), ("prev_act_inp", True), ("recurrent_N", 2)):
        a2 = types.SimpleNamespace(**vars(margs))
        setattr(a2, flag, val)
        with pytest.raises(NotImplementedError):
            R_MADDPGPolicy({"args": a2, "device": emu_engine.device()}, minfo)
    pols = {"policy_%d" % i: QMixPolicy({"args": args, "device": emu_engine.device()}, info) for i in range(3)}
    with pytest.raises(NotImplementedError):                              # one policy per agent (share_policy=False)
        QMix(args, 3, pols, lambda a: "policy_%d" % a, device=emu_engine.device(), episode_length=4)
    # PopArt: applied by the reference only in mqmix.py:184-187 (the recurrent qmix.py constructs it and never uses it)
    from offpolicy.algorithms.mqmix.mqmix import M_QMix
    a2 = types.SimpleNamespace(**vars(args))
    a2.use_popart = True
    one = {"policy_0": pols["policy_0"]}
    QMix(a2, 3, one, lambda a: "policy_0", device=emu_engine.device(), episode_length=4)       # a no-op flag there: accepted
    with pytest.raises(NotImplementedError):
        M_QMix(a2, 3, one, lambda a: "policy_0", device=emu_engine.device())
    from offpolicy.utils.rec_buffer import RecReplayBuffer
    with pytest.raises(NotImplementedError):
        RecReplayBuffer({"policy_0": info}, {"policy_0": [0, 1, 2]}, 8, 4, False, True)               # use_same_share_obs=False


def test_objects_are_freed_by_the_library_that_made_them(emu_engine, monkeypatch):
    """A replay, learner or step graph collected after another build of the library was bound (a process that uses the emulated build
    and then the CUDA one) hands its handle back to the build that made it: the other build would be given a pointer it never issued."""
    import gc
    from offpolicy._b200 import factory
    from offpolicy._b200.graph import StepGraph
    N, O, A, S, T = 2, 4, 3, 5, 3
    buf = factory.make_rec_buffers(N, O, A, S, T, 8, rng="device", max_batch=4)
    buf.insert(4, *_episodes(N, O, A, S, T, 4, np.random.RandomState(2)))
    args, pol, tr = qc.build_trainer(QmixConfig(n_agents=N, obs_dim=O, act_dim=A, state_dim=S), 4, T)
    graph = StepGraph(buf, tr, 4)
    margs, mpol, mtr = factory.build_maddpg(factory.MaddpgLearnerConfig(n_agents=2, obs_dim=5, act_dim=2, state_dim=6), 4, T)
    lib, freed = emu_engine.lib(), []
    names = ("mx_graph_destroy", "mx_qmix_destroy", "mx_replay_destroy", "mx_maddpg_destroy")
    for name in names:
        monkeypatch.setattr(lib, name, lambda h, _f=getattr(lib, name), _n=name: (freed.append(_n), _f(h))[1])

    class OtherBuild(object):
        calls = []

        def __getattr__(self, name):
            self.calls.append(name)
            return lambda *a: 0
    monkeypatch.setattr(emu_engine, "_lib", OtherBuild())
    del buf, args, pol, tr, graph, margs, mpol, mtr
    gc.collect()
    assert OtherBuild.calls == [] and set(freed) == set(names), (OtherBuild.calls, freed)


def test_c_abi_status_codes(emu_engine):
    lib = emu_engine.lib()
    cfg = emu_engine.ReplayCfg(0, 4, 2, 3, 3, 2, 1, 0, 0, 4, 0.0)          # capacity 0
    lay = emu_engine.ReplayLayout()
    assert lib.mx_replay_layout_query(C.byref(cfg), C.byref(lay)) != 0 and b"non-positive" in lib.mx_last_error()
    assert lib.mx_set_option(b"mixer_split", 1) == 0
    args, pol, tr = qc.build_trainer(QmixConfig(), 4, 4)
    b = emu_engine.Batch()
    b.B = 99
    assert lib.mx_qmix_step(tr.handle, C.byref(b), None) != 0 and b"batch size" in lib.mx_last_error()
    b.B = 2
    assert lib.mx_qmix_step(tr.handle, C.byref(b), None) != 0 and b"missing batch field" in lib.mx_last_error()
    off, n = C.c_int64(), C.c_int64()
    assert lib.mx_qmix_ws_lookup(tr.handle, b"no_such_region", C.byref(off), C.byref(n)) != 0
