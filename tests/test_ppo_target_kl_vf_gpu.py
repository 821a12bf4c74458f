"""SB3's clip_range_vf and target_kl through every update path, against autograd and SB3's PPO.train arithmetic
(tests/sb3_ext_oracle.py).

clip_range_vf: the old values travel in the packed record ([ret old_value 0 0]) or are gathered from the rollout's
values (per-launch path).  The problems are built so that, on every minibatch, a good share of the samples is clipped
below, a good share above and a good share not at all; the offsets stay at least c / 2 away from the bounds, so no
sample sits near V - old = +-c.  A sample EXACTLY at the bound is not constructed: the kernel's V differs from torch's
in the last bits, so an offset set to c in torch lands on either side of it on the device.

target_kl: thresholds are picked from SB3's own KL sequence of the same problem with a margin of at least 1 % to every
KL evaluated before the stop, so float rounding cannot move the decision.
"""
import copy

import numpy as np
import pytest
import torch

import sb3_ext_oracle as X
from oracle import sb3_oracle
from perm_ref import device_permutation
from test_ppo_update_gpu import _make_problem, _oracle_batch, _updater
from test_ppo_widths_gpu import _assert_grad_matches, _assert_tail_matches, _dev, _kp

pytestmark = pytest.mark.gpu

KW = dict(clip_range=0.2, ent_coef=0.05, vf_coef=0.5, normalize_advantage=True)
C_VF = 0.3


def _vf_problem(O, T, N, seed, c=C_VF):
    """_make_problem plus rollout values: V(s) of the policy shifted by -u, u a third each in [-c/2, c/2] (kept),
    [1.5c, 3c] (clipped below) and [-3c, -1.5c] (clipped above)."""
    pol, buf = _make_problem(O, T, N, seed)
    with torch.no_grad():
        _, v = pol.mean_value(torch.as_tensor(buf["obs"]).reshape(T * N, O))
    rng = np.random.default_rng(seed + 1)
    kind = rng.integers(0, 3, T * N)
    mag = rng.uniform(1.5, 3.0, T * N) * c
    u = np.where(kind == 0, rng.uniform(-0.5, 0.5, T * N) * c, np.where(kind == 1, mag, -mag))
    buf["values"] = (v.numpy() + u).astype(np.float32).reshape(T, N)
    return pol, buf


def _same_policy_problem(O, T, N, seed):
    """_make_problem with the rollout's log-probs recomputed under the policy being trained: approx_kl starts at 0
    and grows with every step, so a threshold's first crossing can be placed."""
    pol, buf = _make_problem(O, T, N, seed)
    with torch.no_grad():
        mu, _ = pol.mean_value(torch.as_tensor(buf["obs"]).reshape(T * N, O))
        lp = pol.log_prob(mu, torch.as_tensor(buf["actions"]).reshape(T * N, 2))
    buf["log_probs"] = lp.numpy().reshape(T, N)
    return pol, buf


def _autograd_vf(pol, buf, idx, dtype, c=C_VF):
    p = copy.deepcopy(pol).to(dtype)
    batch = tuple(t.to(dtype) for t in _oracle_batch(buf, idx))
    old_v = torch.as_tensor(sb3_oracle.flatten_env_major(buf["values"]))[torch.as_tensor(idx)].flatten().to(dtype)
    loss, st = X.ppo_loss(p, *batch, old_v, clip_range_vf=c, **KW)
    p.zero_grad()
    loss.backward()
    return p.flat_grads().numpy(), st


def _moments(opt):
    return (torch.cat([opt.state[q]["exp_avg"].reshape(-1) for q in opt.param_groups[0]["params"]]).numpy(),
            torch.cat([opt.state[q]["exp_avg_sq"].reshape(-1) for q in opt.param_groups[0]["params"]]).numpy())


# ---- 1. the record ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("O", [1, 15, 16, 31])
def test_packed_record_carries_old_values(cuda_lib, O):
    """[obs | 0 .. | 1 at KP-1 | a0 a1 old_logp adv | ret old_value 0 0], bit exact; without clipping the record is
    the default one (old_value 0) bit for bit."""
    T, N = 7, 13
    rng = np.random.default_rng(O)
    buf = dict(obs=rng.standard_normal((T, N, O)), actions=rng.standard_normal((T, N, 2)),
               log_probs=rng.standard_normal((T, N)), advantages=rng.standard_normal((T, N)),
               returns=rng.standard_normal((T, N)) + 3.0, values=rng.standard_normal((T, N)) - 2.0)
    buf = {k: v.astype(np.float32) for k, v in buf.items()}
    from mobrob_b200.updater import PpoUpdater

    KP = _kp(O)
    plain = PpoUpdater(O, torch.device("cuda", 0)).pack(_dev(buf)).cpu().numpy().reshape(T * N, KP + 8)
    vf = PpoUpdater(O, torch.device("cuda", 0), clip_range_vf=0.2).pack(_dev(buf)).cpu().numpy().reshape(T * N, KP + 8)
    want = np.zeros((T * N, KP + 8), np.float32)
    want[:, :O] = buf["obs"].reshape(T * N, O)
    want[:, KP - 1] = 1.0
    want[:, KP:KP + 2] = buf["actions"].reshape(T * N, 2)
    want[:, KP + 2] = buf["log_probs"].reshape(-1)
    want[:, KP + 3] = buf["advantages"].reshape(-1)
    want[:, KP + 4] = buf["returns"].reshape(-1)
    np.testing.assert_array_equal(plain, want)
    want[:, KP + 5] = buf["values"].reshape(-1)
    np.testing.assert_array_equal(vf, want)


# ---- 2. one minibatch ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["fused", "launches"])
@pytest.mark.parametrize("O,T,N,B", [(14, 16, 64, 100), (26, 16, 64, 100), (14, 296, 64, 18944), (26, 296, 64, 18944)])
def test_one_minibatch_clip_range_vf_matches_autograd(cuda_lib, path, O, T, N, B):
    pol, buf = _vf_problem(O, T, N, seed=O + T)
    up = _updater(pol, O, clip_range_vf=C_VF, **KW)
    dbuf = _dev(buf)
    perm = np.random.default_rng(O).permutation(N * T).astype(np.int64)[:B]
    dperm = torch.as_tensor(perm).cuda()
    stats = up.adv_stats(dbuf["advantages"], dperm, B, N, T)
    g_ref, st = _autograd_vf(pol, buf, perm, torch.float32)
    g_64, _ = _autograd_vf(pol, buf, perm, torch.float64)
    for key in ("vf_low", "vf_high"):   # both bounds bite, and a good share stays inside
        assert 0.15 * B < st[key] < 0.5 * B, (key, st[key], B)
    assert st["vf_low"] + st["vf_high"] < 0.8 * B
    if path == "fused":
        info = torch.zeros((1, 8), device="cuda")
        up.train_epoch_fused(dbuf, dperm, stats, B, N, T, info)
        g = up.grad.cpu().numpy()
        info = info.cpu().numpy()[0]
        norm = np.linalg.norm(g_ref.astype(np.float64))
        np.testing.assert_allclose(info[0], norm, rtol=1e-4)
        assert info[2] == 1.0
        _assert_tail_matches(info[4:], st)
        assert int(up.step[0]) == 1
    else:
        g = up.compute_grad(dbuf, dperm, stats[0], N, T).cpu().numpy()
    _assert_grad_matches(pol, g[:up.n_params], g_ref, g_64)
    _assert_tail_matches(g[up.stride - 16:], st)


# ---- 3. three epochs -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("O", [15, 26])
def test_three_epochs_clip_range_vf_match_sb3_arithmetic(cuda_lib, O):
    """3 epochs of 4.4 minibatches (the last one short), launches and fused, against SB3's PPO.train with
    clip_range_vf: parameters, info rows, Adam moments (test_three_epochs_match_sb3_arithmetic's tolerances)."""
    T, N, B, E = 64, 48, 700, 3
    pol, buf = _vf_problem(O, T, N, seed=O + 5)
    p0 = pol.flat_params().numpy().copy()
    a, b = _updater(pol, O, clip_range_vf=C_VF, **KW), _updater(pol, O, clip_range_vf=C_VF, **KW)
    dbuf = _dev(buf)
    rng = np.random.default_rng(O)
    perms = [rng.permutation(N * T).astype(np.int64) for _ in range(E)]
    n_mb = (N * T + B - 1) // B
    ia, ib = torch.zeros((E * n_mb, 8), device="cuda"), torch.zeros((E * n_mb, 8), device="cuda")
    for e, perm in enumerate(perms):
        dperm = torch.as_tensor(perm).cuda()
        stats = a.adv_stats(dbuf["advantages"], dperm, B, N, T)
        a.train_epoch(dbuf, dperm, stats, B, N, T, ia[e * n_mb:(e + 1) * n_mb])
        b.train_epoch_fused(dbuf, dperm, stats, B, N, T, ib[e * n_mb:(e + 1) * n_mb])
    ref = copy.deepcopy(pol)
    opt = sb3_oracle.make_adam(ref)
    st, stop = X.train_epochs(ref, opt, buf, E, B, perms=perms, clip_range_vf=C_VF, **KW)
    assert stop is None
    assert all(s["vf_low"] > 0 and s["vf_high"] > 0 for s in st)
    p_ref = ref.flat_params().numpy()
    m_ref, _ = _moments(opt)
    moved = np.abs(p_ref - p0).max()
    assert moved > 5e-4
    for name, up, info in (("launches", a, ia), ("fused", b, ib)):
        assert int(up.step[0]) == E * n_mb, name
        err = np.abs(up.params.cpu().numpy() - p_ref).max()
        assert err < 2e-3 * moved + 1e-7, f"{name}: parameters {err:.2e} from SB3's (update {moved:.2e})"
        info = info.cpu().numpy()
        np.testing.assert_allclose(info[:, 0], [s["grad_norm"] for s in st], rtol=1e-3, err_msg=name)
        np.testing.assert_allclose(info[:, 5], [s["value_loss"] for s in st], rtol=1e-3, err_msg=name)
        np.testing.assert_allclose(up.exp_avg.cpu().numpy(), m_ref, rtol=1e-3, atol=1e-7, err_msg=name)


# ---- 4. early stop ---------------------------------------------------------------------------------------------
def _snapshot(up):
    return [t.clone() for t in (up.params, up.exp_avg, up.exp_avg_sq, up.step)]


def _run(up, mode, dbuf, perms, B, N, T, info):
    """Every launch of one update; returns the state copied right after the launch that stopped it (or None)."""
    n = N * T
    n_mb = (n + B - 1) // B
    up.begin_update()
    after_stop = None

    def check():
        nonlocal after_stop
        if after_stop is None and int(up.ctrl[0]) != 0:
            after_stop = _snapshot(up)

    if mode == "fused-one-launch":
        assert n % B == 0
        stats, rows = up.prepare_epochs(dbuf["advantages"], torch.as_tensor(np.stack(perms)).cuda(), B, N, T)
        up.train_epoch_fused(dbuf, None, stats.view(-1, 3), B, N, T, info, rows=rows.view(-1))
        check()
        return after_stop
    for e, perm in enumerate(perms):
        dperm = torch.as_tensor(perm).cuda()
        stats = up.adv_stats(dbuf["advantages"], dperm, B, N, T)
        if mode == "fused-per-epoch":
            up.train_epoch_fused(dbuf, dperm, stats, B, N, T, info[e * n_mb:(e + 1) * n_mb], mb0=e * n_mb)
            check()
        elif mode == "launches-epoch":
            up.train_epoch(dbuf, dperm, stats, B, N, T, info[e * n_mb:(e + 1) * n_mb], mb0=e * n_mb)
        else:   # "launches": mr_ppo_grad + mr_adam_step per minibatch, as the sharded path issues them
            for mb in range(n_mb):
                k = e * n_mb + mb
                up.compute_grad(dbuf, dperm[mb * B:(mb + 1) * B], stats[mb], N, T)
                up.adam_step(info[k], mb_index=k)
                check()
    return after_stop


_MODES = [("fused-one-launch", 512), ("fused-per-epoch", 700), ("launches", 700), ("launches-epoch", 512)]


@pytest.mark.parametrize("O", [14, 26])
@pytest.mark.parametrize("mode,B", _MODES, ids=[m for m, _ in _MODES])
def test_target_kl_stops_where_sb3_stops(cuda_lib, O, mode, B):
    T, N, E = 64, 48, 3
    n_mb = (N * T + B - 1) // B
    pol, buf = _same_policy_problem(O, T, N, seed=O + 11)
    rng = np.random.default_rng(O)
    perms = [rng.permutation(N * T).astype(np.int64) for _ in range(E)]
    ref = copy.deepcopy(pol)
    st_all, _ = X.train_epochs(ref, sb3_oracle.make_adam(ref), buf, E, B, perms=perms, **KW)
    kls = [s["approx_kl"] for s in st_all]
    pick = X.pick_target_kl(kls, n_mb + 1, 2 * n_mb - 1)   # strictly inside the second epoch
    assert pick is not None, kls
    target_kl, j = pick
    margin = min(abs(k / (1.5 * target_kl) - 1.0) for k in kls[:j + 1])
    assert margin >= 0.01, margin
    ref = copy.deepcopy(pol)
    opt = sb3_oracle.make_adam(ref)
    st, stop = X.train_epochs(ref, opt, buf, E, B, perms=perms, target_kl=target_kl, **KW)
    assert stop == j and len(st) == j + 1
    p0 = pol.flat_params().numpy().copy()
    p_ref = ref.flat_params().numpy()
    m_ref, v_ref = _moments(opt)

    up = _updater(pol, O, target_kl=target_kl, **KW)
    info = torch.zeros((E * n_mb, 8), device="cuda")
    after_stop = _run(up, mode, _dev(buf), perms, B, N, T, info)
    assert int(up.ctrl[0]) == j + 1, "evaluated minibatches"
    assert int(up.step[0]) == j, "applied minibatches"
    moved = np.abs(p_ref - p0).max()
    err = np.abs(up.params.cpu().numpy() - p_ref).max()
    assert err < 2e-3 * moved + 1e-7, f"parameters {err:.2e} from SB3's (update {moved:.2e})"
    np.testing.assert_allclose(up.exp_avg.cpu().numpy(), m_ref, rtol=1e-3, atol=1e-7)
    np.testing.assert_allclose(up.exp_avg_sq.cpu().numpy(), v_ref, rtol=1e-3, atol=1e-12)
    info = info.cpu().numpy()[:j + 1]
    np.testing.assert_allclose(info[:j, 0], [s["grad_norm"] for s in st[:j]], rtol=1e-3)
    np.testing.assert_allclose(info[:, 2], np.minimum(np.arange(j + 1) + 1, j))   # the stopping row: step unchanged
    np.testing.assert_allclose(info[:, 3], [s["entropy_loss"] for s in st], rtol=1e-5)
    np.testing.assert_allclose(info[:, 4], [s["policy_loss"] for s in st], rtol=1e-3, atol=1e-6)
    np.testing.assert_allclose(info[:, 5], [s["value_loss"] for s in st], rtol=1e-3)
    np.testing.assert_allclose(info[:, 7], [s["approx_kl"] for s in st], rtol=5e-3, atol=1e-9)
    if after_stop is not None:   # launches after the stopping one changed nothing
        for name, t0, t1 in zip(("params", "exp_avg", "exp_avg_sq", "step"), after_stop, _snapshot(up)):
            assert torch.equal(t0, t1), name


@pytest.mark.parametrize("mode,B", _MODES, ids=[m for m, _ in _MODES])
def test_target_kl_stop_at_first_minibatch(cuda_lib, mode, B):
    """approx_kl of the very first minibatch already exceeds 1.5 target_kl: nothing moves, bit for bit."""
    O, T, N, E = 14, 64, 48, 3
    pol, buf = _make_problem(O, T, N, seed=3)   # rollout policy != trained policy: approx_kl > 0 from the start
    rng = np.random.default_rng(3)
    perms = [rng.permutation(N * T).astype(np.int64) for _ in range(E)]
    ref = copy.deepcopy(pol)
    st, _ = X.train_epochs(ref, sb3_oracle.make_adam(ref), buf, 1, B, perms=perms, **KW)
    target_kl = st[0]["approx_kl"] / 1.5 / 2
    up = _updater(pol, O, target_kl=target_kl, **KW)
    start = _snapshot(up)
    info = torch.zeros((E * ((N * T + B - 1) // B), 8), device="cuda")
    _run(up, mode, _dev(buf), perms, B, N, T, info)
    assert int(up.ctrl[0]) == 1
    for name, t0, t1 in zip(("params", "exp_avg", "exp_avg_sq", "step"), start, _snapshot(up)):
        assert torch.equal(t0, t1), name
    row = info[0].cpu().numpy()
    assert row[2] == 0.0
    _assert_tail_matches(row[4:], st[0])


def test_target_kl_never_reached_matches_default(cuda_lib):
    """A threshold no minibatch reaches: the extended kernel gives the default update's results."""
    O, T, N, B, E = 14, 64, 48, 512, 3
    pol, buf = _make_problem(O, T, N, seed=4)
    rng = np.random.default_rng(4)
    perms = [rng.permutation(N * T).astype(np.int64) for _ in range(E)]
    dbuf = _dev(buf)
    n_mb = N * T // B
    a, b = _updater(pol, O, **KW), _updater(pol, O, target_kl=1e6, **KW)
    ia, ib = torch.zeros((E * n_mb, 8), device="cuda"), torch.zeros((E * n_mb, 8), device="cuda")
    _run(a, "fused-one-launch", dbuf, perms, B, N, T, ia)
    _run(b, "fused-one-launch", dbuf, perms, B, N, T, ib)
    assert int(b.ctrl[0]) == 0 and int(b.step[0]) == int(a.step[0]) == E * n_mb
    p0 = pol.flat_params().cuda()
    moved = float((a.params - p0).abs().max())
    assert float((a.params - b.params).abs().max()) < 2e-3 * moved + 1e-7
    torch.testing.assert_close(ib, ia, rtol=1e-3, atol=1e-6)
    torch.testing.assert_close(b.exp_avg, a.exp_avg, rtol=1e-3, atol=1e-7)


# ---- 5. PPO.learn ----------------------------------------------------------------------------------------------
class _KeepRollouts:
    """learn() callback that keeps a CPU copy of every collected rollout (before its update), the update's device
    stream ids and the clip_range_vf its schedule gives (SB3 evaluates it after the rollout: progress
    1 - num_timesteps / total_timesteps)."""

    def __init__(self, schedule):
        self.schedule, self.bufs, self.stream_ids, self.cvf = schedule, [], [], []

    def init_callback(self, model):
        self.model = model

    def on_training_start(self, *_):
        pass

    def on_rollout_steps(self, _n):
        m = self.model
        self.bufs.append({k: v.cpu().numpy() for k, v in m.buf.items()})
        self.stream_ids.append(m._stream_ids())
        self.cvf.append(float(self.schedule(1.0 - m.num_timesteps / m._total_timesteps)))
        return True

    def on_training_end(self):
        pass


def _train_keys(lg):
    return {k: v for k, v in lg.items() if k.startswith("train/")}


@pytest.mark.parametrize("env_name,cfg,O", [("point", None, 14),
                                            ("car", {"observe_goal_dist": True, "observe_ctrl": True}, 29)],
                         ids=["point14", "car29"])
def test_learn_with_target_kl_and_clip_range_vf(cuda_lib, env_name, cfg, O, capsys):
    """Two PPO.learn() iterations with target_kl and a clip_range_vf schedule, replayed by SB3's PPO.train on the
    rollouts they collected (permutations rebuilt from the device stream ids): parameters, the logged train/* values
    over the evaluated minibatches, train/n_updates = epochs entered, and the schedule evaluated per update."""
    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.ppo import PPO

    n_envs, T, E, B, seed = 64, 32, 3, 512, 7
    n, n_mb = n_envs * T, n_envs * T // B

    def make(target_kl, clip_vf):
        env = GpuVecEnv(env_name, n_envs, seed=None, time_limit=100, terminate_on_goal=True, robot_config=cfg)
        return PPO("MlpPolicy", env, n_steps=T, batch_size=B, n_epochs=E, seed=seed, gae_lambda=0.5, ent_coef=0.05,
                   target_kl=target_kl, clip_range_vf=clip_vf, verbose=1)

    schedule = lambda p: 0.1 + 0.2 * p   # noqa: E731  (progress 0.5 -> 0.2, 0 -> 0.1)
    # the first update's KL sequence without a threshold (same seed and schedule: the same first rollout and update),
    # then a threshold crossing inside its second epoch
    probe = make(None, schedule)
    ref = sb3_oracle.MlpPolicyOracle(O)
    ref.load_state_dict({k: v.cpu() for k, v in probe.policy.state_dict().items()})
    p_init = {k: v.clone() for k, v in ref.state_dict().items()}
    keep = _KeepRollouts(schedule)
    probe.learn(total_timesteps=2 * n, callback=keep)
    perms = [device_permutation(seed, s, n) for s in keep.stream_ids[0]]
    st, _ = X.train_epochs(ref, sb3_oracle.make_adam(ref), keep.bufs[0], E, B, perms=perms, clip_range_vf=keep.cvf[0],
                           **KW)
    target_kl, j = X.pick_target_kl([s["approx_kl"] for s in st], n_mb + 1, 2 * n_mb - 1)

    model = make(target_kl, schedule)
    assert model.updater.obs_dim == O
    logged = []
    dump = model.logger.dump
    model.logger.dump = lambda step=0: (logged.append(dict(model.logger.name_to_value)), dump(step))
    keep = _KeepRollouts(schedule)
    model.learn(total_timesteps=2 * n, callback=keep)
    assert keep.cvf == pytest.approx([0.2, 0.1])
    torch.cuda.synchronize()
    # the second update's train/* (SB3 dumps them with the next iteration): read the snapshot now
    model._drain_episodes(model._snapshot_async())
    model._log_train()
    logged.append(dict(model.logger.name_to_value))

    ref.load_state_dict(p_init)
    opt = sb3_oracle.make_adam(ref)
    n_updates, out = 0, capsys.readouterr().out
    for it, (buf, ids, cvf) in enumerate(zip(keep.bufs, keep.stream_ids, keep.cvf)):
        perms = [device_permutation(seed, s, n) for s in ids]
        st, stop = X.train_epochs(ref, opt, buf, E, B, perms=perms, clip_range_vf=cvf, target_kl=target_kl, **KW)
        if it == 0:
            assert stop == j
        kls = [s["approx_kl"] for s in st]
        assert min(abs(k / (1.5 * target_kl) - 1.0) for k in kls) >= 0.01, "a KL within 1 % of the threshold"
        n_updates += X.epochs_entered(stop, n_mb, E)
        lg = _train_keys(logged[it + 1])
        assert lg["train/n_updates"] == n_updates
        assert lg["train/clip_range_vf"] == pytest.approx(cvf)
        for key, field in (("policy_gradient_loss", "policy_loss"), ("value_loss", "value_loss"),
                           ("entropy_loss", "entropy_loss"), ("clip_fraction", "clip_fraction")):
            np.testing.assert_allclose(lg[f"train/{key}"], np.mean([s[field] for s in st]), rtol=2e-3, atol=1e-6,
                                       err_msg=key)
        np.testing.assert_allclose(lg["train/approx_kl"], np.mean(kls), rtol=5e-3)
        np.testing.assert_allclose(lg["train/loss"], st[-1]["loss"], rtol=2e-3, atol=1e-6)
        if stop is not None:
            assert f"Early stopping at step {stop // n_mb} due to reaching max kl: {kls[-1]:.2f}" in out
    assert model._n_updates == n_updates
    p_ref = ref.flat_params().numpy()
    moved = np.abs(p_ref - torch.cat([p_init[k].reshape(-1) for k in sb3_oracle.PARAM_ORDER]).numpy()).max()
    err = np.abs(model.updater.params.cpu().numpy() - p_ref).max()
    assert err < 2e-3 * moved + 1e-7, (err, moved)


# ---- 6. save / load --------------------------------------------------------------------------------------------
def test_save_load_round_trip_keeps_both_settings(cuda_lib, tmp_path):
    """Both settings are written in SB3's format and restored; a loaded model stops at the same minibatch as the one
    that saved it, on the same rollout and permutations."""
    import json
    import zipfile

    from mobrob_b200 import GpuVecEnv
    from mobrob_b200.ppo import PPO

    n_envs, T, E, B, seed = 64, 32, 3, 512, 5
    n, n_mb = n_envs * T, n_envs * T // B
    env = lambda: GpuVecEnv("point", n_envs, seed=None, time_limit=100, terminate_on_goal=True)  # noqa: E731
    a = PPO("MlpPolicy", env(), n_steps=T, batch_size=B, n_epochs=E, seed=seed, gae_lambda=0.5, ent_coef=0.05,
            clip_range_vf=0.25)
    a.collect_rollouts()
    a.save(tmp_path / "start")
    rng = np.random.default_rng(0)
    perms = [torch.as_tensor(rng.permutation(n).astype(np.int64)) for _ in range(E)]
    a.train(perms=perms)   # the device's KL sequence of this update
    kls = a._log[:, 7].cpu().numpy().astype(np.float64).tolist()
    target_kl, j = X.pick_target_kl(kls, n_mb + 1, 2 * n_mb - 1)

    b = PPO.load(tmp_path / "start", env=env(), target_kl=target_kl)
    assert b.clip_range_vf == 0.25 and b.target_kl == target_kl
    b.save(tmp_path / "b")
    with zipfile.ZipFile(tmp_path / "b.zip") as z:
        data = json.loads(z.read("data"))
    assert data["target_kl"] == target_kl
    assert data["clip_range_vf"]["value"] == 0.25 and data["clip_range_vf"][":type:"] == "<class 'function'>"
    c = PPO.load(tmp_path / "b", env=env())
    assert c.clip_range_vf == 0.25 and c.target_kl == target_kl
    for m in (b, c):
        for k in m.buf:
            m.buf[k].copy_(a.buf[k])
        m.train(perms=perms)
        assert int(m.updater.ctrl[0]) == j + 1
        assert int(m.updater.step[0]) == j
    torch.testing.assert_close(b.updater.params, c.updater.params, rtol=0, atol=1e-5)
    # the shipped zips (both settings null) load as before
    with zipfile.ZipFile(tmp_path / "start.zip") as z:
        assert json.loads(z.read("data"))["target_kl"] is None


def test_ppoctrl_from_config_with_target_kl(cuda_lib):
    from mobrob_b200.rl_control.ppo import PPOCtrl

    cfg = dict(env_name="point", time_limit=100, n_envs=64, vec_env_type="dummy", enable_gui=False, seed=0,
               ppo_kwargs=dict(policy="MlpPolicy", n_steps=32, n_epochs=3, batch_size=512, ent_coef=0.05,
                               gae_lambda=0.5, target_kl=0.01, clip_range_vf=0.2, device="cpu"))
    ctrl = PPOCtrl.from_config(cfg)
    assert ctrl.ppo.target_kl == 0.01 and ctrl.ppo.clip_range_vf == 0.2
    ctrl.learn(total_timesteps=64 * 32)
    ctrl.ppo._settle_updates()
    assert 1 <= ctrl.ppo._n_updates <= 3
