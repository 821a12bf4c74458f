"""clip_range_vf / target_kl without a GPU: constructor validation, the zip fields, and the SB3 restatement's stop rule
(tests/sb3_ext_oracle.py) against oracle/sb3_oracle.py."""
import copy
import json

import numpy as np
import pytest
import torch

import sb3_ext_oracle as X
from oracle import sb3_oracle


def _ppo(**kw):
    from mobrob_b200.ppo import PPO

    return PPO("MlpPolicy", None, **kw)


def test_constructor_accepts_and_validates():
    m = _ppo(clip_range_vf=0.2, target_kl=0.015)
    assert m.clip_range_vf == 0.2 and m.target_kl == 0.015
    m = _ppo(clip_range_vf=lambda p: 0.1 * p)
    assert m.clip_range_vf == pytest.approx(0.1) and m._clip_vf_schedule is not None
    assert _ppo().clip_range_vf is None and _ppo().target_kl is None
    for bad in (0, -0.1):
        with pytest.raises(ValueError, match="clip_range_vf"):
            _ppo(clip_range_vf=bad)
        with pytest.raises(ValueError, match="target_kl"):
            _ppo(target_kl=bad)
    with pytest.raises(NotImplementedError, match="use_sde"):
        _ppo(use_sde=True)


def _json(m):
    from mobrob_b200.spaces import Box

    m.observation_space = Box(-np.inf, np.inf, (14,), np.float32)
    m.action_space = Box(-1.0, 1.0, (2,), np.float32)
    m.n_envs = 1
    return json.loads(json.dumps(m._json_data()))


def test_zip_fields_in_sb3_format():
    from mobrob_b200.ppo import _stored_schedule

    d = _json(_ppo())
    assert d["target_kl"] is None and d["clip_range_vf"] is None
    d = _json(_ppo(clip_range_vf=0.25, target_kl=0.02))
    assert d["target_kl"] == 0.02
    cvf = d["clip_range_vf"]
    assert cvf[":type:"] == "<class 'function'>" and cvf["value"] == 0.25
    assert _stored_schedule(cvf, "clip_range_vf") == 0.25   # what PPO.load passes back to the constructor


def _problem(seed=0, T=16, N=24, O=14):
    torch.manual_seed(seed)
    rng = np.random.default_rng(seed)
    pol = sb3_oracle.MlpPolicyOracle(O)
    obs = (rng.standard_normal((T, N, O)) * 1.5).astype(np.float32)
    with torch.no_grad():
        a, v, lp = pol.forward_with_noise(torch.as_tensor(obs).reshape(T * N, O), torch.randn(T * N, 2))
    buf = dict(obs=obs, actions=a.numpy().reshape(T, N, 2), log_probs=lp.numpy().reshape(T, N),
               advantages=rng.standard_normal((T, N)).astype(np.float32),
               returns=(v.numpy().reshape(T, N) + rng.standard_normal((T, N)).astype(np.float32)),
               values=v.numpy().reshape(T, N) + 0.3 * rng.standard_normal((T, N)).astype(np.float32))
    perms = [rng.permutation(T * N) for _ in range(3)]
    return pol, buf, perms


KW = dict(clip_range=0.2, ent_coef=0.05, vf_coef=0.5)


def test_defaults_compute_what_sb3_oracle_computes():
    pol, buf, perms = _problem()
    a, b = copy.deepcopy(pol), copy.deepcopy(pol)
    st_a = sb3_oracle.train_epochs(a, sb3_oracle.make_adam(a), buf, 3, 100, perms=perms, **KW)
    st_b, stop = X.train_epochs(b, sb3_oracle.make_adam(b), buf, 3, 100, perms=perms, **KW)
    assert stop is None
    assert torch.equal(a.flat_params(), b.flat_params())
    assert [s["value_loss"] for s in st_a] == [s["value_loss"] for s in st_b]


def test_stop_rule_skips_the_step_and_the_rest():
    """The crossing minibatch is evaluated (its stats are returned) but not applied, and nothing after it runs."""
    pol, buf, perms = _problem(1)
    n_mb = (16 * 24 + 99) // 100
    full = copy.deepcopy(pol)
    st, _ = X.train_epochs(full, sb3_oracle.make_adam(full), buf, 3, 100, perms=perms, **KW)
    kls = [s["approx_kl"] for s in st]
    target_kl, j = X.pick_target_kl(kls, n_mb + 1, 2 * n_mb - 1)
    assert min(abs(k / (1.5 * target_kl) - 1) for k in kls[:j + 1]) >= 0.01
    stopped = copy.deepcopy(pol)
    st_s, stop = X.train_epochs(stopped, sb3_oracle.make_adam(stopped), buf, 3, 100, perms=perms,
                                target_kl=target_kl, **KW)
    assert stop == j and len(st_s) == j + 1 and "grad_norm" not in st_s[-1]
    assert X.epochs_entered(stop, n_mb, 3) == 2 and X.epochs_entered(None, n_mb, 3) == 3
    # the same as running exactly the j minibatches before the stop
    ref = copy.deepcopy(pol)
    opt = sb3_oracle.make_adam(ref)
    fl = {key: torch.as_tensor(sb3_oracle.flatten_env_major(buf[key])) for key in buf}
    for k in range(j):
        e, s = divmod(k, n_mb)
        idx = np.asarray(perms[e])[s * 100:(s + 1) * 100]
        b = torch.as_tensor(idx.astype(np.int64))
        sb3_oracle.train_minibatch(ref, opt, (fl["obs"][b], fl["actions"][b], fl["log_probs"][b].flatten(),
                                              fl["advantages"][b].flatten(), fl["returns"][b].flatten()), **KW)
    assert torch.equal(ref.flat_params(), stopped.flat_params())


def test_clip_range_vf_value_loss():
    """values_pred = old + clamp(V - old, -c, c): the logged value_loss is the clipped MSE, and both bounds bite."""
    pol, buf, _ = _problem(2)
    idx = np.arange(64)
    fl = {k: torch.as_tensor(sb3_oracle.flatten_env_major(buf[k]))[torch.as_tensor(idx)] for k in buf}
    old = fl["values"].flatten()
    c = 0.1
    loss, st = X.ppo_loss(pol, fl["obs"], fl["actions"], fl["log_probs"].flatten(), fl["advantages"].flatten(),
                          fl["returns"].flatten(), old, clip_range_vf=c, **KW)
    with torch.no_grad():
        _, v = pol.mean_value(fl["obs"])
    pred = old + torch.clamp(v - old, -c, c)
    np.testing.assert_allclose(st["value_loss"], float(((fl["returns"].flatten() - pred) ** 2).mean()), rtol=1e-6)
    assert st["vf_low"] > 0 and st["vf_high"] > 0
