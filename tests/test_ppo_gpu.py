"""GPU numerics of the PPO rollout kernels against plain PyTorch / NumPy fp32-fp64 references of the same ops
(stable_baselines3 semantics restated in SURVEY.md section 8 u10)."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def model():
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(1000, preset="waypoints_v3", seed=5)
    m = PPO("MlpPolicy", env, n_steps=16, batch_size=4000, n_epochs=2, seed=5, ent_coef=0.001)
    with torch.no_grad():   # make the towers non-trivial: bias and log_std away from their zero init
        m.policy.theta.add_(0.05 * torch.randn(m.policy.count, device=m.device, generator=m._gen))
    yield m
    env.close()


def test_param_layout_counts(model):
    assert model.policy.count == 12361 and model.d == 28
    assert model.policy.view("action_net.weight").shape == (4, 64)


def test_running_moments_match_sb3_formula(model):
    from pyflyt_drone_b200 import _lib
    from pyflyt_drone_b200.ppo import DeviceVecNormalize, _p, _stream
    vn = DeviceVecNormalize(28, 3000, model.device)
    rng = np.random.default_rng(0)
    mean, var, count = np.zeros(28), np.ones(28), 1e-4
    for it in range(4):
        x = (rng.normal(size=(3000, 28)) * rng.uniform(0.1, 30, 28) + rng.uniform(-50, 50, 28)).astype(np.float32)
        xt = torch.from_numpy(x).to(model.device)
        _lib.check(model.lib.ppo_moments_update(_p(xt), 3000, 28, _p(vn.obs_stats), _p(vn.obs_scratch), _p(vn.obs_accum),
                                                _stream()))
        bm, bv, bc = x.astype(np.float64).mean(0), x.astype(np.float64).var(0), 3000
        delta, tot = bm - mean, count + bc
        m2 = var * count + bv * bc + delta ** 2 * count * bc / tot
        mean, var, count = mean + delta * bc / tot, m2 / tot, tot
    got = vn.obs_stats.cpu().numpy()
    assert np.allclose(got[:28], mean, rtol=1e-6, atol=1e-6)
    assert np.allclose(got[28:56], var, rtol=1e-5)
    assert got[56] == pytest.approx(count)
    assert float(vn.obs_scratch.abs().max()) == 0.0
    # the raw-sum accumulator reproduces the same statistics through the host-side merge
    merged = DeviceVecNormalize._merge(vn.obs_base, vn.obs_accum, 28).cpu().numpy()
    assert np.allclose(merged[:28], mean, rtol=1e-5, atol=1e-5) and np.allclose(merged[28:56], var, rtol=1e-4)


def test_policy_forward_matches_torch(model):
    from pyflyt_drone_b200 import _lib
    from pyflyt_drone_b200.ppo import _p, _stream
    N, D = 1000, 28
    dev = model.device
    obs = (torch.randn(N, D, device=dev, generator=model._gen) * 20).contiguous()
    stats = model.vecnorm.obs_stats
    stats[:D] = torch.linspace(-3, 3, D, dtype=torch.float64)
    stats[D:2 * D] = torch.linspace(0.5, 90, D, dtype=torch.float64)
    obs_norm = torch.zeros(N, D, device=dev); act_env = torch.zeros(N, 4, device=dev); act_raw = torch.zeros(N, 4, device=dev)
    logp = torch.zeros(N, device=dev); val = torch.zeros(N, device=dev)
    _lib.check(model.lib.ppo_policy_forward(_p(model.policy.theta), D, _p(obs), _p(stats), 10.0, N, 77, 0, 3, None, 0, _p(obs_norm),
                                            _p(act_env), _p(act_raw), _p(logp), _p(val), _stream()))
    ref_norm = torch.clamp((obs.double() - stats[:D]) / torch.sqrt(stats[D:2 * D] + 1e-8), -10, 10).float()
    assert torch.allclose(obs_norm, ref_norm, atol=2e-6, rtol=1e-6)
    with torch.no_grad():
        torch.backends.cuda.matmul.allow_tf32 = False
        mean, value = model.policy.towers(ref_norm)
        v2, lp2, ent = model.policy.evaluate_actions(ref_norm, act_raw)
    assert torch.allclose(val, value, atol=2e-5, rtol=1e-5)
    assert torch.allclose(logp, lp2, atol=2e-4, rtol=1e-5)        # log-prob of the sampled (unclipped) action
    assert torch.equal(act_env, act_raw.clamp(-1, 1))
    eps = (act_raw - mean) * torch.exp(-model.policy.view("log_std"))
    assert abs(float(eps.detach().mean())) < 0.06 and abs(float(eps.detach().std()) - 1) < 0.05
    # deterministic mode returns the mean; a different step index draws different noise
    det = torch.zeros(N, 4, device=dev)
    _lib.check(model.lib.ppo_policy_forward(_p(model.policy.theta), D, _p(obs), _p(stats), 10.0, N, 77, 0, 3, None, 1, None,
                                            _p(det), None, None, _p(val), _stream()))
    assert torch.allclose(det, mean.clamp(-1, 1), atol=2e-5)
    v_only = torch.zeros(N, device=dev)
    _lib.check(model.lib.ppo_value_forward(_p(model.policy.theta), D, _p(obs), _p(stats), 10.0, N, _p(v_only), _stream()))
    assert torch.allclose(v_only, value, atol=2e-5, rtol=1e-5)


def test_tensor_core_forward_matches_fp32_within_tf32_tolerance(model):
    """tcgen05 kind::tf32 path vs the fp32 torch towers.  TF32 keeps 10 mantissa bits: pre-activations carry
    ~5e-4 relative error, so means / values agree to ~5e-3 absolute and log-probs (sigma = 1) likewise."""
    from pyflyt_drone_b200 import _lib
    from pyflyt_drone_b200.ppo import _p, _stream
    D, dev = 28, model.device
    for N in (1, 127, 128, 1000, 40000):
        obs = (torch.randn(N, D, device=dev, generator=model._gen) * 20).contiguous()
        stats = model.vecnorm.obs_stats
        stats[:D] = torch.linspace(-3, 3, D, dtype=torch.float64)
        stats[D:2 * D] = torch.linspace(0.5, 90, D, dtype=torch.float64)
        outs = {}
        for name, fn in (("tc", model.lib.ppo_policy_forward_tc), ("cc", model.lib.ppo_policy_forward)):
            o = dict(obs_norm=torch.zeros(N, D, device=dev), act_env=torch.zeros(N, 4, device=dev),
                     act_raw=torch.zeros(N, 4, device=dev), logp=torch.zeros(N, device=dev), val=torch.zeros(N, device=dev))
            _lib.check(fn(_p(model.policy.theta), D, _p(obs), _p(stats), 10.0, N, 77, 5, 3, None, 0, _p(o["obs_norm"]),
                          _p(o["act_env"]), _p(o["act_raw"]), _p(o["logp"]), _p(o["val"]), _stream()))
            outs[name] = o
        torch.cuda.synchronize()
        tc, cc = outs["tc"], outs["cc"]
        assert torch.equal(tc["obs_norm"], cc["obs_norm"])
        assert torch.equal(tc["logp"], cc["logp"])                    # same noise stream, log-prob depends on eps only
        assert float((tc["val"] - cc["val"]).abs().max()) < 1e-2
        assert float((tc["act_raw"] - cc["act_raw"]).abs().max()) < 1e-2
        with torch.no_grad():
            mean, value = model.policy.towers(cc["obs_norm"])
            _, lp, _ = model.policy.evaluate_actions(cc["obs_norm"], tc["act_raw"])
        assert float((tc["val"] - value).abs().max()) < 1e-2
        assert float((lp - tc["logp"]).abs().max()) < 3e-2            # what the PPO ratio sees at epoch 0
        assert float((lp - tc["logp"]).abs().mean()) < 3e-3


def test_reward_normalize_and_bootstrap(model):
    from pyflyt_drone_b200 import _lib
    from pyflyt_drone_b200.ppo import DeviceVecNormalize, _p, _stream
    N, D, dev = 1000, 28, model.device
    vn = DeviceVecNormalize(D, N, dev)
    rng = np.random.default_rng(1)
    ret = np.zeros(N); mean, var, count = 0.0, 1.0, 1e-4
    for it in range(3):
        rew = rng.normal(size=N).astype(np.float32) * 5
        flags = (rng.uniform(size=N) < 0.1).astype(np.uint8) * rng.integers(1, 4, N).astype(np.uint8)
        r_t, f_t = torch.from_numpy(rew).to(dev), torch.from_numpy(flags).to(dev)
        out, done = torch.zeros(N, device=dev), torch.zeros(N, device=dev)
        _lib.check(model.lib.ppo_reward_normalize(_p(r_t), _p(f_t), N, 0.99, 10.0, _p(vn.ret), _p(vn.ret_stats),
                                                  _p(vn.ret_scratch), _p(vn.ret_accum), _p(out), _p(done), _stream()))
        ret = ret * 0.99 + rew
        bm, bv = ret.mean(), ret.var()
        delta, tot = bm - mean, count + N
        m2 = var * count + bv * N + delta ** 2 * count * N / tot
        mean, var, count = mean + delta * N / tot, m2 / tot, tot
        expect = np.clip(rew / np.sqrt(var + 1e-8), -10, 10)
        d = (flags & 3) != 0
        ret[d] = 0
        assert np.allclose(out.cpu().numpy(), expect, rtol=2e-5, atol=1e-6)
        assert np.array_equal(done.cpu().numpy() > 0.5, d)
        assert np.allclose(vn.ret.cpu().numpy(), ret, rtol=1e-5, atol=1e-5)
    # bootstrap: only truncated-and-not-terminated rows get gamma * V(terminal obs)
    term = (torch.randn(N, D, device=dev, generator=model._gen) * 10).contiguous()
    flags = torch.from_numpy(rng.integers(0, 4, N).astype(np.uint8)).to(dev)
    rew = torch.zeros(N, device=dev)
    stats = model.vecnorm.obs_stats
    scratch = torch.zeros(N, device=dev)
    _lib.check(model.lib.ppo_timeout_bootstrap(_p(model.policy.theta), D, _p(term), _p(stats), 10.0, _p(flags), N, 0.99,
                                               _p(rew), _p(scratch), _stream()))
    with torch.no_grad():
        norm = torch.clamp((term.double() - stats[:D]) / torch.sqrt(stats[D:2 * D] + 1e-8), -10, 10).float()
        _, v = model.policy.towers(norm)
    mask = flags == 2
    assert torch.allclose(rew[mask], 0.99 * v[mask], atol=3e-5, rtol=1e-5)
    assert float(rew[~mask].abs().max()) == 0.0


def test_gae_matches_sb3_loop(model):
    from pyflyt_drone_b200 import _lib
    from pyflyt_drone_b200.ppo import _p, _stream
    T, N, dev = 37, 777, model.device
    g = model._gen
    rew = torch.randn(T, N, device=dev, generator=g); val = torch.randn(T, N, device=dev, generator=g)
    done = (torch.rand(T, N, device=dev, generator=g) < 0.1).float(); last = torch.randn(N, device=dev, generator=g)
    adv, ret = torch.zeros(T, N, device=dev), torch.zeros(T, N, device=dev)
    _lib.check(model.lib.ppo_gae(_p(rew), _p(val), _p(done), _p(last), T, N, 0.99, 0.95, _p(adv), _p(ret), _stream()))
    r, v, d, l = rew.double().cpu(), val.double().cpu(), done.double().cpu(), last.double().cpu()
    exp = torch.zeros(T, N, dtype=torch.float64)
    gae = torch.zeros(N, dtype=torch.float64)
    for t in reversed(range(T)):
        nv = l if t == T - 1 else v[t + 1]
        nnt = 1.0 - d[t]
        delta = r[t] + 0.99 * nv * nnt - v[t]
        gae = delta + 0.99 * 0.95 * nnt * gae
        exp[t] = gae
    assert torch.allclose(adv.cpu().double(), exp, atol=1e-4, rtol=1e-5)
    assert torch.allclose(ret.cpu().double(), exp + v, atol=1e-4, rtol=1e-5)


def test_learn_runs_and_counts_timesteps(model):
    before = model.policy.theta.detach().clone()
    model.learn(2 * 16 * 1000)
    assert model.num_timesteps == 2 * 16 * 1000
    assert torch.isfinite(model.policy.theta).all() and not torch.equal(before, model.policy.theta)
    b = model.buf
    assert torch.isfinite(b["adv"]).all() and torch.isfinite(b["obs"]).all()
    assert float(b["obs"].abs().max()) <= 10.0 + 1e-5
    # stored log-probs are consistent with the stored (normalised obs, raw action) pairs under the policy that
    # generated them -- re-collect one rollout and compare before any update
    model.collect_rollouts()
    with torch.no_grad():
        _, lp, _ = model.policy.evaluate_actions(b["obs"].view(-1, 28), b["act"].view(-1, 4))
    err = (lp - b["logp"].view(-1)).abs()
    if model.tensor_core_forward:       # TF32 tensor-core rollout vs fp32 re-evaluation
        assert float(err.max()) < 3e-2 and float(err.mean()) < 3e-3
    else:
        assert float(err.max()) < 5e-4


def test_checkpoint_round_trip(model, tmp_path):
    p = str(tmp_path / "ck.pt")
    model.save(p)
    sd = model.policy.state_dict()
    assert "mlp_extractor.policy_net.0.weight" in sd and "value_net.bias" in sd and "log_std" in sd
    theta = model.policy.theta.detach().clone()
    with torch.no_grad():
        model.policy.theta.zero_()
    model.load(p)
    assert torch.equal(theta, model.policy.theta)


def _torch_minibatch_grad(model, idx):
    """Plain PyTorch fp32 reference of one SB3 PPO minibatch gradient on the flat parameter vector."""
    b = model.buf
    D = model.d
    obs, act = b["obs"].view(-1, D)[idx], b["act"].view(-1, model.a)[idx]
    adv, ret, lp_old = b["adv"].view(-1)[idx], b["ret"].view(-1)[idx], b["logp"].view(-1)[idx]
    a = (adv - adv.mean()) / (adv.std() + 1e-8)
    torch.backends.cuda.matmul.allow_tf32 = False
    values, logp, entropy = model.policy.evaluate_actions(obs, act)
    ratio = torch.exp(logp - lp_old)
    pl = -torch.min(a * ratio, a * torch.clamp(ratio, 1 - model.clip_range, 1 + model.clip_range)).mean()
    vl = torch.nn.functional.mse_loss(ret, values)
    loss = pl - model.ent_coef * entropy.mean() + model.vf_coef * vl
    model.policy.theta.grad = None
    loss.backward()
    g = model.policy.theta.grad.detach().clone()
    model.policy.theta.grad = None
    return g, float(pl.detach()), float(vl.detach()), float(((ratio - 1) - (logp - lp_old)).mean().detach())


def _check_fused_gradient(model, batch):
    model.collect_rollouts()
    with torch.no_grad():      # move the policy away from the data-collecting one so that ratios / clipping are live
        model.policy.theta.add_(0.01 * torch.randn(model.policy.count, device=model.device, generator=model._gen))
    total = model.n_steps * model.n_envs
    perm = torch.randperm(total, device=model.device, generator=model._gen)
    # Samples whose ratio sits within 3e-3 of a clip boundary are left out: there the indicator 1[unclipped] depends on
    # whether the forward pass ran in TF32 or fp32, which is a property of the loss (a jump), not of the kernel.
    with torch.no_grad():
        b = model.buf
        _, lp_all, _ = model.policy.evaluate_actions(b["obs"].view(-1, model.d), b["act"].view(-1, model.a))
        ratio_all = torch.exp(lp_all - b["logp"].view(-1))
        safe = ((ratio_all - (1 - model.clip_range)).abs() > 3e-3) & ((ratio_all - (1 + model.clip_range)).abs() > 3e-3)
    idx = perm[safe[perm]][:batch]
    assert idx.numel() == batch
    ref, pl, vl, kl = _torch_minibatch_grad(model, idx)
    got = torch.zeros_like(ref)
    stats = torch.zeros(8, device=model.device)
    model._minibatch_grad_kernel(idx, got, stats)
    torch.cuda.synchronize()
    for name, (a, b, shp) in model.policy.slices.items():
        r, g = ref[a:b], got[a:b]
        rel = float((g - r).norm() / (r.norm() + 1e-12))
        cos = float(torch.dot(g, r) / (g.norm() * r.norm() + 1e-20))
        assert rel < 4e-2 and cos > 0.999, (name, rel, cos, float(r.norm()))
    assert float((got - ref).norm() / ref.norm()) < 2e-2
    n = float(stats[5])
    assert n == batch
    assert float(stats[0]) / n == pytest.approx(pl, rel=2e-2, abs=2e-3)
    assert float(stats[1]) / n == pytest.approx(vl, rel=2e-2, abs=2e-3)
    assert float(stats[2]) / n == pytest.approx(kl, rel=5e-2, abs=1e-3)


@pytest.mark.parametrize("batch", [100, 128, 4000, 12000])
def test_fused_tensor_core_gradient_matches_torch_autograd(model, batch):
    """ppo_minibatch_grad (tcgen05: TF32 forward, bf16 backward operands, fp32 accumulate) vs torch autograd in fp32.
    Tolerance per parameter tensor: relative L2 error <= 4e-2 and cosine >= 0.999 (bf16 backward operands, TF32 +
    MUFU.TANH forward), on samples away from the PPO clip boundary."""
    _check_fused_gradient(model, batch)


@pytest.mark.parametrize("batch", [100, 4000])
def test_fused_gradient_for_the_six_channel_policy(batch):
    """The same kernel compiled for action width 6 (csrc/ppo_update_tc_a6.cu): the low-level env's MlpPolicy, D = 21, A = 6
    (train/train_lowlevel_cmd.py:97-110)."""
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(512, preset="lowlevel", seed=5)
    m = PPO("MlpPolicy", env, n_steps=32, batch_size=4096, n_epochs=2, ent_coef=0.001, seed=5, use_cuda_graph=False)
    assert m.a == 6 and m.d == 21 and m.update == "kernel"
    with torch.no_grad():      # the action head starts near zero (gain 0.01): give every gradient path signal
        m.policy.theta.add_(0.05 * torch.randn(m.policy.count, device=m.device, generator=m._gen))
    _check_fused_gradient(m, batch)
    env.close()


@pytest.mark.parametrize("batch", [100, 4000])
def test_fused_gradient_for_the_56_float_duck_observation(batch):
    """The same kernel compiled with a 64-wide layer-1 slab (csrc/ppo_update_tc_d64.cu; layer 2 of the forward pass as a
    bf16 hi/lo split): the duck-only ObjLock policy, D = 56, A = 4 (train/train_objlock.py:186-290)."""
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(512, preset="objlock_duck", seed=5)
    m = PPO("MlpPolicy", env, n_steps=32, batch_size=4096, n_epochs=2, ent_coef=0.001, seed=5, use_cuda_graph=False)
    assert m.a == 4 and m.d == 56 and m.update == "kernel"
    with torch.no_grad():
        m.policy.theta.add_(0.05 * torch.randn(m.policy.count, device=m.device, generator=m._gen))
    _check_fused_gradient(m, batch)
    env.close()


def test_random_permutation_is_a_fresh_bijection_every_epoch(model):
    """RolloutBuffer.get draws np.random.permutation(n) per epoch; the kernel's keyed Feistel bijection must be a
    permutation for awkward sizes (cycle walking) and change with the epoch and the seed."""
    import ctypes as C
    lib = model.lib
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for n in (1, 2, 3, 127, 4096, 100003, 65536 * 64):
        a = torch.empty(n, dtype=torch.int64, device="cuda")
        b = torch.empty_like(a)
        c = torch.empty_like(a)
        assert lib.ppo_random_permutation(C.c_void_p(a.data_ptr()), n, 7, 1, st) == 0
        assert lib.ppo_random_permutation(C.c_void_p(b.data_ptr()), n, 7, 2, st) == 0
        assert lib.ppo_random_permutation(C.c_void_p(c.data_ptr()), n, 8, 1, st) == 0
        ar = torch.arange(n, device="cuda")
        for p in (a, b, c):
            assert torch.equal(torch.sort(p).values, ar), n
        if n >= 4096:
            assert (a != b).float().mean() > 0.99 and (a != c).float().mean() > 0.99
            assert (a != ar).float().mean() > 0.99
            # no obvious structure: neighbouring outputs are far apart on average (a sorted or strided order is not)
            d = (a[1:] - a[:-1]).abs().double().mean().item()
            assert 0.2 * n < d < 0.5 * n, (n, d)


def test_windowed_permutation_walks_the_same_permutation(model):
    """ppo_random_permutation_window (device-side epoch / window counters) yields exactly the slices of
    ppo_random_permutation, window after window, and rolls over to the next epoch's permutation."""
    import ctypes as C
    lib = model.lib
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    n, wl = 10000, 2048                      # five windows per epoch, the last one short
    ctr = torch.tensor([7, 0], dtype=torch.int32, device="cuda")
    full = torch.empty(n, dtype=torch.int64, device="cuda")
    for epoch in (7, 8):
        assert lib.ppo_random_permutation(C.c_void_p(full.data_ptr()), n, 99, epoch, st) == 0
        for w in range(5):
            win = torch.full((wl,), -1, dtype=torch.int64, device="cuda")
            assert lib.ppo_random_permutation_window(C.c_void_p(win.data_ptr()), n, 99, C.c_void_p(ctr.data_ptr()), wl, st) == 0
            m = min(wl, n - w * wl)
            assert torch.equal(win[:m], full[w * wl:w * wl + m]) and bool((win[m:] == -1).all())
    assert ctr.tolist() == [9, 0]


def test_graph_replayed_update_equals_the_eager_update():
    """From the second train() call on, windows of optimizer steps run as one replayed CUDA graph: from the same rollout
    buffer, parameters and optimizer state, the graph-replayed update and the eager loop end bit-identical (parameters, Adam
    moments, step and epoch counters)."""
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(256, preset="waypoints_v3", seed=9)
    m = PPO("MlpPolicy", env, n_steps=16, batch_size=128, n_epochs=3, seed=9)
    m.update_graph_steps = 8                 # 32 minibatches per epoch -> four windows of eight
    m.fused_steps_max_batch = 0              # not the single-CTA multi-step kernel: the launch-per-kernel path under test
    m.collect_rollouts()
    m.train()                                # first call: eager warm-up
    snap = [t.clone() for t in (m.policy.theta.data, m._adam_m, m._adam_v, m._adam_t)]
    epoch0 = m._perm_epoch
    out = {}
    for mode in (True, False):
        for dst, src in zip((m.policy.theta.data, m._adam_m, m._adam_v, m._adam_t), snap):
            dst.copy_(src)
        m._perm_epoch = epoch0
        m.update_graph = mode
        m.train()
        torch.cuda.synchronize()
        out[mode] = (m.policy.theta.detach().clone(), m._adam_m.clone(), m._adam_v.clone(), int(m._adam_t), m._perm_epoch,
                     m._stats_mb.clone())
    assert m._ugraph is not None
    assert out[True][3] == out[False][3] == 2 * 3 * 32 and out[True][4] == out[False][4] == epoch0 + 3
    assert not torch.equal(out[True][0], snap[0])
    for a, b in zip(out[True][:3] + out[True][5:], out[False][:3] + out[False][5:]):
        assert torch.equal(a, b)
    env.close()


@pytest.mark.parametrize("preset,batch", [("waypoints_v3", 128), ("waypoints_v3", 200), ("lowlevel", 128), ("objlock_duck", 128),
                                          ("waypoints_v3", 1)])
def test_single_cta_optimizer_steps_equal_the_launch_per_kernel_update(preset, batch):
    """ppo_minibatch_steps_a (a window of optimizer steps in one single-CTA launch: advantage statistics, gradient, clip,
    Adam per step) against the same steps as separate launches (ppo_minibatch_grad_a + ppo_adam_step): same gradient kernel
    body, so parameters after 12 steps agree to fp32 reduction-order noise, step counter and last-step statistics match."""
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(256, preset=preset, seed=4)
    m = PPO("MlpPolicy", env, n_steps=16, batch_size=batch, n_epochs=1, seed=4, use_cuda_graph=False)
    m.collect_rollouts()
    with torch.no_grad():
        m.policy.theta.add_(0.02 * torch.randn(m.policy.count, device=m.device, generator=m._gen))
    snap = [t.clone() for t in (m.policy.theta.data, m._adam_m, m._adam_v, m._adam_t)]
    perm = m._epoch_permutation(16 * 256).clone()
    steps, out = 12, {}
    for fused in (True, False):
        for dst, src in zip((m.policy.theta.data, m._adam_m, m._adam_v, m._adam_t), snap):
            dst.copy_(src)
        if fused:
            b = m.buf
            _lib_check = __import__("pyflyt_drone_b200")._lib.check
            from pyflyt_drone_b200.ppo import _p, _stream
            _lib_check(m.lib.ppo_minibatch_steps_a(
                _p(m.policy.theta.data), m.d, m.a, _p(b["obs"]), _p(b["act"]), _p(b["logp"]), _p(b["adv"]), _p(b["ret"]),
                _p(perm), batch, steps, m.clip_range, m.ent_coef, m.vf_coef, _p(m._adam_m), _p(m._adam_v), 3e-4, 0.9, 0.999, 1e-5,
                m.max_grad_norm, _p(m._adam_t), _p(m._grad_norm), _p(m._grad), _p(m._stats_mb), _stream()))
        else:
            for k in range(steps):
                m._optimizer_step(perm[k * batch:(k + 1) * batch], 3e-4, 0.9, 0.999, 1e-5)
        torch.cuda.synchronize()
        out[fused] = (m.policy.theta.detach().clone(), m._adam_m.clone(), m._adam_v.clone(), int(m._adam_t), m._stats_mb.clone(),
                      float(m._grad_norm), m._grad.clone())
    assert out[True][3] == out[False][3] == int(snap[3]) + steps
    moved = float((out[False][0] - snap[0]).abs().max())
    assert moved > 1e-3
    assert float((out[True][0] - out[False][0]).abs().max()) < 1e-3 * moved
    assert torch.allclose(out[True][1], out[False][1], rtol=1e-3, atol=1e-6) and torch.allclose(out[True][2], out[False][2], rtol=1e-3, atol=1e-9)
    assert torch.allclose(out[True][4], out[False][4], rtol=1e-3, atol=1e-4) and float(out[True][4][5]) == batch
    assert out[True][5] == pytest.approx(out[False][5], rel=1e-3)
    assert float((out[True][6] - out[False][6]).norm() / out[False][6].norm()) < 1e-3
    env.close()


@pytest.mark.parametrize("preset,batch", [("waypoints_v3", 1000), ("lowlevel", 512), ("objlock_duck", 700), ("waypoints_v3", 1)])
def test_window_update_is_bit_identical_to_separate_launches(preset, batch):
    """ppo_window_update_a (one advantage-statistics launch per window, clip + Adam by the last block of the gradient
    reduction) against ppo_minibatch_grad_a + ppo_adam_step per minibatch: same kernels' arithmetic, so parameters, Adam
    moments, step counter, gradient, norm and statistics are bit-identical."""
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(256, preset=preset, seed=4)
    m = PPO("MlpPolicy", env, n_steps=16, batch_size=batch, n_epochs=1, seed=4, use_cuda_graph=False)
    m.collect_rollouts()
    with torch.no_grad():
        m.policy.theta.add_(0.02 * torch.randn(m.policy.count, device=m.device, generator=m._gen))
    snap = [t.clone() for t in (m.policy.theta.data, m._adam_m, m._adam_v, m._adam_t)]
    perm = m._epoch_permutation(16 * 256).clone()
    nmb, out = 4, {}
    for window in (True, False):
        for dst, src in zip((m.policy.theta.data, m._adam_m, m._adam_v, m._adam_t), snap):
            dst.copy_(src)
        if window:
            m._window_steps(perm[:nmb * batch], batch, nmb, 3e-4, 0.9, 0.999, 1e-5)
        else:
            for k in range(nmb):
                m._optimizer_step(perm[k * batch:(k + 1) * batch], 3e-4, 0.9, 0.999, 1e-5)
        torch.cuda.synchronize()
        out[window] = (m.policy.theta.detach().clone(), m._adam_m.clone(), m._adam_v.clone(), m._adam_t.clone(), m._stats_mb.clone(),
                       m._grad_norm.clone(), m._grad.clone())
    assert int(out[True][3]) == int(snap[3]) + nmb and not torch.equal(out[True][0], snap[0])
    for a, b in zip(out[True], out[False]):
        assert torch.equal(a, b)
    env.close()


@pytest.mark.parametrize("preset,n", [("waypoints_v3", 1000), ("lowlevel", 4096), ("waypoint_objlock", 700), ("objlock_duck", 333)])
def test_obs_moments_accumulated_by_the_step_kernels(preset, n):
    """SURVEY 8 f1: the env-step kernels add the column sums / sums of squares of the observations they return to the
    accumulator slots (fw_set_obs_accumulator); ppo_moments_finalize folds them into the running statistics like
    RunningMeanStd.update.  Checked against NumPy on the very observations the steps returned, over three steps, for every
    step kernel (K1 Waypoints / low-level, K3 ObjLock / duck-only) and ragged batch sizes."""
    from pyflyt_drone_b200 import _lib
    from pyflyt_drone_b200.ppo import DeviceVecNormalize, _p, _stream
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(n, preset=preset, seed=6)
    env.reset_tensor()
    d, dev = env.obs_dim, torch.device("cuda", 0)
    vn = DeviceVecNormalize(d, n, dev)
    acc = torch.zeros(64 * 2 * d, dtype=torch.float64, device=dev)
    env.set_obs_accumulator(acc)
    g = torch.Generator(device=dev).manual_seed(1)
    mean, var, count = np.zeros(d), np.ones(d), 1e-4
    plib = _lib.load()
    for _ in range(3):
        a = (torch.rand(n, env.act_dim, device=dev, generator=g) * 2 - 1).contiguous()
        obs = env.step_tensor(a, want_terminal_obs=False)[0]
        _lib.check(plib.ppo_moments_finalize(_p(acc), 64, n, d, _p(vn.obs_stats), _p(vn.obs_accum), _stream()))
        x = obs.cpu().numpy().astype(np.float64)
        bm, bv = x.mean(0), x.var(0)
        tot = count + n
        delta = bm - mean
        m2 = var * count + bv * n + delta ** 2 * count * n / tot
        mean, var, count = mean + delta * n / tot, m2 / tot, tot
    torch.cuda.synchronize()
    got = vn.obs_stats.cpu().numpy()
    assert float(acc.abs().max()) == 0.0                        # slots are left zeroed
    assert got[2 * d] == pytest.approx(count)
    assert np.allclose(got[:d], mean, rtol=1e-5, atol=1e-5)
    assert np.allclose(got[d:2 * d], var, rtol=1e-4, atol=1e-6)
    env.set_obs_accumulator(None)
    env.step_tensor(a, want_terminal_obs=False)
    torch.cuda.synchronize()
    assert float(acc.abs().max()) == 0.0                        # cleared accumulator: steps add nothing
    env.close()


def test_adam_step_matches_torch_optim(model):
    from pyflyt_drone_b200 import _lib
    from pyflyt_drone_b200.ppo import _p, _stream
    P, dev = model.policy.count, model.device
    g = model._gen
    theta = torch.randn(P, device=dev, generator=g) * 0.1
    ref = torch.nn.Parameter(theta.clone())
    opt = torch.optim.Adam([ref], lr=3e-4, eps=1e-5)
    mine = theta.clone()
    m, v = torch.zeros(P, device=dev), torch.zeros(P, device=dev)
    t = torch.zeros(1, dtype=torch.int32, device=dev)
    norm = torch.zeros(1, device=dev)
    for it in range(5):
        grad = torch.randn(P, device=dev, generator=g) * (0.001 if it % 2 else 0.05)      # below and above the clip norm
        ref.grad = (grad / 2).clone()
        ref_norm = torch.nn.utils.clip_grad_norm_([ref], 0.5)
        opt.step()
        _lib.check(model.lib.ppo_adam_step(_p(mine), _p(grad), _p(m), _p(v), P, 3e-4, 0.9, 0.999, 1e-5, 0.5, 0.5, _p(t), _p(norm),
                                           _stream()))
        torch.cuda.synchronize()
        assert float(norm) == pytest.approx(float(ref_norm), rel=1e-5)
        assert torch.allclose(mine, ref.detach(), atol=1e-7, rtol=1e-5)
    assert int(t) == 5


def test_kernel_update_learns_like_the_torch_update():
    """Same seed, same rollouts at iteration 0: after one PPO iteration the two update paths must land on nearly
    the same parameters (TF32 + MUFU.TANH forward / bf16 backward vs fp32 gradients through 8 Adam steps)."""
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    out = {}
    for mode in ("kernel", "torch"):
        env = FixedwingVecEnv(512, preset="waypoints_v3", seed=9)
        m = PPO("MlpPolicy", env, n_steps=16, batch_size=2048, n_epochs=2, seed=9, ent_coef=0.001, update=mode,
                tensor_core_forward=False, use_cuda_graph=False)
        m.learn(16 * 512)
        out[mode] = m.policy.theta.detach().clone()
        env.close()
    theta0 = FlatInit.theta(28, 9)
    dk, dt = out["kernel"] - theta0, out["torch"] - theta0
    moved = dt.abs().max()
    assert float(moved) > 1e-4
    # Adam normalises every coordinate's step to ~lr, so coordinates with near-zero gradients amplify the TF32/bf16
    # rounding of the kernel path; the displacement as a whole must agree in direction and size.
    cos = float(torch.dot(dk, dt) / (dk.norm() * dt.norm()))
    rel = float((dk - dt).norm() / dt.norm())
    assert cos > 0.99 and rel < 0.12, (cos, rel)
    assert float((dk - dt).abs().max()) < 0.25 * float(moved) + 2e-5


@pytest.mark.parametrize("n_envs,n_steps,batch", [(4, 4, 1), (1, 129, 128)])
def test_one_sample_minibatches_update_like_the_torch_update(n_envs, n_steps, batch):
    """stable_baselines3 does not normalise the advantage of a one-sample minibatch.  batch_size 1 runs the single-CTA
    optimizer steps (ppo_minibatch_steps_a); 129 samples in minibatches of 128 end with a ragged one-sample step
    (ppo_minibatch_grad_a + ppo_adam_step).  From the same rollout, parameters and fresh Adam state, one epoch of the kernel
    update must land where the torch update does, within the bounds of test_kernel_update_learns_like_the_torch_update."""
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(n_envs, preset="waypoints_v3", seed=9)
    m = PPO("MlpPolicy", env, n_steps=n_steps, batch_size=batch, n_epochs=1, seed=9, ent_coef=0.001, use_cuda_graph=False)
    m.collect_rollouts()
    theta0, epoch0 = m.policy.theta.detach().clone(), m._perm_epoch
    out = {}
    for mode in ("kernel", "torch"):          # both start from zero Adam moments and draw the same permutation
        with torch.no_grad():
            m.policy.theta.copy_(theta0)
        m._perm_epoch = epoch0
        m.update = mode
        m.train()
        torch.cuda.synchronize()
        out[mode] = m.policy.theta.detach() - theta0
    dk, dt = out["kernel"], out["torch"]
    moved = dt.abs().max()
    assert float(moved) > 1e-4
    cos = float(torch.dot(dk, dt) / (dk.norm() * dt.norm()))
    rel = float((dk - dt).norm() / dt.norm())
    assert cos > 0.99 and rel < 0.12, (cos, rel)
    assert float((dk - dt).abs().max()) < 0.25 * float(moved) + 2e-5
    env.close()


class FlatInit:
    @staticmethod
    def theta(d, seed):
        from pyflyt_drone_b200.ppo import FlatMlpPolicy
        return FlatMlpPolicy(d, torch.device("cuda", 0), seed=seed).theta.detach()


def test_evaluate_policy_reports_raw_episode_returns():
    """The reference's eval flow (eval/eval_waypoints.py:96-160): frozen statistics, raw rewards, deterministic policy.
    On the sparse Waypoints task the first thing PPO learns is to stay in the air (the return first DROPS: -0.1 per
    step for many more steps), then to reach waypoints: a briefly trained policy must reach more waypoints than the
    random-initialised one, and evaluation must not touch the training statistics."""
    from pyflyt_drone_b200.ppo import PPO
    from pyflyt_drone_b200.vec_env import FixedwingVecEnv
    env = FixedwingVecEnv(2048, preset="waypoints_v3", seed=21)
    m = PPO("MlpPolicy", env, n_steps=64, batch_size=2048 * 16, n_epochs=10, seed=21)
    r0, s0, l0, t0 = m.evaluate_policy(n_eval_episodes=256)
    assert np.isfinite([r0, s0, l0, t0]).all() and l0 >= 1 and r0 < 0          # an untrained policy crashes: -100 - 0.1/step
    count = float(m.vecnorm.obs_stats[-1])
    m.learn(40 * 64 * 2048)
    before = m.vecnorm.obs_stats.clone()
    r1, s1, l1, t1 = m.evaluate_policy(n_eval_episodes=256)
    assert torch.equal(before, m.vecnorm.obs_stats)                             # env.training = False
    assert float(m.vecnorm.obs_stats[-1]) > count
    print(f"\n[evaluate_policy] untrained: return {r0:.1f} +- {s0:.1f}, length {l0:.0f}, targets {t0:.3f}; after 5.2 M steps: "
          f"return {r1:.1f} +- {s1:.1f}, length {l1:.0f}, targets {t1:.3f}")
    # (flight length is far too variable between runs this early in training to assert on; waypoints reached is not)
    assert t1 > 1.5 * t0, (r0, r1, l0, l1, t0, t1)
    env.close()
