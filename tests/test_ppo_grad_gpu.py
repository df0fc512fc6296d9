"""The fused PPO minibatch gradient (ppo_minibatch_grad_a, csrc/ppo_update_tc.cu) and the forward kernels against a plain
float64 reference of the same operations, on synthetic data built so that every sample's place in the loss is known.

The data keep every probability ratio at least 0.1 in log space away from 1 +- clip_range, so the TF32 forward cannot flip a
clip indicator: the clip count is compared exactly and the gradient to a tolerance.  Batches cover the tile (128 rows) and
grid (one CTA per SM, G = SM count) edges: one sample, a partial tile, a lone row in a last tile, CTAs that walk two or more
tiles and CTAs that walk one tile more than their neighbours; widths cover every build (a = 4 with a 32- and a 64-wide
observation slab, a = 6), the 4-byte observation gather (d % 4 != 0) and a nearly empty second slab (d = 33).

Tolerances were set from the errors measured on an NVIDIA B200 (1,000 W power limit), at most 3x the worst value across the
matrix.  Worst measured, with the bound used:
  gradient, relative L2 error per tensor          2.0e-2  (d = 1, vf.0.weight, leverage, 131,072)   5e-2
  gradient, max-abs error / max-abs per tensor    2.3e-2  (d = 1, vf.0.bias, leverage, 3 G 128 + 37)  6e-2
  statistics 0, 1, 2, 4 (scale: see reference)   1.2e-3  (a = 6, d = 32, one sample)                3e-3
  forward, tcgen05 action mean and value          3.0e-3  absolute                                   9e-3
  forward, CUDA-core action mean and value        1.4e-6  absolute                                   4e-6
Away from d = 1 the gradient errors are 4e-3 to 1.5e-2; every leverage row moves the fp64 gradient by >= 10x the bound.
"""
import math

import pytest
import torch

CLIP, ENT, VF = 0.2, 0.001, 0.5
HALF_LN_2PI = 0.5 * math.log(2.0 * math.pi)
TOL_REL = 5e-2          # per-tensor relative L2 error of the gradient
TOL_MAX = 6e-2          # per-tensor max-abs error over the tensor's max-abs value
TOL_STAT = 3e-3         # loss statistics: |kernel - fp64| over the statistic's scale (see reference)
TOL_TC = 9e-3           # tcgen05 forward (TF32): action mean and value, absolute
TOL_CC = 4e-6           # CUDA-core forward (fp32): action mean and value, absolute
# log-ratio bands: inside the clip band, below 1 - clip, above 1 + clip; each >= 0.1 from log(1 -+ clip)
BAND_IN, BAND_LO, BAND_HI = (-0.12, 0.08), (-0.7, -0.33), (0.29, 0.7)


# ----------------------------------------------------------------------------------------------------- fp64 reference
def _towers64(pol, theta, obs):
    v = lambda n: pol.view(n, theta)  # noqa: E731
    h = torch.tanh(torch.addmm(v("pi.0.bias"), obs, v("pi.0.weight").t()))
    h = torch.tanh(torch.addmm(v("pi.2.bias"), h, v("pi.2.weight").t()))
    mean = torch.addmm(v("action_net.bias"), h, v("action_net.weight").t())
    g = torch.tanh(torch.addmm(v("vf.0.bias"), obs, v("vf.0.weight").t()))
    g = torch.tanh(torch.addmm(v("vf.2.bias"), g, v("vf.2.weight").t()))
    value = torch.addmm(v("value_net.bias"), g, v("value_net.weight").t()).squeeze(-1)
    return mean, value


def _loss64(pol, theta, obs, act, logp_old, adv, ret, clip=CLIP, ent_coef=ENT, vf_coef=VF):
    """stable_baselines3 PPO.train's minibatch loss in float64; the advantage is normalised (unbiased std) unless the
    minibatch has one sample.  Returns the loss and the per-sample terms behind the kernel's statistics."""
    mean, value = _towers64(pol, theta, obs)
    log_std = pol.view("log_std", theta)
    a = (adv - adv.mean()) / (adv.std() + 1e-8) if adv.numel() > 1 else adv
    z = (act - mean) * torch.exp(-log_std)
    lr = (-0.5 * z * z - log_std - HALF_LN_2PI).sum(-1) - logp_old
    ratio = torch.exp(lr)
    surr = torch.min(a * ratio, a * torch.clamp(ratio, 1.0 - clip, 1.0 + clip))
    verr = (ret - value) ** 2
    entropy = (0.5 + HALF_LN_2PI + log_std).sum()
    loss = -surr.mean() + vf_coef * verr.mean() - ent_coef * entropy
    return loss, surr, verr, ratio, lr, a


def reference(pol, theta, obs, act, logp_old, adv, ret, clip=CLIP, ent_coef=ENT, vf_coef=VF):
    """Gradient of the loss on the flat parameter vector (autograd, float64) and the kernel's six statistics
    (include/fwppo.h: sums of policy loss, squared value error, approx KL, clipped, ratio; samples), each with a scale: the
    sum over samples of the term's sensitivity to the log-probability (or value) the forward pass computes, plus the term."""
    th = theta.detach().double().clone().requires_grad_(True)
    loss, surr, verr, ratio, lr, a = _loss64(pol, th, obs.double(), act.double(), logp_old.double(), adv.double(), ret.double(),
                                          clip, ent_coef, vf_coef)
    (grad,) = torch.autograd.grad(loss, th)
    with torch.no_grad():
        kl, clipped = (ratio - 1.0) - lr, ((ratio - 1.0).abs() > clip).double()
        n = torch.tensor(float(adv.numel()), dtype=torch.float64, device=th.device)
        stats = torch.stack([(-surr).sum(), verr.sum(), kl.sum(), clipped.sum(), ratio.sum(), n])
        scale = torch.stack([(a.abs() * ratio).sum(), (verr + 2 * verr.sqrt()).sum(), (ratio - 1.0).abs().sum(), n,
                             ratio.sum(), n])
    return grad.detach(), stats, scale


# ----------------------------------------------------------------------------------------------------- synthetic data
def make_policy(d, a, seed, device):
    from pyflyt_drone_b200.ppo import FlatMlpPolicy
    pol = FlatMlpPolicy(d, device, seed=seed, act_dim=a)
    g = torch.Generator(device="cpu").manual_seed(1000 + seed)
    with torch.no_grad():
        pol.theta.add_((0.05 * torch.randn(pol.count, generator=g)).to(device))
        pol.view("log_std").copy_(torch.linspace(-0.5, 0.3, a))        # a distinct sigma per channel
    return pol


def make_data(pol, batch, kind="plain", seed=0, lev_rows=()):
    """Rollout-buffer tensors (fp32) and a minibatch idx into them.
    kind: plain       N(0.3, 1.5) advantages, ratios spread over the three bands (row 0 inside), returns V + 1 + N(0, 1): the
                      value gradient has a systematic part (with a zero-mean residual it would be O(1 / sqrt(batch)) and the
                      TF32 forward's value rounding, which does not average out, would be measured instead of the kernel)
          leverage    plain, plus the minibatch rows lev_rows carrying advantage / return outliers, ratios inside the band
          zero_adv    plain with every advantage 0
          zero_quad   advantages exactly +-1 in balanced counts (one 0 for an odd batch > 1), every sample where the clipped
                      branch wins: (A > 0, r > 1 + clip) or (A < 0, r < 1 - clip)
          flowing     the same advantages in the other two quadrants: (A > 0, r < 1 - clip) or (A < 0, r > 1 + clip)"""
    dev, d, a = pol.theta.device, pol.d, pol.a
    theta = pol.theta.detach().double()
    nbuf = batch + batch // 4 + 61
    g = torch.Generator(device=dev).manual_seed(seed)
    f64 = dict(dtype=torch.float64, device=dev)
    u = lambda shape, lo, hi: lo + (hi - lo) * torch.rand(shape, generator=g, **f64)  # noqa: E731
    obs = (2.0 * torch.randn(nbuf, d, generator=g, **f64)).clamp(-10.0, 10.0)
    edge = torch.arange(0, nbuf, 53, device=dev)                          # rows at exactly +-10
    obs[edge] = torch.where(torch.rand(len(edge), d, generator=g, **f64) < 0.5, -10.0, 10.0).double()
    obs = obs.float()
    idx = torch.randperm(nbuf, generator=g, device=dev)[:batch]
    with torch.no_grad():
        mean, value = _towers64(pol, theta, obs.double())
    log_std = pol.view("log_std", theta)
    eps = torch.randn(nbuf, a, generator=g, **f64)
    far = torch.arange(0, nbuf, 41, device=dev)                           # a few |eps| > 3
    eps[far, far % a] = torch.where(far % 2 == 0, 3.5, -3.3).double()
    act = (mean + torch.exp(log_std) * eps).float()
    logp = (-0.5 * ((act.double() - mean) * torch.exp(-log_std)) ** 2 - log_std - HALF_LN_2PI).sum(-1)
    adv = 1.5 * torch.randn(nbuf, generator=g, **f64) + 0.3
    ret = value + 1.0 + torch.randn(nbuf, generator=g, **f64)
    band = torch.randint(0, 4, (nbuf,), generator=g, device=dev)         # 0, 1: inside; 2: below; 3: above
    lr = torch.where(band < 2, u(nbuf, *BAND_IN), torch.where(band == 2, u(nbuf, *BAND_LO), u(nbuf, *BAND_HI)))
    lr[idx[0]] = u(1, *BAND_IN)
    if kind == "leverage":
        rows = idx[torch.tensor(list(lev_rows), device=dev, dtype=torch.long)]
        sign = torch.tensor([(-1.0) ** k for k in range(len(lev_rows))], **f64)
        adv[rows] = sign * 6.0 * math.sqrt(batch) * torch.linspace(1.0, 1.5, len(lev_rows), **f64)
        ret[rows] = value[rows] - sign * (6.0 * math.sqrt(batch) + batch) * torch.linspace(1.5, 1.0, len(lev_rows), **f64)
        lr[rows] = u(len(lev_rows), *BAND_IN)
    elif kind == "zero_adv":
        adv.zero_()
    elif kind in ("zero_quad", "flowing"):
        s = torch.where(torch.arange(batch, device=dev) % 2 == 0, 1.0, -1.0).double()
        if batch % 2 and batch > 1:
            s[-1] = 0.0
        adv[idx] = s
        up = (s > 0) if kind == "zero_quad" else (s < 0)                 # ratio above the band
        lr[idx] = torch.where(up, u(batch, *BAND_HI), u(batch, *BAND_LO))
    return dict(obs=obs, act=act, logp=(logp - lr).float(), adv=adv.float(), ret=ret.float(), idx=idx)


def _take(data):
    i = data["idx"]
    return data["obs"][i], data["act"][i], data["logp"][i], data["adv"][i], data["ret"][i]


def leverage_rows(batch, G):
    """Minibatch rows at the kernel's tile and grid edges: the first row, both sides of the first tile boundary, the last row
    (the lone row of a last partial tile when batch % 128 == 1) and, once there are more tiles than CTAs, the first row of
    CTA 0's second tile and a row of a CTA that walks one tile more than its neighbour."""
    rows = {0, batch - 1} | {r for r in (127, 128) if r < batch}
    ntiles = -(-batch // 128)
    if ntiles > G:
        rows.add(G * 128)
        q, r = divmod(ntiles, G)
        if r:
            rows.add(min((q * G + r - 1) * 128 + 77, batch - 1))
    return sorted(rows)


def _tensor_errors(pol, got, ref):
    """{tensor: (relative L2 error, max-abs error / max-abs value)}; a zero reference must be met exactly."""
    out = {}
    for name, (lo, hi, _) in pol.slices.items():
        r, e = ref[lo:hi], got[lo:hi].double() - ref[lo:hi]
        rn, rm = float(r.norm()), float(r.abs().max())
        out[name] = (float(e.norm()) / rn if rn > 0 else (0.0 if float(e.norm()) == 0 else math.inf),
                     float(e.abs().max()) / rm if rm > 0 else (0.0 if float(e.abs().max()) == 0 else math.inf))
    return out


# ----------------------------------------------------------------------------------------------------- CPU: the reference
@pytest.mark.parametrize("a", [4, 6])
@pytest.mark.parametrize("batch", [7, 1])
def test_reference_gradient_matches_central_differences(a, batch):
    """The float64 reference's autograd gradient against central finite differences of its own loss (d = 5), at every
    coordinate of the small tensors and a sample of the large ones; for one sample the advantage is not normalised."""
    pol = make_policy(5, a, seed=3, device=torch.device("cpu"))
    data = make_data(pol, batch, seed=4)
    obs, act, lpo, adv, ret = (t.double() for t in _take(data))
    theta = pol.theta.detach().double()
    grad, stats, _ = reference(pol, theta, obs, act, lpo, adv, ret)
    g = torch.Generator().manual_seed(5)
    coords = []
    for name, (lo, hi, _) in pol.slices.items():
        n = hi - lo
        coords += list(range(lo, hi)) if n <= 64 else (lo + torch.randperm(n, generator=g)[:24]).tolist()
    h = 1e-6
    for k in coords:
        tp, tm = theta.clone(), theta.clone()
        tp[k] += h
        tm[k] -= h
        fd = (float(_loss64(pol, tp, obs, act, lpo, adv, ret)[0]) - float(_loss64(pol, tm, obs, act, lpo, adv, ret)[0])) / (2 * h)
        assert abs(fd - float(grad[k])) <= 1e-6 * max(1.0, abs(fd)), (k, fd, float(grad[k]))
    # ratios are where the data put them: no sample within 0.1 (log) of a clip boundary
    ratio = _loss64(pol, theta, obs, act, lpo, adv, ret)[3]
    dist = torch.minimum((ratio.log() - math.log(1 - CLIP)).abs(), (ratio.log() - math.log(1 + CLIP)).abs())
    assert float(dist.min()) >= 0.1 - 1e-6
    if batch == 1:   # stable_baselines3 leaves a one-sample minibatch's advantage as it is
        r = float(ratio[0])
        assert float(stats[0]) == pytest.approx(-min(float(adv[0]) * r, float(adv[0]) * min(max(r, 1 - CLIP), 1 + CLIP)), rel=1e-12)
        assert float(pol.view("action_net.bias", grad).abs().max()) > 1e-3


def test_leverage_rows_sit_at_the_tile_and_grid_edges():
    G = 148
    assert leverage_rows(1, G) == [0] and leverage_rows(2, G) == [0, 1]
    assert leverage_rows(129, G) == [0, 127, 128]
    assert leverage_rows(G * 128 + 1, G) == [0, 127, 128, G * 128]
    # 1,024 tiles on 148 CTAs: CTAs 0-135 walk seven tiles, 136-147 six; tile 1023 is CTA 135's seventh
    assert leverage_rows(131072, G) == [0, 127, 128, G * 128, 1023 * 128 + 77, 131071]


# ----------------------------------------------------------------------------------------------------- GPU: the kernel
def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _batch(spec):
    G = _sm_count()
    return {"G*128": G * 128, "G*128+1": G * 128 + 1, "3G*128+37": 3 * G * 128 + 37}.get(spec) or int(spec)


def run_kernel(pol, data, batch, clip=CLIP, ent_coef=ENT, vf_coef=VF):
    from pyflyt_drone_b200 import _lib
    from pyflyt_drone_b200.ppo import _p, _stream
    lib = _lib.load()
    dev = pol.theta.device
    ws = torch.zeros(int(lib.ppo_update_workspace_floats_a(pol.d, pol.a)), dtype=torch.float32, device=dev)
    grad = torch.full((pol.count,), float("nan"), dtype=torch.float32, device=dev)
    stats = torch.full((8,), float("nan"), dtype=torch.float32, device=dev)
    idx = data["idx"][:batch].contiguous()
    _lib.check(lib.ppo_minibatch_grad_a(_p(pol.theta.data), pol.d, pol.a, _p(data["obs"]), _p(data["act"]), _p(data["logp"]),
                                        _p(data["adv"]), _p(data["ret"]), _p(idx), batch, clip, ent_coef, vf_coef, _p(ws),
                                        _p(grad), _p(stats), _stream()))
    torch.cuda.synchronize()
    return grad, stats


def _check_case(pol, data, batch, label, lev=()):
    grad, stats = run_kernel(pol, data, batch)
    theta = pol.theta.detach()
    ref, rstats, rscale = reference(pol, theta, *_take(data))
    errs = _tensor_errors(pol, grad, ref)
    worst_rel = max(errs.items(), key=lambda kv: kv[1][0])
    worst_max = max(errs.items(), key=lambda kv: kv[1][1])
    st = stats.double()
    stat_err = [float((st[k] - rstats[k]).abs() / rscale[k].clamp_min(1e-30)) for k in (0, 1, 2, 4)]
    print(f"\n[grad-err] {label}: rel {worst_rel[1][0]:.3e} ({worst_rel[0]}) max {worst_max[1][1]:.3e} ({worst_max[0]}) "
          f"stats {max(stat_err):.3e}")
    for name, (rel, mx) in errs.items():
        assert rel <= TOL_REL and mx <= TOL_MAX, (label, name, rel, mx)
    assert float(st[3]) == float(rstats[3]), (label, float(st[3]), float(rstats[3]))       # clipped samples: exact
    assert float(st[5]) == batch and float(st[6]) == 0.0 and float(st[7]) == 0.0
    assert max(stat_err) <= TOL_STAT, (label, stat_err)
    # on the leverage dataset each outlier row matters: dropping or duplicating it moves the fp64 gradient by >= 10x the
    # tolerance in some tensor, so a kernel that lost or double-counted that row could not pass the bound above
    obs, act, lpo, adv, ret = _take(data)
    for p in lev:
        keep = torch.cat([torch.arange(p, device=obs.device), torch.arange(p + 1, batch, device=obs.device)])
        twice = torch.cat([torch.arange(batch, device=obs.device), torch.tensor([p], device=obs.device)])
        for sel in ((keep,) if batch > 1 else ()) + (twice,):
            moved, _, _ = reference(pol, theta, obs[sel], act[sel], lpo[sel], adv[sel], ret[sel])
            shift = max(e[0] for e in _tensor_errors(pol, moved.float(), ref).values())
            assert shift >= 10 * TOL_REL, (label, p, shift)


_WIDTHS = [(4, 1), (4, 28), (4, 29), (4, 32), (4, 33), (4, 56), (4, 64), (6, 21), (6, 32)]
_BATCHES = ["1", "2", "127", "128", "129", "G*128", "G*128+1", "3G*128+37", "131072"]
_CASES = [(a, d, b) for a, d in _WIDTHS for b in _BATCHES] + [(4, 32, "1048576"), (4, 64, "1048576"), (6, 32, "1048576")]


@pytest.mark.gpu
@pytest.mark.parametrize("a,d,spec", _CASES)
def test_minibatch_gradient_matches_fp64(a, d, spec):
    """ppo_minibatch_grad_a (tcgen05: TF32 forward, bf16 backward operands, fp32 accumulation) against the float64 reference,
    per parameter tensor, with the clip count exact and the other statistics to a tolerance; on bulk data and on data whose
    outliers sit at the tile and grid edges."""
    batch = _batch(spec)
    pol = make_policy(d, a, seed=d + 7 * a, device=torch.device("cuda", 0))
    _check_case(pol, make_data(pol, batch, "plain", seed=batch + d), batch, f"a={a} d={d} batch={batch} plain")
    lev = leverage_rows(batch, _sm_count())
    _check_case(pol, make_data(pol, batch, "leverage", seed=batch + d + 1, lev_rows=lev), batch,
                f"a={a} d={d} batch={batch} leverage", lev)


_EXACT = [(a, d, b) for a, d in [(4, 28), (4, 56), (6, 21)] for b in ["1", "2", "129", "G*128+1", "3G*128+37"]]


@pytest.mark.gpu
@pytest.mark.parametrize("a,d,spec", _EXACT)
def test_gradient_without_policy_signal_is_exactly_the_entropy_term(a, d, spec):
    """With every advantage 0, or every sample in a quadrant where the clipped branch of the surrogate wins, no policy
    gradient flows: every pi / action_net entry is exactly 0 and log_std is exactly -ent_coef.  The value tower still
    matches fp64; samples in the two flowing quadrants match fp64 throughout."""
    batch = _batch(spec)
    pol = make_policy(d, a, seed=11, device=torch.device("cuda", 0))
    for kind in ("zero_adv", "zero_quad"):
        data = make_data(pol, batch, kind, seed=batch + 3)
        grad, stats = run_kernel(pol, data, batch)
        for name, (lo, hi, _) in pol.slices.items():
            if name.startswith(("pi.", "action_net.")):
                assert bool((grad[lo:hi] == 0).all()), (kind, name)
        assert torch.equal(pol.view("log_std", grad), torch.full((a,), -ENT, device=grad.device)), kind
        ref, rstats, _ = reference(pol, pol.theta.detach(), *_take(data))
        for name, (rel, mx) in _tensor_errors(pol, grad, ref).items():
            assert rel <= TOL_REL and mx <= TOL_MAX, (kind, name, rel, mx)
        assert float(stats[3]) == float(rstats[3]) and float(stats[5]) == batch
    _check_case(pol, make_data(pol, batch, "flowing", seed=batch + 4), batch, f"a={a} d={d} batch={batch} flowing")


# ----------------------------------------------------------------------------------------------------- GPU: forward family
def _obs_and_stats(d, n, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    obs = 8.0 * torch.randn(n, d, generator=g, device=dev)
    obs[::17] *= 40.0                                                     # rows that the clip at +-10 reaches
    stats = torch.zeros(2 * d + 1, dtype=torch.float64, device=dev)
    stats[:d] = torch.linspace(-3, 3, d, dtype=torch.float64)
    stats[d:2 * d] = torch.linspace(0.5, 90, d, dtype=torch.float64)
    stats[2 * d] = 1000.0
    return obs.contiguous(), stats


def _norm64(obs, stats, d):
    return torch.clamp((obs.double() - stats[:d]) / torch.sqrt(stats[d:2 * d] + 1e-8), -10, 10)


def _forward(fn, pol, obs, stats, n):
    from pyflyt_drone_b200 import _lib
    from pyflyt_drone_b200.ppo import _p, _stream
    dev = obs.device
    o = dict(obs_norm=torch.zeros(n, pol.d, device=dev), act_env=torch.zeros(n, pol.a, device=dev),
             act_raw=torch.zeros(n, pol.a, device=dev), logp=torch.zeros(n, device=dev), value=torch.zeros(n, device=dev))
    _lib.check(fn(_p(pol.theta.data), pol.d, pol.a, _p(obs), _p(stats), 10.0, n, 77, 0, 5, None, 1, _p(o["obs_norm"]),
                  _p(o["act_env"]), _p(o["act_raw"]), _p(o["logp"]), _p(o["value"]), _stream()))
    torch.cuda.synchronize()
    return o


@pytest.mark.gpu
@pytest.mark.parametrize("d,a", [(28, 4), (29, 4), (21, 6), (56, 4)])
@pytest.mark.parametrize("spec", ["1", "129", "G*128+1"])
def test_forward_kernels_match_fp64_towers(d, a, spec):
    """Deterministic ppo_policy_forward_tc_a (TF32) and ppo_policy_forward_a (fp32): the action (= mean) and the value against
    the float64 towers on the same normalised observations; both kernels normalise bit-identically, to fp32 rounding of fp64."""
    from pyflyt_drone_b200 import _lib
    n, dev = _batch(spec), torch.device("cuda", 0)
    lib = _lib.load()
    pol = make_policy(d, a, seed=21, device=dev)
    obs, stats = _obs_and_stats(d, n, seed=n + d, dev=dev)
    tc = _forward(lib.ppo_policy_forward_tc_a, pol, obs, stats, n)
    cc = _forward(lib.ppo_policy_forward_a, pol, obs, stats, n)
    assert torch.equal(tc["obs_norm"], cc["obs_norm"])
    assert torch.allclose(cc["obs_norm"].double(), _norm64(obs, stats, d), atol=2e-6, rtol=1e-6)
    with torch.no_grad():
        mean, value = _towers64(pol, pol.theta.detach().double(), cc["obs_norm"].double())
    errs = {}
    for name, o, tol in (("tc", tc, TOL_TC), ("cc", cc, TOL_CC)):
        errs[name] = (float((o["act_raw"].double() - mean).abs().max()), float((o["value"].double() - value).abs().max()))
        assert torch.equal(o["act_env"], o["act_raw"].clamp(-1, 1))
    print(f"\n[fwd-err] d={d} a={a} n={n}: tc mean {errs['tc'][0]:.3e} value {errs['tc'][1]:.3e} "
          f"cc mean {errs['cc'][0]:.3e} value {errs['cc'][1]:.3e}")
    assert max(errs["tc"]) <= TOL_TC and max(errs["cc"]) <= TOL_CC, errs


@pytest.mark.gpu
@pytest.mark.parametrize("d,a", [(21, 6), (56, 4)])
@pytest.mark.parametrize("spec", ["1", "129", "G*128+1"])
def test_value_and_timeout_bootstrap_match_fp64(d, a, spec):
    """ppo_value_forward_a (a rollout's last values) and ppo_timeout_bootstrap_a (rew += gamma * V(terminal obs) for rows that
    were truncated and not terminated) against the float64 value tower; every other row's reward is left bit-identical."""
    from pyflyt_drone_b200 import _lib
    from pyflyt_drone_b200.ppo import _p, _stream
    n, dev = _batch(spec), torch.device("cuda", 0)
    lib = _lib.load()
    pol = make_policy(d, a, seed=23, device=dev)
    obs, stats = _obs_and_stats(d, n, seed=n + d + 1, dev=dev)
    with torch.no_grad():
        _, value = _towers64(pol, pol.theta.detach().double(), _norm64(obs, stats, d))
    v = torch.zeros(n, device=dev)
    _lib.check(lib.ppo_value_forward_a(_p(pol.theta.data), d, a, _p(obs), _p(stats), 10.0, n, _p(v), _stream()))
    g = torch.Generator(device=dev).manual_seed(n)
    flags = torch.randint(0, 4, (n,), generator=g, device=dev, dtype=torch.uint8)
    flags[0] = 2
    rew0 = torch.randn(n, generator=g, device=dev)
    rew = rew0.clone()
    _lib.check(lib.ppo_timeout_bootstrap_a(_p(pol.theta.data), d, a, _p(obs), _p(stats), 10.0, _p(flags), n, 0.99, _p(rew),
                                           _stream()))
    torch.cuda.synchronize()
    verr = float((v.double() - value).abs().max())
    boot = flags == 2
    berr = float((rew[boot].double() - (rew0[boot].double() + 0.99 * value[boot])).abs().max())
    print(f"\n[val-err] d={d} a={a} n={n}: value {verr:.3e} bootstrap {berr:.3e}")
    assert verr <= TOL_CC and berr <= TOL_CC
    assert torch.equal(rew[~boot], rew0[~boot])
