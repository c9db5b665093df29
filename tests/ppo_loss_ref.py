"""Float64 NumPy references of the learner-side kernels: the fused PPO-Lagrangian loss (`csrc/ppo_loss.cu`,
`mapf_adv_moments` + `mapf_ppo_loss`) and the masked GAE scan (`csrc/gae.cu`).

The loss is an independent statement of model.py:104-164: the ten per-element statistics in the order of the kernel's
partials (include/mapf_b200.h, `mapf_ppo_loss`) and the gradients with respect to the four network outputs, written out
analytically.  It does not call ppo/loss.py; tests/test_ppo_loss_reference.py checks it against float64 autograd
through that module.

Conventions, chosen so that a correct f32 kernel agrees with it:
- every boundary constant is the kernel's f32 value, widened: f32(1e-6), f32(1) - f32(1e-6), f32(1) -/+ f32(clip), and
  +/- f32(clip);
- every decision on an input value is taken on that value: the clamp masks on p, sig, f32(1 - sig) and the value delta
  (exact in f32 when the old value is 0), and the tie tests.  Decisions on computed values (the ratio clamp, the clip
  count, the value-loss branch) can differ from the kernel's within a few ulp of a boundary; tests keep random inputs
  out of that band with `near_boundary`;
- gradients follow PyTorch: clamp passes the gradient on the closed interval; minimum / maximum split it 50/50 on ties;
- every output comes with a magnitude, the sum of the absolute values of the terms that make it up (with the
  conditioning of the ratio's logarithms and of the f32 subtractions it rests on), so a tolerance can be stated per
  element in units of f32 rounding.
"""
import numpy as np

NA = 5
F32 = np.float32
P_LO = float(F32(1e-6))                       # clamp(p, 1e-6f, 1.0f)
SIG_LO = float(F32(1e-6))                     # clamp(sig, 1e-6f, 1.0f - 1e-6f)
SIG_HI = float(F32(1.0) - F32(1e-6))


def kernel_clip_bounds(clip):
    """(1.0f - clip, 1.0f + clip, clip) as the kernel forms them in f32, widened to double."""
    c = F32(clip)
    return float(F32(1.0) - c), float(F32(1.0) + c), float(c)


def adv_moments(returns, cost_returns, old_v, old_cv):
    """[sum a, sum a^2, sum c, sum c^2] in double with a = f32(returns - old_v), c = f32(cost_returns - old_cv)."""
    a = (np.asarray(returns, F32) - np.asarray(old_v, F32)).astype(np.float64).ravel()
    c = (np.asarray(cost_returns, F32) - np.asarray(old_cv, F32)).astype(np.float64).ravel()
    return np.array([a.sum(), (a * a).sum(), c.sum(), (c * c).sum()])


def two_pass_std(x):
    """Unbiased std of the double values x by the two-pass formula (NaN for fewer than two values, like torch.std)."""
    x = np.asarray(x, np.float64).ravel()
    if x.size < 2:
        return float("nan")
    return float(np.sqrt(((x - x.mean()) ** 2).sum() / (x.size - 1)))


def loss_config(ppo_cfg, lagrangian, returns, cost_returns, old_v, old_cv):
    """The MapfPpoLossConfig fields for one global minibatch, with two-pass double statistics of the f32 differences."""
    a = (np.asarray(returns, F32) - np.asarray(old_v, F32)).astype(np.float64)
    c = (np.asarray(cost_returns, F32) - np.asarray(old_cv, F32)).astype(np.float64)
    return dict(clip_range=ppo_cfg.clip_range, entropy_coef=ppo_cfg.entropy_coef, value_coef=ppo_cfg.value_coef,
                valid_coef=ppo_cfg.valid_coef, cost_value_coef=ppo_cfg.cost_value_coef, cost_coef=ppo_cfg.cost_coef,
                lagrangian=float(lagrangian), minus_adv_with_cadv=bool(ppo_cfg.minus_adv_with_cadv), n_global=float(a.size),
                adv_mean=float(a.mean()), adv_std=two_pass_std(a), cadv_mean=float(c.mean()), cadv_std=two_pass_std(c))


def _coefs(cfg):
    """The config's f32 fields widened to double, as the kernel sees them."""
    return {k: float(F32(cfg[k])) for k in ("clip_range", "entropy_coef", "value_coef", "valid_coef", "cost_value_coef",
                                             "cost_coef", "lagrangian")}


def _advantages(cfg, returns, cost_returns, old_v, old_cv):
    """(adv, mag_adv, cadv, mag_cadv) per element, model.py:106-113."""
    lam = _coefs(cfg)["lagrangian"]
    a = (np.asarray(returns, F32) - np.asarray(old_v, F32)).astype(np.float64)
    c = (np.asarray(cost_returns, F32) - np.asarray(old_cv, F32)).astype(np.float64)
    aden, cden = cfg["adv_std"] + 1e-6, cfg["cadv_std"] + 1e-6
    adv, cadv = (a - cfg["adv_mean"]) / aden, (c - cfg["cadv_mean"]) / cden
    madv, mcadv = (np.abs(a) + abs(cfg["adv_mean"])) / aden, (np.abs(c) + abs(cfg["cadv_mean"])) / cden
    if cfg["minus_adv_with_cadv"]:
        adv, madv = (adv - lam * cadv) / (lam + 1.0), (madv + abs(lam) * mcadv) / abs(lam + 1.0)
    return adv, madv, cadv, mcadv


def _closed(x, lo, hi):
    return ((x >= lo) & (x <= hi)).astype(np.float64)


def ppo_loss_ref(cfg, policy, value, cost_value, sig, returns, cost_returns, old_v, old_cv, actions, old_ps, train_valid):
    """cfg: dict with the MapfPpoLossConfig fields.  Inputs are f32 arrays of n elements ([n] or [n, 5]) and int actions.

    Returns a dict of float64 arrays: g_policy [n,5], g_value [n], g_cost_value [n], g_sig [n,5] (the gradients of the
    loss, every mean taken as sum / n_global), each with a `<name>_mag`; `stats` [n,10], the per-element terms of the
    kernel's partial sums (column 9 is unused and 0), with `stats_mag`; and `clipped`, the boolean clip decisions."""
    k = _coefs(cfg)
    lo, hi, c = kernel_clip_bounds(cfg["clip_range"])
    lam = k["lagrangian"]
    s = 1.0 / cfg["n_global"]
    p = np.asarray(policy, F32).reshape(-1, NA).astype(np.float64)
    op = np.asarray(old_ps, F32).reshape(-1, NA).astype(np.float64)
    sg32 = np.asarray(sig, F32).reshape(-1, NA)
    sg = sg32.astype(np.float64)
    q = (F32(1.0) - sg32).astype(np.float64)              # the kernel's f32(1 - sig); exact when sig >= 0.5
    t = np.asarray(train_valid, F32).reshape(-1, NA).astype(np.float64)
    v, cv = (np.asarray(x, F32).ravel().astype(np.float64) for x in (value, cost_value))
    R, CR, ov, ocv = (np.asarray(x, F32).ravel().astype(np.float64) for x in (returns, cost_returns, old_v, old_cv))
    act = np.asarray(actions).ravel().astype(np.int64)
    assert ((act >= 0) & (act < NA)).all()
    n = act.size
    rows = np.arange(n)
    adv, madv, cadv, mcadv = _advantages(cfg, returns, cost_returns, old_v, old_cv)

    # ratio (model.py:119) and its conditioning: exp(log cn - log co) carries the error of both logarithms
    new_p, old_p = p[rows, act], op[rows, act]
    cn, co = np.clip(new_p, P_LO, 1.0), np.clip(old_p, P_LO, 1.0)
    ratio = cn / co
    mratio = ratio * (2.0 + np.abs(np.log(cn)) + np.abs(np.log(co)))
    pass_n = _closed(new_p, P_LO, 1.0)
    dratio, mdratio = ratio / cn * pass_n, mratio / cn * pass_n

    # clipped surrogate (model.py:139-143): min(adv*ratio, adv*clamp(ratio)); ties split 50/50
    rc = np.clip(ratio, lo, hi)
    t1, t2 = adv * ratio, adv * rc
    inside = _closed(ratio, lo, hi)
    dsur = np.where(t1 < t2, adv, np.where(t1 > t2, adv * inside, 0.5 * adv + 0.5 * adv * inside))
    sur = np.minimum(t1, t2)

    # entropy (model.py:121) and the gradient of -entropy_coef * entropy
    ck = np.clip(p, P_LO, 1.0)
    lk = np.log(ck)
    ent = -(p * lk).sum(1)
    ment = (p * (np.abs(lk) + 1.0)).sum(1)
    pk = p / ck * _closed(p, P_LO, 1.0)
    g_pol = k["entropy_coef"] * s * (lk + pk)
    m_pol = abs(k["entropy_coef"]) * s * (np.abs(lk) + 1.0 + pk)
    gpa = (-dsur + k["cost_coef"] * lam * cadv) * s * dratio
    mgpa = (madv + abs(k["cost_coef"] * lam) * mcadv) * s * mdratio
    g_pol[rows, act] += gpa
    m_pol[rows, act] += mgpa

    # clipped value losses (model.py:124-136): max(e1, e2); ties split 50/50
    def clipped(nv, old, target):
        d = nv - old
        vcl = old + np.clip(d, -c, c)
        e1, e2 = (nv - target) ** 2, (vcl - target) ** 2
        g1, g2 = 2.0 * (nv - target), 2.0 * (vcl - target) * _closed(d, -c, c)
        M = np.abs(nv) + np.abs(old) + np.abs(target) + c
        return np.maximum(e1, e2), M * M, np.where(e1 > e2, g1, np.where(e1 < e2, g2, 0.5 * g1 + 0.5 * g2)), 2.0 * M
    lv, mlv, gv, mgv = clipped(v, ov, R)
    lcv, mlcv, gcv, mgcv = clipped(cv, ocv, CR)

    # valid-action log-likelihood (model.py:146-148) over the five sigmoid outputs
    c1, c2 = np.clip(sg, SIG_LO, SIG_HI), np.clip(q, SIG_LO, SIG_HI)
    l1, l2 = np.log(c1), np.log(c2)
    vl = (l1 * t + l2 * (1.0 - t)).sum(1)
    mvl = ((np.abs(l1) + 1.0) * np.abs(t) + (np.abs(l2) + 1.0) * np.abs(1.0 - t)).sum(1)
    d1 = t / c1 * _closed(sg, SIG_LO, SIG_HI)
    d2 = -(1.0 - t) / c2 * _closed(q, SIG_LO, SIG_HI)
    g_sig = -k["valid_coef"] * (s / NA) * (d1 + d2)
    m_sig = abs(k["valid_coef"]) * (s / NA) * 2.0 * (np.abs(d1) + np.abs(d2))

    clipped_mask = np.abs(ratio - 1.0) > c
    stats = np.zeros((n, 10))
    mags = np.zeros((n, 10))
    for j, (x, m) in enumerate(((sur, madv * mratio), (ent, ment), (lv, mlv), (lcv, mlcv), (vl, mvl),
                                (ratio * cadv, mratio * mcadv), (clipped_mask.astype(np.float64), 0.0 * ratio),
                                (adv, madv), (cadv, mcadv))):
        stats[:, j], mags[:, j] = x, m
    return dict(g_policy=g_pol, g_policy_mag=m_pol,
                g_value=k["value_coef"] * s * gv, g_value_mag=abs(k["value_coef"]) * s * mgv,
                g_cost_value=k["cost_value_coef"] * s * gcv, g_cost_value_mag=abs(k["cost_value_coef"]) * s * mgcv,
                g_sig=g_sig, g_sig_mag=m_sig, stats=stats, stats_mag=mags, clipped=clipped_mask)


STAT_NAMES = ("all_loss", "policy_loss", "policy_entropy", "critic_loss", "valid_loss", "cost_critic_loss", "cost_loss",
              "clipfrac", "advantage", "cost_advantage")


def stat_means(cfg, sums):
    """The loss and the named statistics of ppo/loss.py from the ten partial sums: every mean is sum / n_global, the
    valid loss is minus the mean over the five actions (model.py:146-164)."""
    k = _coefs(cfg)
    x = np.asarray(sums, np.float64) / cfg["n_global"]
    valid = -x[4] / NA
    loss = (-x[0] - k["entropy_coef"] * x[1] + k["value_coef"] * x[2] + k["valid_coef"] * valid
            + k["cost_value_coef"] * x[3] + k["cost_coef"] * k["lagrangian"] * x[5])
    return dict(zip(STAT_NAMES, (loss, x[0], x[1], x[2], valid, x[3], x[5], x[6], x[7], x[8])))


def stat_mags(cfg, mags):
    """The magnitudes of `stat_means` from the ten sums of per-element magnitudes."""
    k = {key: abs(v) for key, v in _coefs(cfg).items()}
    m = np.asarray(mags, np.float64) / cfg["n_global"]
    loss = (m[0] + k["entropy_coef"] * m[1] + k["value_coef"] * m[2] + k["valid_coef"] * m[4] / NA
            + k["cost_value_coef"] * m[3] + k["cost_coef"] * k["lagrangian"] * m[5])
    return dict(zip(STAT_NAMES, (loss, m[0], m[1], m[2], m[4] / NA, m[3], m[5], m[6], m[7], m[8])))


def near_boundary(cfg, policy, value, cost_value, sig, returns, cost_returns, old_v, old_cv, actions, old_ps, rel=1e-5,
                  inputs=True):
    """Elements within `rel` (relative) of a decision boundary where an f32 kernel and this reference may decide
    differently: the ratio against 1 -/+ clip, |value delta| against clip, e1 against e2 where the two value-loss
    branches have different gradients, and (with `inputs`) p or sig against a clamp bound."""
    lo, hi, c = kernel_clip_bounds(cfg["clip_range"])
    p = np.asarray(policy, F32).reshape(-1, NA).astype(np.float64)
    op = np.asarray(old_ps, F32).reshape(-1, NA).astype(np.float64)
    sg = np.asarray(sig, F32).reshape(-1, NA).astype(np.float64)
    act = np.asarray(actions).ravel().astype(np.int64)
    rows = np.arange(act.size)
    ratio = np.clip(p[rows, act], P_LO, 1.0) / np.clip(op[rows, act], P_LO, 1.0)
    bad = (np.abs(ratio - lo) <= rel * lo) | (np.abs(ratio - hi) <= rel * hi)

    def near(x, b):
        return np.abs(x - b) <= rel * abs(b)
    if inputs:
        bad |= (near(p, P_LO) | near(p, 1.0) | near(sg, SIG_LO) | near(sg, SIG_HI) | near(1.0 - sg, SIG_LO)
                | near(1.0 - sg, SIG_HI)).any(1)
    for nv, old, target in ((value, old_v, returns), (cost_value, old_cv, cost_returns)):
        nv, old, target = (np.asarray(x, F32).ravel().astype(np.float64) for x in (nv, old, target))
        d = nv - old
        if inputs:
            bad |= near(np.abs(d), c)
        vcl = old + np.clip(d, -c, c)
        M = np.abs(nv) + np.abs(old) + np.abs(target) + c
        gap = np.abs((nv - target) ** 2 - (vcl - target) ** 2)      # an exact tie (constructed, exact in f32) is kept
        bad |= (np.abs(d) > c) & (gap > 0) & (gap <= rel * M * M)
    return bad


def gae_masked_ref(r, v, last_v, nonterminal, gamma=0.95, lam=0.95):
    """runner.py:120-149 with a nonterminal mask, restated op by op in NumPy f32 (each *, +, - rounded separately, as the
    GAE kernel does): nonterminal[t] = 0 cuts the bootstrap and the advantage carry at step t.  Returns (returns, adv)."""
    r, v = np.asarray(r, F32), np.asarray(v, F32)
    T = r.shape[0]
    cols = r[0].size
    r, v = r.reshape(T, cols), v.reshape(T, cols)
    nt = np.asarray(nonterminal).reshape(T, cols)
    g, gl = F32(gamma * 1.0), F32(gamma * lam * 1.0)
    ret, adv = np.zeros_like(r), np.zeros_like(r)
    last, nv = np.zeros(cols, dtype=F32), np.asarray(last_v, F32).reshape(cols).copy()
    for t in range(T - 1, -1, -1):
        m = nt[t].astype(bool)
        m1 = np.where(m, g * nv, F32(0)).astype(F32)
        delta = ((r[t] + m1).astype(F32) - v[t]).astype(F32)
        m2 = np.where(m, gl * last, F32(0)).astype(F32)
        last = (delta + m2).astype(F32)
        adv[t] = last
        ret[t] = (last + v[t]).astype(F32)
        nv = v[t]
    return ret, adv
