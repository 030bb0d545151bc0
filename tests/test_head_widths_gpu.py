"""The PPO head kernels at every action width they accept, against plain references of the same operations.  The action width A is
where these kernels branch most: vector or scalar arena loads and stores, the four-way action split of the tcgen05 loss epilogue, the
Philox quads, the padding of the 16-column head tile.  The fp32 kernels take 1 <= A <= 31, the tcgen05 ones 1 <= A <= 15.

  a. fp32 ppo_head_loss + ppo_loss_finalize against float64 autograd through the oracle's loss functions, on chunked arena rows
     whose 128-row blocks straddle chunks.  Tolerances of tests/test_kernels_gpu.py::_loss_case; d_alast and d_logstd, sums whose
     terms cancel, take its rtol relative to the sum of the terms' magnitudes.
  b. fp32 policy_head_sample against a float64 head, with the noise tape and with Philox.  A Philox draw does not depend on A: the
     first A columns of a 31-wide draw are the draw at width A.
  c. tcgen05 fwd_train + bwd against the kernel-faithful reference of tests/test_tc_faithful_gpu.py, restated with A as a parameter.
     Its tolerances.
  d. tcgen05 fwd_rollout: mu and value against the same reference; the Philox noise equals the fp32 kernel's; the scalar stores
     taken for unaligned outputs give the bytes of the vector stores.
  e. The tcgen05 workspaces need no initialisation: buffers filled with 0xFF bytes (NaN as bf16, fp32 and fp64) must give results
     bit-identical to zeroed ones.
"""
import math
import os
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import ppo_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_mlp_tc_gpu import decode_tiles, rel_l2, cosine  # noqa: E402
from test_tc_faithful_gpu import ACTS, NATIVE, bf, mm  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = 'cuda'
WIDTHS = (1, 3, 4, 6, 8, 15, 31)     # 31 = the fp32 kernels' MAXA - 1


# ------------------------------------------------------------------------------------------ a. fp32 loss head
LOSS_CFGS = {'default': {}, 'noppo': {'ppo': False}, 'hardclip': {'use_smooth_clamp': False, 'clip_value': False},
             'bound': {'bound_loss_type': 'bound', 'bounds_loss_coef': 0.01},
             'reg': {'bound_loss_type': 'regularisation', 'bounds_loss_coef': 0.01}}
ACT_LAST = {0: (lambda x: x, lambda a: torch.ones_like(a)), 1: (F.elu, lambda a: torch.where(a > 0, torch.ones_like(a), a + 1.0)),
            2: (torch.relu, lambda a: (a > 0).to(a.dtype)), 3: (torch.tanh, lambda a: 1.0 - a * a)}
HLS = (16, 64, 128, 256)       # 128 and 256 stage more than 48 KB of shared memory
MASKS = (None, 'random', 'zero')


def _pairwise_loss_cases():
    """every (A, Hl) pair once; act_last, config and mask rotate so that every pair of values of any two of the five factors occurs"""
    cfgs = list(LOSS_CFGS)
    cases = [(A, Hl, (i + j) % 4, cfgs[(i + 2 * j) % 5], MASKS[(i + j) % 3]) for i, A in enumerate(WIDTHS) for j, Hl in enumerate(HLS)]
    for i, A in enumerate(WIDTHS):       # the fifth config of each width, with the act_last values that complete act_last x config
        cases.append((A, HLS[i % 4], (0, 1, 2, 3, 3, 0, 1)[i], cfgs[(i + 3) % 5], MASKS[(i + 2) % 3]))
    return cases


LOSS_CASES = _pairwise_loss_cases()


def _close_to_sum(got, ref, terms_abs, rtol, atol, name):
    err, lim = (got.double() - ref).abs(), atol + rtol * terms_abs
    assert bool((err <= lim).all()), (name, float((err / lim).max()), float(err.max()))


def _off_kinks(nlp, value, old_nlp, old_v, ret, e_clip, smooth):
    """Move old_nlp / old_v of rows whose loss has a kink (or whose clip-fraction test flips) within rounding distance of the kernel's
    fp32 arithmetic, so that per-row gradients and the clip fraction are well defined at fp32 tolerances."""
    mi, mx = 1.0 - e_clip, 1.0 + e_clip
    for _ in range(8):
        ratio = torch.exp(old_nlp - nlp)
        near = ((ratio - mi).abs() < 1e-3) | ((ratio - mx).abs() < 1e-3)
        if smooth:
            near |= (ratio - O.smooth_clamp(ratio, mi, mx)).abs() < 1e-3
        delta = value - old_v
        l1, l2 = (value - ret) ** 2, (old_v + delta.clamp(-e_clip, e_clip) - ret) ** 2
        vnear = ((delta.abs() - e_clip).abs() < 1e-3) | (((l1 - l2).abs() < 1e-3) & (delta.abs() > e_clip))
        if not (near.any() or vnear.any()):
            return old_nlp, old_v
        old_nlp, old_v = old_nlp + 0.05 * near, old_v + 0.05 * vnear
    raise AssertionError('could not move the inputs off the loss kinks')


@pytest.mark.parametrize('A,Hl,act_last,cfg_name,mask_kind', LOSS_CASES)
def test_fp32_loss_head_vs_float64_autograd(A, Hl, act_last, cfg_name, mask_kind):
    from rl_games_b200 import ops
    from rl_games_b200.ops import LossCfg
    g = torch.Generator().manual_seed(1000 * A + Hl + 10 * act_last)
    H, rpc, stride, e0 = 3, 100, 320, 16          # 3 chunks of 100 rows: 128-row blocks straddle chunks
    M = H * rpc
    cfg = dict(O.DEFAULT_CFG); cfg.update(LOSS_CFGS[cfg_name]); cfg['entropy_coef'] = 0.01
    e_clip = cfg['e_clip']
    act_fn, act_grad = ACT_LAST[act_last]
    a_last = act_fn(torch.randn(M, Hl, generator=g) * 1.5).double()
    Wh = torch.randn(A + 1, Hl, generator=g).double() * (1.2 / math.sqrt(Hl)); bh = torch.randn(A + 1, generator=g).double() * 0.1
    logstd = torch.randn(A, generator=g).double() * 0.3
    actions = torch.randn(M, A, generator=g).double()
    old_mu = torch.randn(M, A, generator=g).double() * 0.5; old_sigma = torch.rand(M, A, generator=g).double() + 0.5
    old_v = torch.randn(M, generator=g).double(); ret = torch.randn(M, generator=g).double(); adv = torch.randn(M, generator=g).double()
    mask = {None: None, 'random': (torch.rand(M, generator=g) < 0.7).double(), 'zero': torch.zeros(M, dtype=torch.float64)}[mask_kind]
    # the kernel reads fp32 values: round every input once, then the reference works on exactly those values in float64
    a_last, Wh, bh, logstd, actions, old_mu, old_sigma, old_v, ret, adv = (t.float().double() for t in (a_last, Wh, bh, logstd, actions, old_mu,
                                                                                                          old_sigma, old_v, ret, adv))
    with torch.no_grad():
        head0 = a_last @ Wh.t() + bh
        sg0 = torch.exp(logstd).expand(M, A)
        nlp0 = O.neglogp_fn(actions, head0[:, 1:], sg0, logstd.expand(M, A))
    old_nlp = (nlp0 + torch.randn(M, generator=g).double() * 0.3).float().double()
    old_nlp, old_v = _off_kinks(nlp0, head0[:, 0], old_nlp, old_v, ret, e_clip, cfg['use_smooth_clamp'])
    old_nlp, old_v = old_nlp.float().double(), old_v.float().double()

    # ---------------- float64 reference: the oracle's loss functions + autograd ----------------
    al = a_last.clone().requires_grad_()
    ls = logstd.expand(M, A).clone().requires_grad_()        # one logstd row per sample: its grad holds each sample's d_logstd terms
    head = al @ Wh.t() + bh
    value, mu = head[:, :1], head[:, 1:]
    sigma = torch.exp(ls)
    nlp = O.neglogp_fn(actions, mu, sigma, ls)
    a_l = O.actor_loss(old_nlp, nlp, adv, cfg['ppo'], e_clip, smooth=cfg['use_smooth_clamp'])
    c_l = O.critic_loss(old_v.unsqueeze(1), value, e_clip, ret.unsqueeze(1), cfg['clip_value'])
    ent = (0.5 + 0.5 * math.log(2 * math.pi) + ls).sum(-1)
    b_l = (O.bound_loss if cfg['bound_loss_type'] == 'bound' else O.reg_loss)(mu, cfg['bounds_loss_coef'])
    (a_m, c_m, e_m, b_m), _ = O.apply_masks([a_l.unsqueeze(1), c_l, ent.unsqueeze(1), b_l.unsqueeze(1)], mask)
    loss = a_m + 0.5 * c_m * cfg['critic_coef'] - e_m * cfg['entropy_coef'] + b_m * cfg['bounds_loss_coef']
    head.retain_grad()
    loss.backward()
    mk = torch.ones(M, dtype=torch.float64) if mask is None else mask
    kl_rows = O.policy_kl(mu.detach(), sigma.detach(), old_mu, old_sigma, reduce=False)
    kl = (kl_rows * mk).sum() / mk.sum().clamp(min=1.0)
    lr_ = old_nlp - nlp.detach()
    clipped = ((lr_ < math.log(1.0 - e_clip)) | (lr_ > math.log(1.0 + e_clip))).double()
    ref_stats = [a_m, c_m, e_m, b_m, kl, mk.sum(), (mk * clipped).sum() / mk.sum().clamp(min=1.0)]

    # ---------------- fp32 kernel on chunked arena rows ----------------
    def arena(x):        # row-space [M, ...] -> [H, stride, ...] with the minibatch at rows e0..e0+rpc of each chunk, noise elsewhere
        t = torch.randn((H, stride) + tuple(x.shape[1:]), generator=g)
        t[:, e0:e0 + rpc] = x.float().view((H, rpc) + tuple(x.shape[1:]))
        return t.to(DEV)

    def rows(t):
        return t[:, e0:e0 + rpc].reshape((M,) + tuple(t.shape[2:]))

    def base(t):
        return None if t is None else t[0, e0:]
    ar_act, ar_omu, ar_osg = arena(actions), arena(old_mu), arena(old_sigma)
    ar_ov, ar_ret, ar_onlp, ar_adv = arena(old_v), arena(ret), arena(old_nlp), arena(adv)
    ar_mask = None if mask is None else arena(mask)
    omu_before, osg_before = ar_omu.clone(), ar_osg.clone()
    c = LossCfg(e_clip, cfg['critic_coef'], cfg['bounds_loss_coef'] or 0.0, int(cfg['bounds_loss_coef'] is not None),
                {'bound': 1, 'regularisation': 2}.get(cfg['bound_loss_type'], 0), int(cfg['clip_value']), int(cfg['use_smooth_clamp']),
                int(cfg['ppo']))
    inv = None if mask is None else torch.tensor([1.0 / max(float(mask.sum()), 1.0)], device=DEV)
    partials = torch.zeros((M + 127) // 128, ops.loss_partial_stride(), dtype=torch.float64, device=DEV)
    d_head = torch.empty(M, A + 1, device=DEV); d_al = torch.empty(M, Hl, device=DEV)
    mu_o = torch.empty(M, A, device=DEV); v_o = torch.empty(M, device=DEV); nlp_o = torch.empty(M, device=DEV)
    nb = ops.ppo_head_loss(a_last.float().to(DEV), Wh.float().to(DEV), bh.float().to(DEV), logstd.float().to(DEV), base(ar_act), base(ar_omu),
                           base(ar_osg), base(ar_ov), base(ar_ret), base(ar_onlp), base(ar_adv), base(ar_mask), rpc, stride, M, A, c, inv,
                           d_head, d_al, act_last, partials, mu_out=mu_o, value_out=v_o, neglogp_out=nlp_o)
    stats = torch.zeros(16, device=DEV); dls = torch.empty(A, device=DEV)
    ops.ppo_loss_finalize(partials, nb, A, torch.tensor([cfg['entropy_coef']], device=DEV), stats, dls)
    torch.cuda.synchronize()
    f = lambda t: t.detach().float()    # noqa: E731

    torch.testing.assert_close(mu_o.cpu(), f(mu), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(v_o.cpu(), f(value[:, 0]), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(nlp_o.cpu(), f(nlp), rtol=1e-5, atol=1e-5)
    st = stats.cpu()
    for k, (rt, at) in enumerate([(1e-4, 1e-6), (1e-4, 1e-6), (1e-5, 1e-6), (1e-4, 1e-6), (1e-4, 1e-6)]):
        torch.testing.assert_close(st[k], f(ref_stats[k]), rtol=rt, atol=at, msg=lambda m: f'stat {k}: {m}')
    assert float(st[5]) == float(ref_stats[5])                                   # mask sum (exact: a count)
    assert float(st[6]) == pytest.approx(float(ref_stats[6]), rel=1e-6, abs=0)    # clip fraction (no row sits on its boundary)
    torch.testing.assert_close(d_head.cpu(), f(head.grad), rtol=2e-4, atol=1e-7)
    # d_alast and d_logstd are sums whose terms cancel: each per-sample d_head carries the fp32 rounding of a neglogp of up to ~50
    # (amplified ~10x by the smooth clamp), so their rtol applies to the sum of the terms' magnitudes
    _close_to_sum(d_al.cpu(), al.grad * act_grad(a_last), (head.grad.abs() @ Wh.abs()) * act_grad(a_last).abs(), 2e-4, 1e-7, 'd_alast')
    _close_to_sum(dls.cpu(), ls.grad.sum(0), ls.grad.abs().sum(0), 2e-4, 1e-6, 'd_logstd')
    # mu / sigma written back at the mapped arena rows (datasets.py:33-43), every other arena row untouched
    torch.testing.assert_close(rows(ar_omu).cpu(), f(mu), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(rows(ar_osg).cpu(), f(sigma), rtol=1e-6, atol=1e-6)
    outside = torch.ones(H, stride, dtype=torch.bool); outside[:, e0:e0 + rpc] = False
    assert torch.equal(ar_omu.cpu()[outside], omu_before.cpu()[outside]) and torch.equal(ar_osg.cpu()[outside], osg_before.cpu()[outside])


# ------------------------------------------------------------------------------------------ b. fp32 policy_head_sample
@pytest.mark.parametrize('A,Hl,clip_actions,normalize_value', [(1, 16, True, True), (3, 64, False, True), (4, 128, True, False),
                                                               (6, 256, False, False), (8, 64, True, True), (15, 128, False, True),
                                                               (31, 256, True, False), (31, 16, False, True)])
def test_fp32_policy_head_sample_vs_float64(A, Hl, clip_actions, normalize_value):
    from rl_games_b200 import ops
    g = torch.Generator().manual_seed(100 * A + Hl)
    N, N31, seed, step = 515, 8192, 77, 3
    a_last = F.elu(torch.randn(N, Hl, generator=g))
    Wh = torch.randn(A + 1, Hl, generator=g) * (1.2 / math.sqrt(Hl)); bh = torch.randn(A + 1, generator=g) * 0.1
    logstd = torch.randn(A, generator=g) * 0.3
    noise = torch.randn(N, A, generator=g)
    vm, vv = torch.tensor([1.5], dtype=torch.float64), torch.tensor([4.0], dtype=torch.float64)
    lo, hi = torch.rand(A, generator=g) - 2.0, torch.rand(A, generator=g) + 1.0
    dones_cur = (torch.rand(N, generator=g) < 0.3).to(torch.uint8).to(DEV)
    prev = (torch.rand(N, generator=g) < 0.3).float().to(DEV)
    head = a_last.double() @ Wh.double().t() + bh.double()
    mu, val = head[:, 1:], head[:, 0]
    sigma = torch.exp(logstd.double()).expand_as(mu)
    if normalize_value:
        val = torch.sqrt(vv.float().double() + 1e-5) * val.clamp(-5.0, 5.0) + 1.5
    dev = [x.to(DEV) for x in (a_last, Wh, bh, logstd)]
    ep = torch.full((1,), 5, dtype=torch.int64, device=DEV)

    def run(noise_t, values_only=False):
        o = {k: torch.full((N, A), float('nan'), device=DEV) for k in ('a', 'm', 's', 'env')}
        o.update(nl=torch.full((N,), float('nan'), device=DEV), v=torch.empty(N, device=DEV), d=torch.zeros(N, dtype=torch.uint8, device=DEV),
                 valid=torch.full((N,), float('nan'), device=DEV))
        ops.policy_head_sample(*dev, vm.to(DEV), vv.to(DEV), normalize_value, noise_t, seed, ep, step, o['a'], o['m'], o['s'], o['nl'], o['v'],
                               o['env'], clip_actions, lo.to(DEV), hi.to(DEV), dones_cur, o['d'], prev, o['valid'], N, A, values_only=values_only)
        return o
    # noise tape
    t = run(noise.to(DEV))
    act = mu + sigma * noise.double()
    torch.testing.assert_close(t['m'].cpu(), mu.float(), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(t['s'].cpu(), sigma.float(), rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(t['a'].cpu(), act.float(), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(t['nl'].cpu(), O.neglogp_fn(act, mu, sigma, logstd.double().expand_as(mu)).float(), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(t['v'].cpu(), val.float(), rtol=1e-5, atol=1e-5)
    env = (act.clamp(-1.0, 1.0) * ((hi - lo) * 0.5) + (hi + lo) * 0.5) if clip_actions else act
    torch.testing.assert_close(t['env'].cpu(), env.float(), rtol=1e-5, atol=1e-5)
    assert torch.equal(t['d'], dones_cur) and torch.equal(t['valid'], 1 - prev)
    # Philox: a zero head with unit sigma gives the raw draw; a draw at width A is the first A columns of the one at 31
    e31 = torch.empty(N31, 31, device=DEV); junk = [torch.empty(N31, 31, device=DEV) for _ in range(2)]
    ops.policy_head_sample(torch.zeros(N31, 8, device=DEV), torch.zeros(32, 8, device=DEV), torch.zeros(32, device=DEV),
                           torch.zeros(31, device=DEV), None, None, False, None, seed, ep, step, e31, junk[0], junk[1],
                           torch.empty(N31, device=DEV), torch.empty(N31, device=DEV), None, False, None, None, None, None, None, None, N31, 31)
    p = run(None)
    eps = (p['a'] - p['m']) / p['s']
    torch.testing.assert_close(eps, e31[:N, :A], rtol=0, atol=1e-5)
    torch.testing.assert_close(p['m'], t['m'], rtol=0, atol=0)
    torch.testing.assert_close(p['nl'].double(), 0.5 * (eps.double() ** 2).sum(-1) + 0.5 * math.log(2 * math.pi) * A + float(logstd.sum()),
                               rtol=1e-5, atol=1e-5)
    e = e31.cpu().double()
    assert abs(float(e.mean())) < 0.01 and abs(float(e.var()) - 1.0) < 0.02
    corr = torch.corrcoef(e.t()) - torch.eye(31, dtype=torch.float64)
    assert float(corr.abs().max()) < 0.06, float(corr.abs().max())        # 31 distinct streams (8192 samples: sd of a correlation ~0.011)
    # values_only: the value, and nothing else
    vo = run(noise.to(DEV), values_only=True)
    assert torch.equal(vo['v'], t['v'])
    assert torch.isnan(vo['a']).all() and torch.isnan(vo['m']).all() and torch.isnan(vo['nl']).all()


# ------------------------------------------------------------------------------------------ c. / d. / e. tcgen05 kernels
TC_SHAPES = [   # D, units, A, activation
    (11, [256, 128, 64], 3, 'elu'),       # hopper.yaml (Gymnasium v5: obs 11, 3 actions)
    (17, [128, 64, 32], 6, 'elu'),        # halfcheetah.yaml (obs 17, 6 actions)
    (17, [256, 128, 64], 6, 'elu'),       # walker2d.yaml (obs 17, 6 actions)
    (60, [256, 128, 64], 1, 'elu'),
    (33, [256, 128, 64], 15, 'elu'),      # no head padding left in the 16-column tile
    (44, [128, 64, 32], 12, 'tanh'),
    (100, [256, 128, 64], 5, 'elu'),      # wide observations (kind 2), odd A
]
TC_ROWS = [(4, 512, 256, False), (2, 384, 128, True), (1, 1000, 1000, False), (2, 384, 128, True), (1, 1000, 1000, True),
           (4, 512, 256, False), (2, 384, 128, True)]       # H, N, envs per minibatch, masked: one per shape


def _make_net(g, D, units, A):
    ins, W, b = D, [], []
    for u in units:
        W.append((torch.randn(u, ins, generator=g) / math.sqrt(ins)).to(DEV))
        b.append((torch.randn(u, generator=g) * 0.1).to(DEV))
        ins = u
    Wh = (torch.randn(A + 1, ins, generator=g) / math.sqrt(ins)).to(DEV)
    bh = (torch.randn(A + 1, generator=g) * 0.1).to(DEV)
    logstd = (torch.randn(A, generator=g) * 0.2).to(DEV)
    return W, b, Wh, bh, logstd


def _tc_inputs(D, units, A, H, N, epm, masked, seed):
    g = torch.Generator().manual_seed(seed)
    x = dict(D=D, units=units, A=A, H=H, N=N, epm=epm, M=H * epm, e0=128 if N > epm else 0)
    x['W'], x['b'], x['Wh'], x['bh'], x['logstd'] = _make_net(g, D, units, A)
    x['obs'] = (torch.randn(H, N, D, generator=g) * 2 + 0.5).to(DEV)
    x['nm'] = (torch.randn(D, generator=g) * 0.3).to(DEV); x['ns'] = (torch.rand(D, generator=g) + 0.7).to(DEV)
    x['actions'] = torch.randn(H, N, A, generator=g).to(DEV)
    x['old_mu'] = (torch.randn(H, N, A, generator=g) * 0.5).to(DEV); x['old_sigma'] = (torch.rand(H, N, A, generator=g) + 0.5).to(DEV)
    x['old_v'] = torch.randn(H, N, generator=g).to(DEV); x['ret'] = torch.randn(H, N, generator=g).to(DEV)
    x['old_nlp'] = (torch.randn(H, N, generator=g) * 0.3 + 9.0).to(DEV); x['adv'] = torch.randn(H, N, generator=g).to(DEV)
    x['mask'] = (torch.rand(H, N, generator=g) < 0.7).float().to(DEV) if masked else None
    e0, epm = x['e0'], epm
    x['inv'] = torch.tensor([1.0 / max(float(x['mask'][:, e0:e0 + epm].sum()), 1.0)], device=DEV) if masked else None
    return x


def _rows(x, t):        # kernel row order: t * epm + e
    return torch.cat([t[k, x['e0']:x['e0'] + x['epm']] for k in range(x['H'])])


def _offsets(D, units, A):
    offs, o, ins = {}, A, D
    for i, u in enumerate(units):
        offs[f'W{i}'] = o; o += u * ins
        offs[f'b{i}'] = o; o += u
        ins = u
    offs['W_head'] = o; o += (A + 1) * ins
    offs['b_head'] = o; o += A + 1
    return offs, o


E_CLIP, CRITIC_COEF = 0.2, 2.0


def _tc_train(x, act_id, fill):
    """fwd_train + loss finalise + bwd + split reduce, every workspace the kernels write pre-filled with the byte `fill`"""
    from rl_games_b200 import ops
    from rl_games_b200.ops import LossCfg
    D, units, A, M, N = x['D'], x['units'], x['A'], x['M'], x['N']
    sl = lambda t: None if t is None else t[0, x['e0']:]   # noqa: E731
    buf = lambda n: torch.full((n,), fill, dtype=torch.uint8, device=DEV)   # noqa: E731
    n_tiles = (M + 127) // 128
    tb = ops.tc_tile_bytes(D, units, A)
    wpack = torch.zeros(ops.tc_pack_bytes(D, units, A), dtype=torch.uint8, device=DEV)
    ops.tc_pack_weights(x['W'][0], x['W'][1], x['W'][2], x['Wh'], D, units, A, wpack)
    act = [buf(n_tiles * tb[i]) for i in range(3)]
    dhead, delta2, delta1 = buf(n_tiles * tb[3]), buf(n_tiles * tb[1]), buf(n_tiles * tb[0])
    xt = buf(n_tiles * ops.tc_xtile_bytes(D, units, A))
    stride = ops.loss_partial_stride()
    partials = buf(148 * stride * 8).view(torch.float64).view(148, stride)
    mu_t, sg_t = x['old_mu'].clone(), x['old_sigma'].clone()
    cfg = LossCfg(E_CLIP, CRITIC_COEF, 0.0, 1, 2, 1, 1, 1)
    nbt = ops.tc_mlp_fwd_train(sl(x['obs']), x['epm'], N, D, x['nm'], x['ns'], wpack, x['b'], x['bh'], x['logstd'], units, M, A, sl(x['actions']),
                               sl(mu_t), sl(sg_t), sl(x['old_v']), sl(x['ret']), sl(x['old_nlp']), sl(x['adv']), sl(x['mask']), cfg, x['inv'],
                               act, dhead, partials, xtile=xt, activation=act_id)
    stats = torch.zeros(16, device=DEV); dls = torch.empty(A, device=DEV)
    ops.ppo_loss_finalize(partials, nbt, A, torch.tensor([0.0], device=DEV), stats, dls)
    offs, P = _offsets(D, units, A)
    part = buf(148 * P * 4).view(torch.float32).view(148, P)
    npart = ops.tc_mlp_bwd(sl(x['obs']), x['epm'], N, D, x['nm'], x['ns'], wpack, units, M, A, act, dhead, delta2, delta1, part, P, offs,
                           xtile=xt, activation=act_id)
    grad = torch.zeros(P, device=DEV)
    ops.reduce_splits(part[0, A:], grad[A:], P - A, npart, split_stride=P)
    torch.cuda.synchronize()
    return dict(mu=mu_t, sigma=sg_t, stats=stats, dls=dls, grad=grad, act=act, dhead=dhead, delta2=delta2, delta1=delta1,
                n_tiles=n_tiles, offs=offs)


def _faithful_trunk(x, obs_rows, act_fn):
    """normalised observations and hidden activations as the kernels round them (bf16 operands, exact products, fp32 bias/activation)"""
    xb = bf(torch.clamp((obs_rows - x['nm']) * (1.0 / x['ns']), -5.0, 5.0))
    a = [xb]
    for w, bb in zip(x['W'], x['b']):
        a.append(bf(act_fn(mm(a[-1], bf(w)) + bb)))
    return a


@pytest.mark.parametrize('D,units,A,actname,H,N,epm,masked', [s + r for s, r in zip(TC_SHAPES, TC_ROWS)])
def test_tc_fwd_loss_bwd_widths_vs_kernel_faithful_reference(D, units, A, actname, H, N, epm, masked):
    from rl_games_b200 import ops
    act_id, act_fn, act_grad = ACTS[actname]
    assert ops.tc_kind(D, units, A) == (2 if D > 64 else 1)
    x = _tc_inputs(D, units, A, H, N, epm, masked, seed=7 * H + N + D + 100 * A)
    M, R = x['M'], lambda t: _rows(x, t)    # noqa: E731
    # ---------------- kernel-faithful reference ----------------
    xb, a1, a2, a3 = _faithful_trunk(x, R(x['obs']), act_fn)
    Wb, Whb = [bf(w) for w in x['W']], bf(x['Wh'])
    head = (mm(a3, Whb) + x['bh']).requires_grad_()
    ls = x['logstd'].clone().requires_grad_()
    value, mu = head[:, 0:1], head[:, 1:]
    sigma = torch.exp(ls).expand_as(mu)
    nlp = O.neglogp_fn(R(x['actions']), mu, sigma, ls.expand_as(mu))
    a_l = O.actor_loss(R(x['old_nlp']), nlp, R(x['adv']), True, E_CLIP, smooth=True)
    c_l = O.critic_loss(R(x['old_v']).unsqueeze(1), value, E_CLIP, R(x['ret']).unsqueeze(1), True)
    ent = (0.5 + 0.5 * math.log(2 * math.pi) + ls.expand_as(mu)).sum(-1)
    b_l = (mu * mu).sum(-1)
    mk = None if x['mask'] is None else R(x['mask'])
    (a_m, c_m, e_m, b_m), _ = O.apply_masks([a_l.unsqueeze(1), c_l, ent.unsqueeze(1), b_l.unsqueeze(1)], mk)
    loss = a_m + 0.5 * c_m * CRITIC_COEF - e_m * 0.0 + b_m * 0.0
    loss.backward()
    kl_rows = O.policy_kl(mu.detach(), sigma.detach(), R(x['old_mu']), R(x['old_sigma']), reduce=False)
    kl = kl_rows.mean() if mk is None else (kl_rows * mk).sum() / mk.sum().clamp(min=1.0)
    dh = bf(head.grad)
    d3 = bf(mm(dh, Whb.t().contiguous()) * act_grad(a3))
    d2 = bf(mm(d3, Wb[2].t().contiguous()) * act_grad(a2))
    d1 = bf(mm(d2, Wb[1].t().contiguous()) * act_grad(a1))
    ref = {'W_head': mm(dh.t().contiguous(), a3.t().contiguous()), 'b_head': dh.sum(0),
           'W2': mm(d3.t().contiguous(), a2.t().contiguous()), 'b2': d3.sum(0),
           'W1': mm(d2.t().contiguous(), a1.t().contiguous()), 'b1': d2.sum(0),
           'W0': mm(d1.t().contiguous(), xb.t().contiguous()), 'b0': d1.sum(0)}
    # ---------------- tcgen05 kernels ----------------
    t = _tc_train(x, act_id, 0)
    n_tiles, tanh = t['n_tiles'], actname == 'tanh'
    report = {}
    for i, (C, r) in enumerate(zip(units, (a1, a2, a3))):
        full = decode_tiles(t['act'][i], n_tiles, NATIVE[i])[:M]
        if C < NATIVE[i]:
            assert float(full[:, C:].abs().max()) == 0.0          # padded units are exactly zero
        report[f'a{i + 1}'] = rel_l2(full[:, :C], r)
        assert report[f'a{i + 1}'] < (6e-3 if tanh else 3e-3), (i, report)
    got_mu = R(t['mu'])
    report['mu_rel_l2'] = rel_l2(got_mu, mu.detach())
    assert report['mu_rel_l2'] < (3e-3 if tanh else 1e-3), report
    torch.testing.assert_close(got_mu, mu.detach(), rtol=0, atol=1.5e-2 if tanh else 6e-3)
    torch.testing.assert_close(R(t['sigma']), sigma.detach(), rtol=1e-5, atol=1e-6)
    outside = torch.ones(H, N, dtype=torch.bool, device=DEV); outside[:, x['e0']:x['e0'] + epm] = False
    assert torch.equal(t['mu'][outside], x['old_mu'][outside]) and torch.equal(t['sigma'][outside], x['old_sigma'][outside])
    for k, r in enumerate([a_m, c_m, e_m, b_m, kl]):
        report[f'stat{k}'] = (float(t['stats'][k]), float(r))
        assert float(t['stats'][k]) == pytest.approx(float(r), rel=2e-2 if tanh else 5e-3, abs=2e-5), (k, report)
    assert float(t['stats'][5]) == (float(mk.sum()) if mk is not None else float(M))
    dh_t = decode_tiles(t['dhead'], n_tiles, 16)[:M]
    if A < 15:
        assert float(dh_t[:, A + 1:].abs().max()) == 0.0          # head columns past the last action hold zeros
    dh_t = dh_t[:, :A + 1]
    report['d_head'] = rel_l2(dh_t, dh)
    tol_g, tol_c = (3e-2, 0.999) if tanh else (1e-2, 0.9999)
    assert report['d_head'] < tol_g and cosine(dh_t, dh) > tol_c, report
    report['d_logstd'] = rel_l2(t['dls'], ls.grad)
    assert report['d_logstd'] < 2e-3, report
    for name, C, CN, r in (('delta2', units[1], NATIVE[1], d2), ('delta1', units[0], NATIVE[0], d1)):
        got = decode_tiles(t[name], n_tiles, CN)[:M, :C]
        report[name] = rel_l2(got, r)
        assert report[name] < 1.5 * tol_g and cosine(got, r) > tol_c, report
    for k, r in ref.items():
        got = t['grad'][t['offs'][k]:t['offs'][k] + r.numel()].view_as(r)
        report['g' + k] = rel_l2(got, r)
        assert report['g' + k] < tol_g and cosine(got, r) > tol_c, (k, report)
    print('faithful-reference errors', (D, units, A, actname, H, N, epm, masked),
          {k: (round(v, 6) if isinstance(v, float) else v) for k, v in report.items()})


def _tc_rollout(x, act_id, N, noise, outs, l1_fill=0, ep=None):
    from rl_games_b200 import ops
    D, units, A = x['D'], x['units'], x['A']
    vm, vv = torch.tensor([1.5], dtype=torch.float64, device=DEV), torch.tensor([4.0], dtype=torch.float64, device=DEV)
    lo, hi = torch.full((A,), -1.0, device=DEV), torch.full((A,), 1.0, device=DEV)
    scratch = torch.full(((N + 127) // 128 * ops.tc_tile_bytes(D, units, A)[0],), l1_fill, dtype=torch.uint8, device=DEV) if D > 64 else None
    wpack = torch.zeros(ops.tc_pack_bytes(D, units, A), dtype=torch.uint8, device=DEV)
    ops.tc_pack_weights(x['W'][0], x['W'][1], x['W'][2], x['Wh'], D, units, A, wpack)
    ops.tc_mlp_fwd_rollout(x['obs'][0, :N], D, x['nm'], x['ns'], wpack, x['b'], x['bh'], x['logstd'], units, N, A, vm, vv, True, noise, 123, ep,
                           9, outs['a'], outs['m'], outs['s'], outs['nl'], outs['v'], outs['e'], True, lo, hi, outs['dc'], outs['d'], None, None,
                           l1_scratch=scratch, activation=act_id)
    torch.cuda.synchronize()
    return outs


def _rollout_outs(N, A, offset=0):
    """output arenas; offset = 1 shifts the four [N, A] ones by one float, off the 16-byte alignment of the vector stores"""
    o = {k: torch.full((N * A + offset,), float('nan'), device=DEV)[offset:].view(N, A) for k in ('a', 'm', 's', 'e')}
    o.update(nl=torch.empty(N, device=DEV), v=torch.empty(N, device=DEV), d=torch.zeros(N, dtype=torch.uint8, device=DEV),
             dc=torch.ones(N, dtype=torch.uint8, device=DEV))
    return o


@pytest.mark.parametrize('D,units,A,actname', TC_SHAPES + [(60, [256, 128, 64], 4, 'elu')])
def test_tc_rollout_widths_vs_kernel_faithful_reference(D, units, A, actname):
    from rl_games_b200 import ops
    act_id, act_fn, _ = ACTS[actname]
    N, tanh = 1000, actname == 'tanh'
    x = _tc_inputs(D, units, A, 1, N, N, False, seed=3 + A + D)
    g = torch.Generator().manual_seed(5)
    noise = torch.randn(N, A, generator=g).to(DEV)
    t = _tc_rollout(x, act_id, N, noise, _rollout_outs(N, A))
    a = _faithful_trunk(x, x['obs'][0], act_fn)[-1]
    head = mm(a, bf(x['Wh'])) + x['bh']
    mu, val = head[:, 1:], head[:, 0]
    val = torch.sqrt(torch.tensor(4.0 + 1e-5, device=DEV)) * torch.clamp(val, -5.0, 5.0) + 1.5
    rep = {'mu_max_abs': float((t['m'] - mu).abs().max()), 'mu_rel_l2': rel_l2(t['m'], mu), 'v_max_abs': float((t['v'] - val).abs().max()),
           'v_rel_l2': rel_l2(t['v'], val)}
    print('faithful-reference rollout errors', (D, units, A, actname), {k: round(v, 6) for k, v in rep.items()})
    assert rep['mu_rel_l2'] < (3e-3 if tanh else 1e-3) and rep['v_rel_l2'] < (3e-3 if tanh else 1e-3), rep
    torch.testing.assert_close(t['m'], mu, rtol=0, atol=1.5e-2 if tanh else 6e-3)
    torch.testing.assert_close(t['v'], val, rtol=0, atol=3e-2 if tanh else 1.2e-2)
    sigma = torch.exp(x['logstd']).expand_as(mu)
    torch.testing.assert_close(t['s'], sigma, rtol=1e-6, atol=0)
    torch.testing.assert_close(t['a'], t['m'] + sigma * noise, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(t['e'], torch.clamp(t['a'], -1, 1), rtol=0, atol=1e-6)
    torch.testing.assert_close(t['nl'], O.neglogp_fn(t['a'], t['m'], sigma, x['logstd'].expand_as(mu)), rtol=1e-5, atol=1e-4)
    assert torch.equal(t['d'], t['dc'])
    # Philox: the same (seed, epoch, step, row) draws as the fp32 kernel (zero head, unit sigma: its actions are the raw draw)
    ep = torch.full((1,), 2, dtype=torch.int64, device=DEV)
    p = _tc_rollout(x, act_id, N, None, _rollout_outs(N, A), ep=ep)
    eps_ref = torch.empty(N, A, device=DEV); junk = [torch.empty(N, A, device=DEV) for _ in range(2)]
    ops.policy_head_sample(torch.zeros(N, 8, device=DEV), torch.zeros(A + 1, 8, device=DEV), torch.zeros(A + 1, device=DEV),
                           torch.zeros(A, device=DEV), None, None, False, None, 123, ep, 9, eps_ref, junk[0], junk[1],
                           torch.empty(N, device=DEV), torch.empty(N, device=DEV), None, False, None, None, None, None, None, None, N, A)
    torch.testing.assert_close((p['a'] - p['m']) / p['s'], eps_ref, rtol=0, atol=1e-5)
    if A % 4 == 0:
        # outputs one float off 16-byte alignment take the scalar stores: the same bytes as the vector stores
        u = _tc_rollout(x, act_id, N, None, _rollout_outs(N, A, offset=1), ep=ep)
        for k in ('a', 'm', 's', 'e', 'nl', 'v'):
            assert torch.equal(u[k], p[k]), k


@pytest.mark.parametrize('D,units,A,actname', [(11, [256, 128, 64], 3, 'elu'), (60, [256, 128, 64], 8, 'elu'), (60, [128, 64, 32], 15, 'relu'),
                                               (100, [256, 128, 64], 5, 'elu')])
def test_tc_workspaces_need_no_initialisation(D, units, A, actname):
    """Every byte the tcgen05 kernels read from their workspaces (activation, d_head, delta and X tiles, split and loss partials, the
    wide rollout's layer-1 scratch) was written by the kernel that produces it.  Bytes of 0xFF (NaN) left in any of them must not
    reach a result: the run must be finite and bit-identical to one on zeroed buffers.  1000 rows: the last tile is partial."""
    act_id = ACTS[actname][0]
    x = _tc_inputs(D, units, A, 1, 1000, 1000, True, seed=11 + A)
    zero, poison = _tc_train(x, act_id, 0), _tc_train(x, act_id, 0xFF)
    for k in ('mu', 'sigma', 'stats', 'dls', 'grad'):
        assert torch.isfinite(poison[k]).all(), (k, int((~torch.isfinite(poison[k])).sum()))
        assert torch.equal(poison[k], zero[k]), k
    if D > 64:
        N = 1000
        noise = torch.randn(N, A, generator=torch.Generator().manual_seed(2)).to(DEV)
        rz = _tc_rollout(x, act_id, N, noise, _rollout_outs(N, A), l1_fill=0)
        rp = _tc_rollout(x, act_id, N, noise, _rollout_outs(N, A), l1_fill=0xFF)
        for k in ('a', 'm', 's', 'e', 'nl', 'v'):
            assert torch.isfinite(rp[k]).all() and torch.equal(rp[k], rz[k]), k
