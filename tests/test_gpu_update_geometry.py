"""The hand-written PPO update (csrc/policy_train.cu, policy_wgrad.cu, policy_dense.cu) and the rollout forward
(csrc/policy_fused.cu) at the launch geometry production runs: a minibatch of T*B/4 = 32*16384/4 = 131072 windows
(agents/ppo.py:151) and a 65536-env rollout.  Several update kernels change what each warp does as the minibatch
grows (rows per warp of ln_bwd / embed_mask, samples per warp of head_bwd, grid-stride passes of the attention and loss
kernels); `geometry` restates those launch formulas and every test first checks that its size really reaches them.

The forward is row-local, so the big run must equal a small handle run over chunks bit for bit.  The backward is
row-local up to its fp32 column sums: with the output gradient nonzero only on a set S of 1024 windows placed on the
warp-run, grid-stride-pass and 128-row-tile boundaries, the big run's parameter gradient may differ from a 1024-window
run on S by fp32 re-association only (1e-4 of each tensor's largest entry; one dropped or doubled row moves a tensor
by ~3e-2 of it), and it is also tied to fp64 autograd of the mirror network with the bf16 bounds of
test_gpu_policy_train.py."""
import copy

import pytest
import torch

from helpers import assert_logits_close

pytestmark = pytest.mark.gpu

N_PROD = 131072                 # T*B/4 at the default 16384 envs x 32 steps
N_RAGGED = 131035               # same per-warp counts, partial last warp run / attention pass / 128-row tile
N_SET = 1024                    # |S|
CHUNK, CHUNK_CAP = 4000, 4096   # the small handle's chunks: ragged in windows and in 128-row tiles
REASSOC = 1e-4                  # fp32 re-association bound for ~1024 summed terms (expected ~1e-6)


def _cdiv(a, b):
    return -(-a // b)


def geometry(n, sms):
    """Launch geometry of policy_train.cu for an n-window minibatch on `sms` SMs (row_grid, the head_bwd_kernel launch in
    backward_impl, the attention grids of full_layer_fwd / full_layer_bwd, uavtrain_ppo_loss)."""
    def row_run(rows):                                  # row_grid: 8 CTAs of 8 warps per SM, at least 4 rows per warp
        return max(4, _cdiv(rows, sms * 8 * 8))
    attn_warps = min(_cdiv(n, 8), sms * 16) * 8
    loss_threads = min(_cdiv(n, 256), sms * 4) * 256
    return {"row_run": row_run(n),                      # ln_bwd of the last layers (n rows), embed_mask (n windows)
            "token_run": row_run(5 * n),                # ln_bwd of the critic's inner layer (5n token rows)
            "head_run": max(1, _cdiv(n, sms * 8 * 4)),  # head_bwd_kernel
            "attn_warps": attn_warps, "attn_passes": _cdiv(n, attn_warps),
            "loss_passes": _cdiv(n, loss_threads)}


def _assert_reaches_production_paths(n, sms):
    g = geometry(n, sms)
    assert g["row_run"] > 4 and g["token_run"] > 4, ("rows per warp stay at the floor of 4: the register runs of "
                                                      "ln_bwd / embed_mask are not exercised", n, sms, g)
    assert g["head_run"] > 2, ("head_bwd walks <= 2 samples per warp", n, sms, g)
    assert g["attn_passes"] >= 2, ("the attention kernels run one grid-stride pass only", n, sms, g)
    return g


def boundary_windows(n, sms, seed=0):
    """(S, named): S = N_SET sorted window indices holding the first / last window of a spread of warp runs (including the
    last, partial warp and the last CTA), both sides of every attention pass boundary, the rows on either side of a spread
    of 128-row tile edges (5n token rows and n window rows), windows 0 and n - 1, and seeded random windows.  named maps
    each boundary kind to the windows it requires."""
    g = geometry(n, sms)
    named = {}

    def runs(name, units, run, per_window):             # `units` rows in runs of `run`; per_window rows per window
        nruns = _cdiv(units, run)
        picks = set(torch.linspace(0, nruns - 1, 24).round().long().tolist())
        last_cta = (nruns - 1) // 8 * 8                  # the warps of the last CTA
        picks |= set(range(last_cta, nruns))
        rows = set()
        for k in picks:
            rows |= {k * run, min(units, (k + 1) * run) - 1}
        named[name] = sorted({r // per_window for r in rows})

    runs("ln_bwd / embed_mask runs", n, g["row_run"], 1)
    runs("inner-layer ln_bwd runs", 5 * n, g["token_run"], 5)
    runs("head_bwd runs", n, g["head_run"], 1)
    named["attention pass edges"] = sorted({w for k in range(1, g["attn_passes"]) for w in (k * g["attn_warps"] - 1, k * g["attn_warps"])})
    for name, rows, per_window in (("token-row tile edges", 5 * n, 5), ("window-row tile edges", n, 1)):
        ks = set(torch.linspace(1, (rows - 1) // 128, 40).round().long().tolist())
        named[name] = sorted({r // per_window for k in ks for r in (128 * k - 1, 128 * k)} | {128 * ((rows - 1) // 128) // per_window})
    named["ends"] = [0, n - 1]
    chosen = set().union(*named.values())
    assert len(chosen) <= N_SET, len(chosen)
    gen = torch.Generator().manual_seed(seed)
    for w in torch.randperm(n, generator=gen).tolist():
        if len(chosen) == N_SET:
            break
        chosen.add(w)
    return torch.tensor(sorted(chosen), dtype=torch.long), named


def _perturbed_net(seed=0):
    """test_gpu_policy_train.py's network: biases / LayerNorm parameters moved off 0 / 1 so every one of them matters."""
    import uavenv_b200 as ub
    torch.manual_seed(seed)
    net = ub.TransformerActorCritic().cuda()
    with torch.no_grad():
        for p in net.parameters():
            if p.dim() == 1:
                p.add_(torch.randn_like(p) * 0.1)
    return net


def _windows(B, seed):
    """Random windows with 0..4 leading padding rows (episode starts), as in test_gpu_evaluate.py."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    obs = torch.rand(B, 5, 14, device="cuda", generator=g)
    obs[:, :, 13] = 1.0
    lead = torch.arange(B, device="cuda") % 5
    obs[torch.arange(5, device="cuda")[None, :] < lead[:, None]] = 0.0
    return obs


def _cos(a, b):
    return torch.nn.functional.cosine_similarity(a.flatten().double(), b.flatten().double(), dim=0).item()


def _grads(net, outputs, seeds):
    net.zero_grad()
    torch.autograd.backward(list(outputs), list(seeds))
    return {k: (p.grad.clone() if p.grad is not None else None) for k, p in net.named_parameters()}


def _reassoc_ratios(g_big, g_small):
    """max|g_big - g_small| / max|g_small| per parameter tensor (tensors the op leaves at zero are skipped)."""
    out = {}
    for k, s in g_small.items():
        scale = s.abs().max().item()
        if scale > 0:
            out[k] = (g_big[k] - s).abs().max().item() / scale
    return out


def _report(tag, values, fmt="%.2e", pick=max):
    """Print the worst value per tensor family (net + layer kind: 'critic_net.linear1', 'actor_head', ...)."""
    worst = {}
    for k, v in values.items():
        parts = [x for x in k.split(".") if not x.isdigit() and x not in ("weight", "bias")]
        f = ".".join(parts[:1] + parts[-1:] if len(parts) > 1 else parts)
        worst[f] = pick(worst.get(f, v), v)
    print("\n[%s] " % tag + ", ".join(("%s " + fmt) % kv for kv in sorted(worst.items())))


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


@pytest.fixture(scope="module")
def net():
    return _perturbed_net(0)


@pytest.fixture(scope="module")
def net64(net):
    return copy.deepcopy(net).double()


@pytest.fixture(scope="module")
def big():
    from target_allocation_ppo_transformer_b200.networks.fused_train import FusedTrunks
    free0 = torch.cuda.mem_get_info()[0]
    h = FusedTrunks(N_PROD, "cuda")
    print("\n[FusedTrunks(%d)] device memory taken: %.2f GB" % (N_PROD, (free0 - torch.cuda.mem_get_info()[0]) / 1e9))
    yield h
    h.close()


@pytest.fixture(scope="module")
def small():
    from target_allocation_ppo_transformer_b200.networks.fused_train import FusedTrunks
    h = FusedTrunks(CHUNK_CAP, "cuda")
    yield h
    h.close()


SIZES = pytest.mark.parametrize("n", [N_PROD, N_RAGGED])


# ---- 1. the forward is row-local at production size ----------------------------------------------------------------

@SIZES
def test_forward_at_production_size_equals_a_chunked_small_batch_run(n, sms, net, net64, big, small):
    """embed_kernel, dense_kernel with its LayerNorm epilogues, add_ln_train_kernel and the attention kernels compute each
    window by the same per-row operations whatever the batch: features (actor: one layer, critic: two) and logits / value
    must be bit-identical to a 4096-window handle run over chunks of 4000 (ragged last chunk)."""
    _assert_reaches_production_paths(n, sms)
    obs = _windows(n, n)
    S, _ = boundary_windows(n, sms)
    with torch.no_grad():
        feat = big.features(net, obs)
        parts = [small.features(net, obs[i:i + CHUNK]) for i in range(0, n, CHUNK)]
        chunked = torch.cat(parts)
        for k, name in ((0, "actor"), (1, "critic")):
            bad = (feat[:, k] != chunked[:, k]).any(-1).nonzero().flatten()
            assert bad.numel() == 0, "%s features depend on the batch at %d windows, first %s" % (name, bad.numel(), bad[:8].tolist())
        logits, value = big.logits_and_value(net, obs)
        parts = [small.logits_and_value(net, obs[i:i + CHUNK]) for i in range(0, n, CHUNK)]
        assert torch.equal(logits, torch.cat([p[0] for p in parts])) and torch.equal(value, torch.cat([p[1] for p in parts]))
        o64 = obs[S.cuda()].double()
        ref = torch.stack([net64.actor_net.forward_last(o64), net64.critic_net.forward_last(o64)], 1)
        err = (feat[S.cuda()].double() - ref).abs().max().item()
    print("\n[forward n=%d] features on S vs fp64: max abs %.3e" % (n, err))
    assert err < 5e-2


# ---- 2. trunk backward, rows isolated ------------------------------------------------------------------------------

@SIZES
def test_trunk_backward_at_production_size_rows_isolated(n, sms, net, net64, big, small):
    """dfeat nonzero on S only: the 131072-window backward against a 1024-window backward of obs[S] (fp32 re-association
    only: register runs, CTA column sums and atomics of ln_bwd / embed_mask, split-K partials of wgrad_tma_kernel), and
    against fp64 autograd of the mirror network (relative L2 <= 8e-2, cosine >= 0.997 per tensor)."""
    _assert_reaches_production_paths(n, sms)
    obs = _windows(n, n + 1)
    S, named = boundary_windows(n, sms)
    assert all(set(v) <= set(S.tolist()) for v in named.values())
    Sd = S.cuda()
    g = torch.Generator(device="cuda").manual_seed(7)
    d_s = torch.randn(N_SET, 2, 128, device="cuda", generator=g) / N_SET
    dfeat = torch.zeros(n, 2, 128, device="cuda")
    dfeat[Sd] = d_s
    feat = big.features(net, obs)
    g_big = _grads(net, [feat], [dfeat])
    feat_s = small.features(net, obs[Sd])
    assert torch.equal(feat_s, feat[Sd].detach())
    g_small = _grads(net, [feat_s], [d_s])
    o64 = obs[Sd].double()
    ref = torch.stack([net64.actor_net.forward_last(o64), net64.critic_net.forward_last(o64)], 1)
    g64 = _grads(net64, [ref], [d_s.double()])
    for k in g_big:
        if "head" in k:
            assert not g_big[k].any() and not g_small[k].any(), k
    ratios = _reassoc_ratios(g_big, g_small)
    assert set(ratios) == {k for k in g_big if "head" not in k}, "every trunk parameter gets a gradient"
    rel = {k: ((g_big[k].double() - g64[k]).norm() / g64[k].norm()).item() for k in ratios}
    cos = {k: _cos(g_big[k], g64[k]) for k in ratios}
    _report("trunk n=%d re-association" % n, ratios)
    _report("trunk n=%d fp64 rel L2" % n, rel, "%.3f")
    _report("trunk n=%d fp64 cos" % n, cos, "%.5f", min)
    for k in ratios:
        assert ratios[k] <= REASSOC, (k, ratios[k])
        assert rel[k] <= 8e-2 and cos[k] >= 0.997, (k, rel[k], cos[k])


# ---- 3. backward through the heads, rows isolated ------------------------------------------------------------------

@SIZES
def test_heads_backward_at_production_size_rows_isolated(n, sms, net, net64, big, small):
    """dlogits / dvalue nonzero on S only: head_bwd_kernel at its production samples per warp and the head weight
    gradients, against the 1024-window run of obs[S] (fp32 re-association) and fp64 autograd (relative L2 <= 0.15,
    cosine >= 0.99: through the heads' ReLU bf16 flips a few masks, test_gpu_policy_train.py)."""
    _assert_reaches_production_paths(n, sms)
    obs = _windows(n, n + 2)
    S, named = boundary_windows(n, sms, seed=1)
    assert all(set(v) <= set(S.tolist()) for v in named.values())
    Sd = S.cuda()
    g = torch.Generator(device="cuda").manual_seed(8)
    dl_s = torch.randn(N_SET, 2, device="cuda", generator=g) / N_SET
    dv_s = torch.randn(N_SET, 1, device="cuda", generator=g) / N_SET
    dl, dv = torch.zeros(n, 2, device="cuda"), torch.zeros(n, 1, device="cuda")
    dl[Sd], dv[Sd] = dl_s, dv_s
    logits, value = big.logits_and_value(net, obs)
    g_big = _grads(net, [logits, value], [dl, dv])
    ls, vs = small.logits_and_value(net, obs[Sd])
    assert torch.equal(ls, logits[Sd].detach()) and torch.equal(vs, value[Sd].detach())
    g_small = _grads(net, [ls, vs], [dl_s, dv_s])
    l64, v64 = net64.logits_and_value(obs[Sd].double())
    g64 = _grads(net64, [l64, v64], [dl_s.double(), dv_s.double()])
    ratios = _reassoc_ratios(g_big, g_small)
    assert set(ratios) == set(g_big), "every parameter gets a gradient through the heads"
    rel = {k: ((g_big[k].double() - g64[k]).norm() / g64[k].norm()).item() for k in ratios}
    cos = {k: _cos(g_big[k], g64[k]) for k in ratios}
    _report("heads n=%d re-association" % n, ratios)
    _report("heads n=%d fp64 rel L2" % n, rel, "%.3f")
    _report("heads n=%d fp64 cos" % n, cos, "%.5f", min)
    for k in ratios:
        assert ratios[k] <= REASSOC, (k, ratios[k])
        assert rel[k] <= 0.15 and cos[k] >= 0.99, (k, rel[k], cos[k])


# ---- 4. PPO loss past one grid-stride pass -------------------------------------------------------------------------

EPS, C_V, C_E = 0.2, 0.5, 0.01


def _ppo_inputs(n, clipped_branch, seed):
    """fp32 inputs of uavtrain_ppo_loss that are decisive where fp32 and fp64 could decide differently: every ratio and
    every |v - old_v| at least 1e-4 from the clip edges, and the two value-loss means 1e-3 apart, with the clipped mean
    the larger one iff clipped_branch."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    f64 = torch.float64
    logits = torch.randn(n, 2, device="cuda", generator=g) * 1.5
    act = torch.randint(0, 2, (n,), device="cuda", generator=g)
    logp = torch.log_softmax(logits.double(), -1).gather(-1, act[:, None]).squeeze(-1)
    r = 0.5 + torch.rand(n, device="cuda", generator=g, dtype=f64)
    for edge in (1 - EPS, 1 + EPS):
        d = r - edge
        r = torch.where(d.abs() < 3e-4, edge + torch.where(d >= 0, 3e-4, -3e-4), r)
    old_logp = (logp - r.log()).float()
    value = torch.randn(n, device="cuda", generator=g)
    ret = torch.randn(n, device="cuda", generator=g)
    adv = torch.randn(n, device="cuda", generator=g)
    inside = torch.rand(n, device="cuda", generator=g) < 0.5
    mag = torch.where(inside, torch.rand(n, device="cuda", generator=g, dtype=f64) * (EPS - 3e-3),
                      EPS + 3e-3 + torch.rand(n, device="cuda", generator=g, dtype=f64) * 0.5)
    toward = torch.sign(ret.double() - value.double())              # old_v between v and R pulls v_clip toward R
    old_v = (value.double() + (-1.0 if clipped_branch else 1.0) * toward * mag).float()
    return logits, value, act, old_logp, adv, ret, old_v


def _ppo_reference(logits, value, act, old_logp, adv, ret, old_v):
    """agents/ppo.py:126-153 in fp64 from the fp32 inputs: (terms of the four sums, the three statistics, dlogits, dvalue)."""
    l64 = logits.double().requires_grad_()
    v64 = value.double().requires_grad_()
    old_logp, adv, ret, old_v = (t.double() for t in (old_logp, adv, ret, old_v))
    logp_all = torch.log_softmax(l64, -1)
    ratio = torch.exp(logp_all.gather(-1, act[:, None]).squeeze(-1) - old_logp)
    surr = -torch.min(ratio * adv, torch.clamp(ratio, 1 - EPS, 1 + EPS) * adv)
    vclip = old_v + torch.clamp(v64 - old_v, -EPS, EPS)
    sq1, sq2 = (v64 - ret) ** 2, (vclip - ret) ** 2
    ent = -(logp_all.exp() * logp_all).sum(-1)
    la, lc, le = surr.mean(), torch.max(sq1.mean(), sq2.mean()), ent.mean()
    (la + C_V * lc - C_E * le).backward()
    terms = [t.detach() for t in (surr, sq1, sq2, ent)]
    return terms, ratio.detach(), torch.stack([la, lc, le]).detach(), l64.grad, v64.grad


@pytest.mark.parametrize("n", [N_PROD, 300001])
@pytest.mark.parametrize("clipped_branch", [False, True])
def test_ppo_loss_kernel_past_one_grid_stride_pass(n, clipped_branch, sms):
    """uavtrain_ppo_loss at the production minibatch and at a size where ppo_loss_sums_kernel's grid-stride loop takes
    two passes.  Statistics within 1e-5 of the mean |term| of their own sum; dL/dlogits, dL/dvalue per element within
    2e-5 * max(|ref|, 1/n)."""
    import ctypes as C
    from target_allocation_ppo_transformer_b200.networks.fused_train import FusedTrunks
    if n > N_PROD:
        assert geometry(n, sms)["loss_passes"] >= 2, ("ppo_loss_sums_kernel runs one grid-stride pass", n, sms)
    inputs = _ppo_inputs(n, clipped_branch, seed=n + clipped_branch)
    logits, value, act, old_logp, adv, ret, old_v = inputs
    terms, ratio, ref, ref_dl, ref_dv = _ppo_reference(*inputs)
    edge = torch.minimum((ratio - (1 - EPS)).abs(), (ratio - (1 + EPS)).abs()).min().item()
    vedge = ((value.double() - old_v.double()).abs() - EPS).abs().min().item()
    m1, m2 = terms[1].mean().item(), terms[2].mean().item()
    assert edge >= 1e-4 and vedge >= 1e-4, (edge, vedge)
    assert (m2 > m1) == clipped_branch and abs(m2 - m1) > 1e-3 * max(m1, m2), (m1, m2)
    tr = FusedTrunks(8, "cuda")                         # the loss reads no activations: any handle serves
    p = lambda t: C.c_void_p(t.data_ptr())
    dl, dv, st = torch.empty(n, 2, device="cuda"), torch.empty(n, device="cuda"), torch.empty(3, device="cuda")
    rc = tr._lib.uavtrain_ppo_loss(tr._h, p(logits), p(value), p(act), p(old_logp), p(adv), p(ret), p(old_v), n, EPS, C_V, C_E,
                                   p(dl), p(dv), p(st), None)
    torch.cuda.synchronize()
    tr.close()
    assert rc == 0
    scales = [terms[0].abs().mean().item(), terms[2 if clipped_branch else 1].abs().mean().item(), terms[3].abs().mean().item()]
    errs = [abs(st[i].item() - ref[i].item()) / scales[i] for i in range(3)]
    floor = torch.full_like(ref_dl, 1.0 / n)
    dl_err = ((dl.double() - ref_dl).abs() / torch.maximum(ref_dl.abs(), floor)).max().item()
    dv_err = ((dv.double() - ref_dv).abs() / torch.maximum(ref_dv.abs(), floor[:, 0])).max().item()
    print("\n[ppo loss n=%d clipped=%d] statistic errors / mean|term|: %.2e %.2e %.2e; dlogits %.2e, dvalue %.2e"
          % (n, clipped_branch, *errs, dl_err, dv_err))
    assert max(errs) <= 1e-5, (errs, st.tolist(), ref.tolist())
    assert dl_err <= 2e-5 and dv_err <= 2e-5, (dl_err, dv_err)


# ---- 5. rollout forward at the evaluation / bench size -------------------------------------------------------------

@pytest.mark.parametrize("B", [65536, 65536 - 13])
def test_rollout_forward_at_65536_envs(B, net):
    """uavpolicy_get_action / uavpolicy_act at the batch DESIGN §4.5 / §4.7 quote: logits within helpers.LOGIT_TOL of
    their spread across windows and values within 3e-2 of the fp32 network; bit-identical to a 4096-env handle run over
    chunks (row-local fused kernels, same Philox key per env id); act's logits equal get_action's and its greedy actions are l1 > l0."""
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    obs = _windows(B, B)
    big_h = FusedPolicyForward(65536, "cuda", seed=5)
    big_h.sync(net)
    a, lp, v, e = (t.clone() for t in big_h.get_action(obs, step=4))
    logits = big_h.logits[:B].clone()
    with torch.no_grad():
        ref_l, ref_v = net.logits_and_value(obs)
    assert_logits_close(logits, ref_l, net)
    assert float((v - ref_v).abs().max()) < 3e-2 * max(1.0, float(ref_v.abs().max()))
    ga, glp = (t.clone() for t in big_h.act(obs, step=4, greedy=True))
    assert torch.equal(big_h.logits[:B], logits)
    assert torch.equal(ga, (logits[:, 1] > logits[:, 0]).long())
    sa, slp = big_h.act(obs, step=4, greedy=False)
    assert torch.equal(big_h.logits[:B], logits) and torch.equal(sa, a) and torch.equal(slp, lp)
    big_h.close()
    small_h = FusedPolicyForward(CHUNK_CAP, "cuda", seed=5)
    small_h.sync(net)
    for i in range(0, B, CHUNK):
        small_h.env_id_base = i                          # the same env ids, so the same Philox draws
        ca, clp, cv, ce = small_h.get_action(obs[i:i + CHUNK], step=4)
        m = ca.shape[0]
        assert torch.equal(small_h.logits[:m], logits[i:i + m]) and torch.equal(cv, v[i:i + m]), i
        assert torch.equal(ca, a[i:i + m]) and torch.equal(clp, lp[i:i + m]) and torch.equal(ce, e[i:i + m]), i
    small_h.close()
