"""The fused rollout forward (csrc/policy_fused.cu) feature by feature: the trunk output z of the last token and the head's
hidden layer of both networks, read out of the kernels exactly and compared with the mirror network in fp64.

Why not the logits: the actor head's last layer is initialised with std 0.01 (networks/transformer_net.py:146-147), so the
logits of the golden network vary across windows by ~4e-3 and barely depend on the trunk. Replacing the actor's trunk
output by zeros moves them by 1.1e-2; a tolerance on them cannot see the actor's half of the kernels.

Readout.  The kernels write relu(W1 z + b1) as bf16 [B, 64] per network, and heads_out_kernel forms W2 h + b2 in fp32.
With b2 = 0 and unit rows in W2 the public logits / value ARE the stored bf16 hidden units (64 forwards read all of them);
with W1 = s [I_64 | 0] or s [0 | I_64] (s = +-1, exact in bf16) and b1 = 0 the hidden units are relu(+-z_i), and four such
passes give z = pos - neg exactly (256 forwards).  The readout checks its own premises: every value is bf16-representable,
and at most one of pos / neg is nonzero.

Reference: the mirror network in fp64, with the weights the kernels consume in bf16 rounded to bf16 first (the embedding
weight, in_proj, out_proj, linear1, linear2, head W1: kGemmW / emb_w2p of policy_weights.cuh); positions, LayerNorm
parameters and biases at their fp32 values (the kernels carry biases and observations as bf16 hi + lo).  What remains is
the kernels' bf16 rounding of activations, which is zero-mean noise.  Checks on z of each network: (a) max abs error,
(b) largest per-window relative L2 error, (c) largest |per-feature mean error| over >= 4096 windows, which sees
systematic errors that are too small for (a) (a dropped position row, a lost bias remainder).

Measured on a B200 (148 SMs, power limit 1000 W) over every case below (15 batch sizes, golden / perturbed /
large-bias weights, mixed and UAVEnvBatched windows), worst values: (a) 0.0625 (critic; actor 0.047), (b) 0.0074,
(c) 2.6e-3 (critic; actor 2.3e-3).  TOL_* are at most twice these.  Mutant references (one parameter- or mask-level
change of the fp64 reference each) must all be rejected by the same checks: the closest calls are a dropped position
row 0 (actor: (b) 0.0175, (c) 5.0e-3) and dropped bias remainders on the large-bias network ((c) 5.1e-3 actor, 5.8e-3
critic).  Runtime of the file on a B200: 11 s."""
import pytest
import torch
import torch.nn.functional as F

from helpers import policy_fixture

import uavenv_b200 as ub

TOL_ABS = 0.1       # (a)  measured worst 0.0625 (critic; 0.047 actor)
TOL_REL = 0.011     # (b)  measured worst 0.0074
TOL_MEAN = 3.5e-3   # (c)  measured worst 2.6e-3
MEAN_MIN_WINDOWS = 4096

GEMM_WEIGHTS = ("embedding.0.weight", "self_attn.in_proj_weight", "self_attn.out_proj.weight", "linear1.weight",
                "linear2.weight")
BIASES = ("embedding.0.bias", "in_proj_bias", "out_proj.bias", "linear1.bias", "linear2.bias")


# ---- fp64 reference -------------------------------------------------------------------------------------------------

def reference_params(sd, net):
    """fp64 parameters of one network ("actor" / "critic") as the kernels consume them: trunk tensors by their name under
    <net>_net., and the head's W1 / b1 / W2 / b2."""
    pre, head = net + "_net.", net + "_head."
    P = {}
    for k, v in sd.items():
        v = torch.as_tensor(v).detach()
        if k.startswith(pre):
            k = k[len(pre):]
            P[k] = (v.bfloat16() if k.endswith(GEMM_WEIGHTS) else v).double()
    P["head.w1"] = torch.as_tensor(sd[head + "0.weight"]).detach().bfloat16().double()
    P["head.b1"] = torch.as_tensor(sd[head + "0.bias"]).detach().double()
    P["head.w2"] = torch.as_tensor(sd[head + "2.weight"]).detach().double()
    P["head.b2"] = torch.as_tensor(sd[head + "2.bias"]).detach().double()
    return P


def num_layers(P):
    return sum(1 for k in P if k.endswith("norm2.weight"))


def trunk64(P, obs, mask="zero rows", swap_keys=None):
    """Last-token trunk output [B, 128] of one network in fp64 (networks/transformer_net.py: embedding + positions, post-LN
    encoder layers with the key-padding mask of all-zero rows, the newest row never masked).  Mutations for the detection
    checks: mask = "none" (no key is masked) or "leading" (only the leading run of zero rows); swap_keys = (i, j) swaps
    the keys of tokens i and j in the last layer while their values stay in place."""
    x = obs.double()
    pad = x.abs().sum(-1) == 0
    if mask == "leading":
        pad = pad.cumprod(1).bool()
    pad[:, -1] = False
    if mask == "none":
        pad[:] = False
    h = torch.relu(x @ P["embedding.0.weight"].T + P["embedding.0.bias"]) + P["pos_embedding"][0]
    L = num_layers(P)
    for l in range(L):
        p, last = "transformer.layers.%d." % l, l == L - 1
        q, k, v = (h @ P[p + "self_attn.in_proj_weight"].T + P[p + "self_attn.in_proj_bias"]).split(128, -1)
        if last:
            q = q[:, -1:]
            if swap_keys:
                k = k.clone()
                k[:, list(swap_keys)] = k[:, list(swap_keys[::-1])]
        q, k, v = (t.unflatten(-1, (8, 16)).transpose(1, 2) for t in (q, k, v))
        s = (q @ k.transpose(-1, -2) / 4.0).masked_fill(pad[:, None, None, :], float("-inf"))
        a = (torch.softmax(s, -1) @ v).transpose(1, 2).flatten(2)
        res = h[:, -1:] if last else h
        y = F.layer_norm(res + a @ P[p + "self_attn.out_proj.weight"].T + P[p + "self_attn.out_proj.bias"], (128,),
                         P[p + "norm1.weight"], P[p + "norm1.bias"])
        f = torch.relu(y @ P[p + "linear1.weight"].T + P[p + "linear1.bias"])
        h = F.layer_norm(y + f @ P[p + "linear2.weight"].T + P[p + "linear2.bias"], (128,), P[p + "norm2.weight"],
                         P[p + "norm2.bias"])
    return h[:, 0]


def metrics(z, z_ref):
    """(a) max abs error, (b) max per-window relative L2 error, (c) max |per-feature mean error| (None below 4096 windows).
    The kernels store z in bf16, so the reference is rounded to bf16 too: a feature that is nearly constant across windows
    would otherwise carry its rounding error into (c) as a bias of up to half a bf16 ulp."""
    e = z - z_ref.float().bfloat16().double()
    return (float(e.abs().max()), float((e.norm(dim=1) / z_ref.norm(dim=1)).max()),
            float(e.mean(0).abs().max()) if z.shape[0] >= MEAN_MIN_WINDOWS else None)


def within(m):
    return m[0] <= TOL_ABS and m[1] <= TOL_REL and (m[2] is None or m[2] <= TOL_MEAN)


# ---- weights and windows ----------------------------------------------------------------------------------------------

def state_dict(kind):
    """'golden': tests/golden/policy_net.npz; 'perturbed': LayerNorm gamma 1 +- 0.5, beta +- 0.5; 'large_bias': every
    bias of the trunks and of the head's first layer uniform in +-4."""
    sd = {k: torch.from_numpy(v.copy()) for k, v in policy_fixture()[1].items()}
    g = torch.Generator().manual_seed({"golden": 0, "perturbed": 1, "large_bias": 2}[kind])
    for k, v in sd.items():
        u = torch.rand(v.shape, generator=g, dtype=torch.float64) * 2 - 1
        if kind == "perturbed" and ".norm" in k:
            sd[k] = (1.0 + 0.5 * u if k.endswith("weight") else 0.5 * u).float()
        if kind == "large_bias" and (k.endswith(BIASES) or k.endswith("_head.0.bias")):
            sd[k] = (4.0 * u).float()
    return sd


def module(sd):
    net = ub.TransformerActorCritic().cuda()
    net.load_state_dict(sd)
    return net.eval()


def mixed_windows(B, seed, big=10.0):
    """Random windows with 0..4 leading zero rows; window b also gets, by (b // 5) % 8: nothing more, an interior zero row
    (masked by the reference too, transformer_net.py:125), -0.0 rows, a zero newest row (never masked), all zeros, rows
    whose only nonzero entry is 1e-30 / a denormal, entries up to +-`big` (the hi + lo split of the observation)."""
    g = torch.Generator().manual_seed(seed)
    obs = torch.rand(B, 5, 14, generator=g)
    obs[:, :, 13] = 1.0
    b = torch.arange(B)
    lead = b % 5
    obs[torch.arange(5)[None, :] < lead[:, None]] = 0.0
    kind = (b // 5) % 8
    inner = kind == 1                                       # one zero row after the leading run, before the newest
    tok = torch.clamp(lead + 1 + (b // 40) % 2, max=3)
    obs[inner, tok[inner]] = 0.0
    neg = kind == 2
    obs[neg, : 4] = torch.where(obs[neg, :4] == 0, -0.0, obs[neg, :4])
    obs[neg, 2] = -0.0
    obs[kind == 3, 4] = 0.0
    obs[kind == 4] = 0.0
    tiny = kind == 5
    obs[tiny, 1:3] = 0.0
    obs[tiny, 1, 5] = 1e-30
    obs[tiny, 2, 0] = 1e-40                                 # fp32 denormal
    band = kind == 6
    obs[band] = (torch.rand(int(band.sum()), 5, 14, generator=g) * 2 - 1) * big
    assert ((obs[tiny, 2, 0] > 0) & (obs[tiny, 2, 0] < torch.finfo(torch.float32).tiny)).all()
    return obs


def env_windows(B, steps=12):
    """Observation windows of UAVEnvBatched itself after `steps` random steps (episode starts included)."""
    env = ub.UAVEnvBatched(B, device="cuda", seed=7)
    obs = env.reset(full_reset=True)
    g = torch.Generator(device="cuda").manual_seed(3)
    for _ in range(steps):
        obs, _, _, _ = env.step(torch.randint(0, 2, (B,), device="cuda", generator=g))
    obs = obs.clone().cpu()
    env.close()
    return obs


# ---- launch geometry (launch_fused_blocks) --------------------------------------------------------------------------

def _cdiv(a, b):
    return -(-a // b)


def geometry(B, sms):
    """(work items, CTAs) of the two fused launches: phase 0 = (network, tile of 25 samples), phase 1 = (network, 128
    samples), each on min(items, SMs) persistent CTAs."""
    i0, i1 = 2 * _cdiv(B, 25), 2 * _cdiv(B, 128)
    return (i0, min(i0, sms)), (i1, min(i1, sms))


SIZE_LABELS = ["1", "24", "25", "26", "127", "128", "129", "150", "phase0 items = SMs", "phase0 items = SMs + 1",
               "phase1 items = SMs", "phase1 items = SMs + 1", "16384", "65535", "65536"]


def size_of(label, sms):
    """A label of SIZE_LABELS as a batch size on a device with `sms` SMs; the SM-count crossings are checked here."""
    if not label.startswith("phase"):
        return int(label)
    phase, per = (0, 25) if label.startswith("phase0") else (1, 128)
    B = per * (sms // 2)                                   # the largest batch whose items fit the SMs
    (g0, g1) = geometry(B, sms), geometry(B + 1, sms)
    assert g0[phase][0] <= sms < g1[phase][0] and g1[phase][1] == sms, (label, sms, g0, g1)
    return B + 1 if label.endswith("+ 1") else B


def test_sizes_cross_the_launch_boundaries():
    sms = torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148
    (t25, _), (g25, _) = geometry(25, sms)
    assert geometry(24, sms)[0][0] == t25 == 2 and geometry(26, sms)[0][0] == 4      # one tile, then a second
    assert geometry(128, sms)[1][0] == 2 and geometry(129, sms)[1][0] == 4            # one 128-sample group, then two
    assert 125 < 128 < 150                                   # 150: the tile of samples 125..149 straddles group 0 / 1
    sizes = [size_of(lb, sms) for lb in SIZE_LABELS]
    if sms == 148:
        assert sizes[8:12] == [1850, 1851, 9472, 9473]
    for B in (16384, 65535, 65536):
        assert all(g[0] > sms for g in geometry(B, sms))    # several items per persistent CTA in both launches


def test_reference_equals_the_fp32_mirror_network():
    """The fp64 reference without its bf16 weight rounding is the mirror network's forward_last (CPU, fp32)."""
    sd = state_dict("golden")
    net = ub.TransformerActorCritic()
    net.load_state_dict(sd)
    obs = mixed_windows(500, 3)
    with torch.no_grad():
        for name, blk in (("actor", net.actor_net), ("critic", net.critic_net)):
            P = reference_params(sd, name)
            P.update({k[len(name) + 5:]: v.double() for k, v in sd.items() if k.startswith(name + "_net.")})
            err = (trunk64(P, obs) - blk.forward_last(obs).double()).abs().max()
            assert float(err) < 1e-4, (name, float(err))


# ---- the readout ------------------------------------------------------------------------------------------------------

class Readout:
    """Kernel intermediates through the public get_action outputs of one FusedPolicyForward handle (see the module doc)."""

    def __init__(self, fused, sd):
        self.fused, self.net = fused, module(sd)

    def _rows(self, obs):
        """The bf16 head-hidden rows of both networks, [B, 64] fp64 each, for the W1 / b1 currently in self.net."""
        B, f = obs.shape[0], self.fused
        ah, ch = self.net.actor_head[2], self.net.critic_head[2]
        ha = torch.empty(B, 64, dtype=torch.float64, device="cuda")
        hc = torch.empty_like(ha)
        with torch.no_grad():
            ah.bias.zero_(); ch.bias.zero_()
            for k in range(64):
                ah.weight.zero_(); ch.weight.zero_()
                ch.weight[0, k] = 1.0
                if k < 32:
                    ah.weight[0, 2 * k] = 1.0; ah.weight[1, 2 * k + 1] = 1.0
                f.sync(self.net)
                v = f.get_action(obs, 0)[2]
                hc[:, k] = v[:, 0].double()
                if k < 32:
                    ha[:, 2 * k: 2 * k + 2] = f.logits[:B].double()
        for h in (ha, hc):
            assert torch.isfinite(h).all() and (h >= 0).all()
            assert torch.equal(h.float().bfloat16().double(), h), "a read-out value is not a bf16 number"
        return ha, hc

    def hidden(self, obs, sd):
        """relu(W1 z + b1) of both networks with the real W1 / b1."""
        with torch.no_grad():
            for net in ("actor", "critic"):
                head = getattr(self.net, net + "_head")[0]
                head.weight.copy_(sd[net + "_head.0.weight"]); head.bias.copy_(sd[net + "_head.0.bias"])
        return self._rows(obs)

    def trunk(self, obs):
        """The last-token trunk output z of both networks (bf16 values as fp64), from four passes W1 = s [I | 0], s [0 | I]."""
        B = obs.shape[0]
        z = {"actor": torch.zeros(B, 128, dtype=torch.float64, device="cuda")}
        z["critic"] = torch.zeros_like(z["actor"])
        for half in (0, 1):
            parts = {}
            for s in (1.0, -1.0):
                with torch.no_grad():
                    for net in ("actor", "critic"):
                        head = getattr(self.net, net + "_head")[0]
                        head.weight.zero_(); head.bias.zero_()
                        head.weight[:, 64 * half: 64 * half + 64] = s * torch.eye(64, device="cuda")
                parts[s] = self._rows(obs)
            for i, net in enumerate(("actor", "critic")):
                pos, neg = parts[1.0][i], parts[-1.0][i]
                assert not ((pos != 0) & (neg != 0)).any(), "relu(z) and relu(-z) both nonzero"
                z[net][:, 64 * half: 64 * half + 64] = pos - neg
        return z


@pytest.fixture(scope="module")
def fused():
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    f = FusedPolicyForward(65536, "cuda", seed=1)
    yield f
    f.close()


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


_CACHE = {}


def read_case(fused, weights, windows, B):
    """(state_dict, obs on the GPU, z read out, head-hidden rows read out), cached per case for the module."""
    key = (weights, windows, B)
    if key not in _CACHE:
        sd = state_dict(weights)
        obs = (mixed_windows(B, B) if windows == "mixed" else env_windows(B)).cuda()
        r = Readout(fused, sd)
        _CACHE[key] = (sd, obs, r.trunk(obs), r.hidden(obs, sd))
    return _CACHE[key]


CASES = [("golden", "mixed", lb) for lb in SIZE_LABELS] + \
        [("perturbed", "mixed", "16384"), ("large_bias", "mixed", "16384"), ("golden", "env", "16384")]


@pytest.mark.gpu
@pytest.mark.parametrize("weights,windows,size", CASES, ids=["%s-%s-%s" % c for c in CASES])
def test_trunk_and_head_hidden_match_fp64(fused, sms, weights, windows, size):
    B = size_of(size, sms)
    sd, obs, z, h = read_case(fused, weights, windows, B)
    for i, net in enumerate(("actor", "critic")):
        P = {k: v.cuda() for k, v in reference_params(sd, net).items()}
        m = metrics(z[net], trunk64(P, obs))
        print("\n[readout %s %s B=%d %s] max abs %.4g  max rel-L2 %.4g  max |feature mean| %s"
              % (weights, windows, B, net, m[0], m[1], "%.3g" % m[2] if m[2] is not None else "-"))
        assert within(m), (net, m)
        # the head's first layer on the kernel's own z: within one bf16 ulp of relu(bf16(W1) z + b1) (+ fp32 sums)
        pre = z[net] @ P["head.w1"].T + P["head.b1"]
        want = torch.relu(pre)
        ulp = torch.pow(2.0, torch.floor(torch.log2(want.clamp_min(2.0 ** -126))) - 7)
        slack = 1e-6 * (z[net].abs() @ P["head.w1"].abs().T + P["head.b1"].abs())
        assert ((h[i] - want).abs() <= ulp + slack).all(), (net, float((h[i] - want).abs().max()))


@pytest.mark.gpu
@pytest.mark.parametrize("weights", ["golden", "large_bias"])
def test_real_second_head_layer_and_softmax(fused, weights):
    """With the real W2 / b2 the logits and value are fp64 W2 h + b2 of the read-out h to fp32 rounding; with an actor W2 that
    makes the logit gaps reach +-40, log-probs and entropy are fp64 log_softmax of the kernel's own logits, all finite."""
    B = 16384
    sd, obs, _, (ha, hc) = read_case(fused, weights, "mixed", B)
    net = module(sd)
    fused.sync(net)
    a, lp, v, e = (t.clone() for t in fused.get_action(obs, step=2))
    logits = fused.logits[:B].double()
    for got, h, w2, b2 in ((logits, ha, sd["actor_head.2.weight"], sd["actor_head.2.bias"]),
                           (v.double(), hc, sd["critic_head.2.weight"], sd["critic_head.2.bias"])):
        w2, b2 = w2.cuda().double(), b2.cuda().double()
        want = h @ w2.T + b2
        assert ((got - want).abs() <= 1e-6 * (h @ w2.abs().T + b2.abs()) + 1e-30).all(), float((got - want).abs().max())
    # logit gaps up to +-40: W2 rows +-w with w chosen from the read-out hidden rows
    g = torch.Generator(device="cuda").manual_seed(4)
    w = torch.randn(64, device="cuda", dtype=torch.float64, generator=g)
    m = (ha @ w).median()                                   # logits +-(w h - m): gaps of both signs
    c = 20.0 / float((ha @ w - m).abs().max())
    with torch.no_grad():
        net.actor_head[2].weight.copy_(torch.stack([c * w, -c * w]).float())
        net.actor_head[2].bias.copy_(torch.stack([-c * m, c * m]).float())
    fused.sync(net)
    for greedy in (None, True, False):
        if greedy is None:
            a, lp, _, e = fused.get_action(obs, step=3)
        else:
            a, lp = fused.act(obs, step=3, greedy=greedy)
        logits = fused.logits[:B].double()
        gap = logits[:, 0] - logits[:, 1]
        assert float(gap.abs().max()) > 39.0 and float(gap.max()) > 0 > float(gap.min())
        ref = torch.log_softmax(logits, -1)
        assert torch.isfinite(lp).all() and torch.isfinite(logits).all()
        ref_lp = ref.gather(-1, a[:, None]).squeeze(-1)
        assert ((lp.double() - ref_lp).abs() <= 2e-5 + 1e-6 * ref_lp.abs()).all(), float((lp.double() - ref_lp).abs().max())
        if greedy:
            assert torch.equal(a, (logits[:, 1] > logits[:, 0]).long())
        else:
            assert set(a.tolist()) == {0, 1} and float(lp.min()) < -1.0      # the less likely action is drawn too
        if greedy is None:
            ref_e = -(ref.exp() * ref).sum(-1)
            assert torch.isfinite(e).all() and ((e.double() - ref_e).abs() <= 1e-6).all(), float((e.double() - ref_e).abs().max())


@pytest.mark.gpu
def test_observations_up_to_1e3(fused):
    """Entries up to +-1e3 on every row.  At that scale the attention of some windows is so saturated that rounding the
    reference's own weights to bf16 moves z by up to 30 %, and the kernels' bf16 activations move it as much (measured
    0.27 relative L2 even on windows the weight rounding leaves alone): (a) and (b) cannot be held there.  z must be finite,
    and (c) must hold over the windows whose reference moves by less than 5e-3 under the weight rounding (measured
    5.4e-4); the trunk is checked per window at entries up to +-10 in the other tests."""
    B = 8192
    g = torch.Generator().manual_seed(8)
    obs = (torch.rand(B, 5, 14, generator=g) * 2 - 1) * 1e3
    obs[torch.arange(5)[None, :] < (torch.arange(B) % 5)[:, None]] = 0.0
    sd = state_dict("golden")
    obs = obs.cuda()
    z = Readout(fused, sd).trunk(obs)
    for net in ("actor", "critic"):
        assert torch.isfinite(z[net]).all()
        P = {k: v.cuda() for k, v in reference_params(sd, net).items()}
        P32 = dict(P, **{k[len(net) + 5:]: v.cuda().double() for k, v in sd.items() if k.startswith(net + "_net.")})
        ref, ref32 = trunk64(P, obs), trunk64(P32, obs)
        stable = (ref - ref32).norm(dim=1) / ref32.norm(dim=1) < 5e-3
        m = metrics(z[net][stable], ref[stable])
        print("\n[readout golden +-1e3 B=%d %s] %d well-conditioned windows: max abs %.4g  max rel-L2 %.4g  max |feature mean| %s"
              % (B, net, int(stable.sum()), m[0], m[1], m[2]))
        assert int(stable.sum()) > 0.8 * B and m[2] <= TOL_MEAN, (net, int(stable.sum()), m)


# ---- detection power --------------------------------------------------------------------------------------------------

def _drop_v(l, h=7):
    def f(P):
        for k in ("self_attn.in_proj_weight", "self_attn.in_proj_bias"):
            P["transformer.layers.%d.%s" % (l, k)][256 + 16 * h: 272 + 16 * h] = 0.0
    return f


def _zero(key, index=()):
    def f(P):
        P[key][index] = 0.0
    return f


def _bf16_biases(P):
    for k in P:
        if k.endswith(BIASES):
            P[k] = P[k].float().bfloat16().double()


# (name, network, weights, change of P, trunk64 keyword arguments)
MUTANTS = [("head 7 V dropped, layer 0", "actor", "golden", _drop_v(0), {}),
           ("head 7 V dropped, layer 0", "critic", "golden", _drop_v(0), {}),
           ("head 7 V dropped, layer 1", "critic", "golden", _drop_v(1), {})]
for _net, _last in (("actor", 0), ("critic", 1)):
    MUTANTS += [("position row 0 dropped", _net, "golden", _zero("pos_embedding", (0, 0)), {}),
                ("position row 4 dropped", _net, "golden", _zero("pos_embedding", (0, 4)), {}),
                ("last LayerNorm beta dropped", _net, "golden", _zero("transformer.layers.%d.norm2.bias" % _last), {}),
                ("padding mask ignored", _net, "golden", None, {"mask": "none"}),
                ("only leading zero rows masked", _net, "golden", None, {"mask": "leading"}),
                ("keys of tokens 3 and 4 swapped", _net, "golden", None, {"swap_keys": (3, 4)}),
                ("bias remainders dropped", _net, "large_bias", _bf16_biases, {})]
MUTANTS += [("FFN unit 255 of the last layer dropped", "critic", "golden",
             lambda P: (_zero("transformer.layers.1.linear1.weight", 255)(P), _zero("transformer.layers.1.linear1.bias", 255)(P)), {})]


@pytest.mark.gpu
@pytest.mark.parametrize("name,net,weights,change,kw", MUTANTS, ids=["%s-%s" % (m[1], m[0]) for m in MUTANTS])
def test_checks_reject_mutant_references(fused, name, net, weights, change, kw):
    """The kernel's z passes against the clean reference and fails (a), (b) or (c) against each mutant reference."""
    sd, obs, z, _ = read_case(fused, weights, "mixed", 16384)
    P = {k: v.cuda() for k, v in reference_params(sd, net).items()}
    clean = metrics(z[net], trunk64(P, obs))
    if change:
        change(P)
    m = metrics(z[net], trunk64(P, obs, **kw))
    print("\n[mutant %s %s] clean %s  mutant %s" % (net, name, clean, m))
    assert within(clean) and not within(m), (clean, m)


def test_zero_actor_trunk_fails_the_logit_checks():
    """helpers.logits_close, the logit / log-prob check of test_gpu_policy_forward, test_gpu_evaluate,
    test_gpu_update_geometry and test_gpu_ppo, rejects an actor whose trunk output is zero on their kinds of windows (the
    absolute 3e-2 it replaced did not: the zero trunk moves the golden network's logits by 1.1e-2)."""
    from helpers import logits_close
    sd = state_dict("golden")
    net = ub.TransformerActorCritic()
    net.load_state_dict(sd)
    fx = policy_fixture()[0]
    g = torch.Generator().manual_seed(5)
    plain = torch.rand(384, 5, 14, generator=g)
    sets = [torch.from_numpy(fx["obs"]), plain, mixed_windows(1000, 1), mixed_windows(16384, 2)]
    with torch.no_grad():
        for obs in sets:
            ref, _ = net.logits_and_value(obs)
            zero = net.actor_head(torch.zeros(obs.shape[0], 128))
            assert logits_close(ref + 1e-4, ref, net)[0]
            assert not logits_close(zero, ref, net)[0]
            lp_ref, lp_zero = torch.log_softmax(ref, -1), torch.log_softmax(zero, -1)
            a = torch.arange(obs.shape[0])[:, None] % 2
            assert not logits_close(lp_zero.gather(-1, a), lp_ref.gather(-1, a), net, logprobs=True)[0]
