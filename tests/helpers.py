"""Shared helpers of the parity tests."""
import hashlib
import os

import numpy as np

from conftest import GOLDEN

CFG_INT = {"NUM_UAVS", "NUM_TARGETS", "NUM_NFZ", "NUM_INTERCEPTORS"}


def load_fixture(case):
    """A recorded trajectory as a dict.  A fixture too large to store its p_final matrix (traj_n256m256_s0) gets it
    back as p_damage * p_pen[:, None], the product the reference forms (bit-exact in every fixture that stores both)."""
    fx = dict(np.load(os.path.join(GOLDEN, case + ".npz")))
    if "p_final" not in fx:
        fx["p_final"] = fx["p_damage"] * fx["p_pen"][:, None]
    return fx


def _encoder_weight_draws(seed):
    """The reference network's construction replayed on torch's global generator seeded with `seed`: per block a
    Linear(14,128) with orthogonal init, the learned positions, then ONE nn.TransformerEncoderLayer that
    nn.TransformerEncoder deep-copies into every layer of the block; the actor head (two orthogonal Linears) sits
    between the two blocks.  Returns the layers' state_dict entries by full name."""
    import math

    import torch
    import torch.nn as nn
    drawn = {}
    with torch.random.fork_rng(devices=[]):          # the caller's generator state is left as it was
        torch.random.default_generator.manual_seed(seed)
        for block, layers in (("actor_net", 1), ("critic_net", 2)):
            nn.init.orthogonal_(nn.Linear(14, 128).weight, math.sqrt(2.0))
            torch.randn(1, 5, 128)
            layer = nn.TransformerEncoderLayer(128, 8, 256, dropout=0.0, batch_first=True).state_dict()
            for i in range(layers):
                drawn.update({"%s.transformer.layers.%d.%s" % (block, i, k): v.numpy() for k, v in layer.items()})
            if block == "actor_net":
                nn.init.orthogonal_(nn.Linear(128, 64).weight, math.sqrt(2.0))
                nn.init.orthogonal_(nn.Linear(64, 2).weight, 0.01)
    return drawn


def policy_fixture():
    """tests/golden/policy_net.npz and the reference network's state_dict it records (numpy, in state_dict order).
    The encoder layers' uniform-initialised weights (393k of the 419k values) are not stored: they are drawn again
    from the recorded seed and must match the recorded SHA-256 of each tensor's bytes.  Everything that went through a
    QR factorisation or torch's vectorised normal sampler, and the perturbed 1-D parameters, is stored as is."""
    fx = np.load(os.path.join(GOLDEN, "policy_net.npz"))
    drawn = None
    sd = {}
    for k in map(str, fx["keys"]):
        if "p::" + k in fx:
            sd[k] = fx["p::" + k]
            continue
        if drawn is None:
            drawn = _encoder_weight_draws(int(fx["init_seed"]))
        sd[k] = drawn[k]
        assert hashlib.sha256(sd[k].tobytes()).hexdigest() == str(fx["sha256::" + k]), \
            "%s drawn from seed %d differs from the recorded weights" % (k, int(fx["init_seed"]))
    return fx, sd


def config_from_fixture(fx, **extra):
    """Product-side Config carrying the cfg overrides the reference ran the fixture with."""
    import uavenv_b200 as ub
    kw = {}
    for n, v in zip(fx["cfg_names"], fx["cfg_values"]):
        n = str(n)
        if n in ("UAV_GEN_X_RANGE", "TARGET_GEN_X_RANGE"):
            continue
        kw[n] = int(v) if n in CFG_INT else float(v)
    kw["UAV_GEN_X_RANGE"] = tuple(float(x) for x in fx["cfg_uav_gen_x"])
    kw["TARGET_GEN_X_RANGE"] = tuple(float(x) for x in fx["cfg_target_gen_x"])
    kw.update(extra)
    return ub.Config(**kw)


def oracle_cfg_from_config(cfg):
    from oracle import oracle as orc
    return orc.make_cfg(**{k: v for k, v in cfg.as_dict().items() if k in (
        "NUM_UAVS", "NUM_TARGETS", "NUM_NFZ", "NUM_INTERCEPTORS", "PARAM_ZETA_D", "PARAM_K", "PARAM_C1", "PARAM_C2",
        "PARAM_C3", "PARAM_C4", "COST_WEIGHT_OMEGA", "WEATHER_SPEED_FACTOR", "WEATHER_LOAD_FACTOR", "MAP_WIDTH",
        "MAP_HEIGHT", "INTERCEPT_RAD", "UAV_GEN_X_RANGE", "TARGET_GEN_X_RANGE")})


SCENE_KEYS = ["uav_x", "uav_y", "uav_vx", "uav_vy", "uav_load", "uav_cost", "uav_type", "tgt_x", "tgt_y", "tgt_vx",
              "tgt_vy", "tgt_value", "tgt_id", "nfz_x", "nfz_y", "nfz_radius", "int_x", "int_y", "int_vx", "int_vy"]


def scene_from_fixture(fx, copies=1):
    return {k: np.tile(np.asarray(fx[k]), (copies, 1)) for k in SCENE_KEYS}


LOGIT_TOL = 0.1     # of the spread of the logits (log-probs) across windows


def logit_spread(net, logprobs=False):
    """The smallest standard deviation across windows of a column of the actor's logits (or log-probs), fp32 network, over
    4096 seeded random windows with 0..4 leading zero rows.  The actor's last layer is initialised with std 0.01, so the
    logits of a young network differ across windows by a few 1e-3: an absolute tolerance of 1e-2 on them passes even an
    actor whose trunk output is zero."""
    import torch
    g = torch.Generator().manual_seed(0)
    obs = torch.rand(4096, 5, 14, generator=g)
    obs[:, :, 13] = 1.0
    obs[torch.arange(5)[None, :] < (torch.arange(4096) % 5)[:, None]] = 0.0
    with torch.no_grad():
        logits = net.actor_head(net.actor_net.forward_last(obs.to(next(net.parameters()).device)))
    return float((torch.log_softmax(logits, -1) if logprobs else logits).std(0).min())


def logits_close(got, ref, net, logprobs=False):
    """(ok, error): the largest |got - ref| in units of logit_spread(net) is at most LOGIT_TOL."""
    err = float((got.double() - ref.double()).abs().max()) / logit_spread(net, logprobs)
    return err <= LOGIT_TOL, err


def assert_logits_close(got, ref, net, logprobs=False, note=""):
    ok, err = logits_close(got, ref, net, logprobs)
    print("\n[logits_close%s] %.3f of the spread" % (note, err))
    assert ok, ("max |error| is %.3f of the spread across windows, above %g" % (err, LOGIT_TOL), note)


def rel_close(got, want, rtol, atol=0.0):
    np.testing.assert_allclose(np.asarray(got, np.float64), np.asarray(want, np.float64), rtol=rtol, atol=atol)
