"""tcgen05 rollout forward (csrc/policy_forward.cu) against the fp32 PyTorch network with the reference's weights
(tests/golden/policy_net.npz).  bf16 operands: logits and log-probs within helpers.LOGIT_TOL of their spread across
windows (the actor's last layer has std 0.01: an absolute tolerance would pass a zero actor trunk), values within 3e-2;
sampling follows the returned probabilities; the library has no CPU fallback."""
import numpy as np
import pytest
import torch

from helpers import assert_logits_close, policy_fixture

import uavenv_b200  # noqa: F401  (registers the package under an importable name)

pytestmark = pytest.mark.gpu


def _net():
    import uavenv_b200 as ub
    fx, sd = policy_fixture()
    net = ub.TransformerActorCritic().cuda()
    net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    return net.eval(), fx


def test_handwritten_tcgen05_gemm_tile_selftest():
    """The hand-written UMMA path on its own: descriptors, canonical operand layout, TMEM lane mapping."""
    import ctypes as C
    from target_allocation_ppo_transformer_b200 import _capi
    L = _capi.load_policy()
    torch.manual_seed(0)
    for N, K in ((128, 128), (384, 128), (128, 256), (64, 128)):
        A = torch.randn(128, K, device="cuda").bfloat16()
        W = (torch.randn(N, K, device="cuda") * 0.2).bfloat16()
        Dst = torch.zeros(128, N, device="cuda")
        assert L.uavpolicy_selftest_gemm_tile(C.c_void_p(A.data_ptr()), C.c_void_p(W.data_ptr()), C.c_void_p(Dst.data_ptr()),
                                              N, K, None) == 0
        torch.cuda.synchronize()
        assert float((Dst - A.float() @ W.float().t()).abs().max()) < 1e-4


def test_forward_matches_fp32_network_and_reference_golden():
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    net, fx = _net()
    obs = torch.from_numpy(fx["obs"]).cuda()
    fused = FusedPolicyForward(256, "cuda")
    fused.sync(net)
    a, lp, v, e = fused.get_action(obs, step=0)
    logits = fused.logits[: obs.shape[0]]
    with torch.no_grad():
        ref_logits, ref_v = net.logits_and_value(obs)
    assert_logits_close(logits, ref_logits, net)
    assert float((v - ref_v).abs().max()) < 3e-2 * max(1.0, float(ref_v.abs().max()))
    # against the values recorded from the UNMODIFIED reference network
    assert_logits_close(logits.cpu(), torch.from_numpy(fx["logits"]), net)
    assert float((v.cpu() - torch.from_numpy(fx["value"])).abs().max()) < 3e-2 * max(1.0, float(np.abs(fx["value"]).max()))
    ref_lp = torch.log_softmax(ref_logits, -1).gather(-1, a[:, None]).squeeze(-1)
    assert_logits_close(lp, ref_lp, net, logprobs=True)
    p = torch.softmax(logits, -1)
    assert torch.allclose(e, -(p * p.log()).sum(-1), atol=1e-5)
    assert set(a.tolist()) <= {0, 1}
    fused.close()


def test_padding_rows_and_batch_tails():
    """Episode starts (leading zero rows are masked keys) and batch sizes that are not tile multiples."""
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    net, _ = _net()
    fused = FusedPolicyForward(1000, "cuda")
    fused.sync(net)
    g = torch.Generator(device="cuda").manual_seed(1)
    for B in (1, 7, 24, 26, 129, 1000):
        obs = torch.rand(B, 5, 14, device="cuda", generator=g)
        obs[:, :, 13] = 1.0
        for b in range(B):
            obs[b, : b % 5] = 0.0
        _, _, v, _ = fused.get_action(obs, step=3)
        with torch.no_grad():
            ref_logits, ref_v = net.logits_and_value(obs)
        assert_logits_close(fused.logits[:B], ref_logits, net, note=" B=%d" % B)
        assert float((v - ref_v).abs().max()) < 3e-2 * max(1.0, float(ref_v.abs().max()))
    fused.close()


def test_actor_work_items_of_several_tiles_at_large_batches():
    """From about 3700 windows on, an actor work item covers 2, 3 or 5 tiles whose newest-token rows share one compact
    tile (csrc/policy_fused.cu): sizes around every switch, with ragged last tiles and last groups."""
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    net, _ = _net()
    fused = FusedPolicyForward(16500, "cuda")
    fused.sync(net)
    g = torch.Generator(device="cuda").manual_seed(2)
    for B in (3699, 3700, 3751, 7399, 7437, 14799, 14800 + 13, 16384, 16500):
        obs = torch.rand(B, 5, 14, device="cuda", generator=g)
        obs[:, :, 13] = 1.0
        lead = torch.arange(B, device="cuda") % 5                    # episode starts: 0..4 leading zero rows
        obs[torch.arange(5, device="cuda")[None, :] < lead[:, None]] = 0.0
        _, _, v, _ = fused.get_action(obs, step=3)
        with torch.no_grad():
            ref_logits, ref_v = net.logits_and_value(obs)
        assert_logits_close(fused.logits[:B], ref_logits, net, note=" B=%d" % B)
        assert float((v - ref_v).abs().max()) < 3e-2 * max(1.0, float(ref_v.abs().max())), B
    fused.close()


def test_fused_forward_is_bit_reproducible():
    """Work items are handed out dynamically and shared memory is re-used across phases and items: any race or stale read
    would show up as run-to-run differences.  Ten forwards of the same 15013 windows must agree bit for bit."""
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    net, _ = _net()
    B = 15013
    fused = FusedPolicyForward(B, "cuda")
    fused.sync(net)
    g = torch.Generator(device="cuda").manual_seed(5)
    obs = torch.rand(B, 5, 14, device="cuda", generator=g)
    obs[::3, :2] = 0.0
    v0 = fused.get_action(obs, step=1)[2].clone()
    ref_logits = fused.logits[:B].clone()
    for _ in range(10):
        v = fused.get_action(obs, step=1)[2]
        assert torch.equal(fused.logits[:B], ref_logits) and torch.equal(v, v0)
    fused.close()


def test_sampling_is_counter_based_and_follows_the_probabilities():
    from target_allocation_ppo_transformer_b200.networks.fused_forward import FusedPolicyForward
    net, _ = _net()
    with torch.no_grad():                       # make the policy opinionated so p1 is far from 1/2
        net.actor_head[2].bias.copy_(torch.tensor([0.0, 1.0]))
    B = 8192
    fused = FusedPolicyForward(B, "cuda", seed=11)
    fused.sync(net)
    obs = torch.rand(B, 5, 14, device="cuda")
    a1 = fused.get_action(obs, step=5)[0].clone()
    a2 = fused.get_action(obs, step=5)[0].clone()
    a3 = fused.get_action(obs, step=6)[0].clone()
    assert torch.equal(a1, a2) and not torch.equal(a1, a3)           # same (seed, step, env) -> same draw
    p1 = torch.softmax(fused.logits[:B], -1)[:, 1]
    assert abs(float(a3.float().mean()) - float(p1.mean())) < 4 * 0.5 / np.sqrt(B)
    fused.close()
