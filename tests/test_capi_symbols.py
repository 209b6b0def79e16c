"""CPU-side checks of the drop-in boundary: the shared library builds, loads, and exports every
symbol include/uavenv_b200.h declares; argument validation works without a GPU; and the product
package never reaches into oracle/."""
import ctypes as C
import os
import re

import pytest

from conftest import ROOT

import uavenv_b200 as ub


def _declared(header="uavenv_b200.h", prefix="uavenv|ppo"):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b((?:%s)_[a-z0-9_]+)\s*\(" % prefix, text)))


def test_library_exports_every_declared_symbol():
    L = ub.load_library()
    names = _declared()
    assert len(names) >= 20
    for name in names:
        assert hasattr(L, name), "libuavenv_b200.so does not export %s" % name
    assert L.uavenv_abi_version() == 2


def test_policy_library_exports_every_declared_symbol_and_is_tcgen05():
    import subprocess
    from target_allocation_ppo_transformer_b200 import _build, _capi
    L = _capi.load_policy()
    names = _declared("uavpolicy_b200.h", "uavpolicy|uavtrain")
    assert len(names) == 18
    for name in names:
        assert hasattr(L, name), "libuavpolicy_b200.so does not export %s" % name
    assert L.uavpolicy_abi_version() == 3
    sass = subprocess.run(["cuobjdump", "-sass", _build.POLICY_LIB_PATH], capture_output=True, text=True).stdout
    assert "UTCHMMA" in sass and "UTMALDG" in sass          # tcgen05.mma and TMA loads (B200_PROFILING.md)
    h = C.c_void_p()
    assert L.uavpolicy_create(0, 0, C.byref(h)) == -1       # argument validation without a GPU
    import torch
    if not torch.cuda.is_available():
        assert L.uavpolicy_create(0, 64, C.byref(h)) == -2 and b"no CPU fallback" in L.uavpolicy_last_error(None)
        assert L.uavtrain_create(0, 64, C.byref(h)) == -2 and b"no CPU fallback" in L.uavtrain_last_error(None)
    assert L.uavtrain_create(0, 0, C.byref(h)) == -1


def test_library_is_sm100a_only():
    import subprocess
    from target_allocation_ppo_transformer_b200 import _build
    out = subprocess.run(["cuobjdump", "--list-elf", _build.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_default_cfg_matches_reference_constants():
    from target_allocation_ppo_transformer_b200 import _capi
    c = _capi.UavenvCfg()
    ub.load_library().uavenv_default_cfg(C.byref(c))
    py = ub.Config().to_c()
    for name, _ in _capi.UavenvCfg._fields_:
        assert getattr(c, name) == getattr(py, name), name
    assert (c.num_uavs, c.num_targets, c.num_nfz, c.num_interceptors) == (30, 10, 1, 1)   # configs/config.py:42-49
    assert (c.param_zeta_d, c.param_k, c.cost_weight_omega) == (150.0, 1.2, 0.0)           # :7-8, :53
    assert c.reset_episodes == 200                                                          # :83


def test_create_validates_arguments_without_gpu():
    from target_allocation_ppo_transformer_b200 import _capi
    L = ub.load_library()
    c = ub.Config().to_c()
    h = C.c_void_p()
    assert L.uavenv_create(C.byref(c), 0, 0, 1, 0, C.byref(h)) == -1          # num_envs <= 0
    assert b"num_envs" in L.uavenv_last_error(None)
    bad = ub.Config(NUM_TARGETS=0).to_c()
    assert L.uavenv_create(C.byref(bad), 4, 0, 1, 0, C.byref(h)) == -1
    assert L.uavenv_create(None, 4, 0, 1, 0, C.byref(h)) == -1
    import torch
    if not torch.cuda.is_available():
        # no device: creation must fail loudly, never fall back to the CPU
        assert L.uavenv_create(C.byref(c), 4, 0, 1, 0, C.byref(h)) == -2
        assert b"no CPU fallback" in L.uavenv_last_error(None)
        with pytest.raises(RuntimeError):
            ub.UAVEnvBatched(4)
    assert isinstance(_capi.UavenvError(-1, "x"), RuntimeError)


def test_handle_free_calls_report_their_arguments_without_gpu():
    """Every entry point without a handle leaves its failure in uavenv_last_error(NULL), naming itself and the argument;
    _capi.check raises it."""
    from target_allocation_ppo_transformer_b200 import _capi
    L = ub.load_library()
    p = 64                            # never dereferenced: validation fails first

    def message(rc):
        assert rc == -1
        return L.uavenv_last_error(None).decode()

    def gae(rewards=p, T=4, B=8, normalize=0, stats=None):
        return L.ppo_gae_advantages(rewards, p, p, None, T, B, 0.99, 0.95, p, p, normalize, stats, 0, None)

    assert message(gae(rewards=None)).startswith("ppo_gae_advantages: rewards /")
    assert message(gae(T=0)) == "ppo_gae_advantages: need T > 0 and B > 0 (got 0, 8)"
    assert message(gae(B=-1)) == "ppo_gae_advantages: need T > 0 and B > 0 (got 4, -1)"
    assert message(gae(normalize=1)) == "ppo_gae_advantages: normalize needs adv_stats"
    assert message(L.ppo_normalize_advantages(p, 8, None, 0, None)).startswith("ppo_normalize_advantages: advantages /")
    assert message(L.ppo_normalize_advantages(p, 0, p, 0, None)) == "ppo_normalize_advantages: n must be > 0 (got 0)"

    def attn(q=p, n=8, nq=5, q_stride=128):
        return L.ppo_attn5_forward(q, q_stride, p, p, 384, p, n, nq, p, 0, None)

    assert message(attn(q=None)).startswith("ppo_attn5_forward: q /")
    assert message(attn(n=0)) == "ppo_attn5_forward: n must be > 0 (got 0)"
    assert message(attn(nq=3)) == "ppo_attn5_forward: num_queries 3 is neither 1 nor 5"
    assert "multiples of 4" in message(attn(q_stride=130))

    def adam(params=p, n=10, ends=(4, 10), num_segments=None):
        seg_end, seg_lr = (C.c_int64 * len(ends))(*ends), (C.c_float * len(ends))(*[1e-3] * len(ends))
        return L.ppo_clip_adam_step(params, p, p, p, n, seg_end, seg_lr, len(ends) if num_segments is None else num_segments,
                                    1.0, 0.5, 0.9, 0.999, 1e-8, p, p, None, 0, None)

    assert message(adam(params=None)).startswith("ppo_clip_adam_step: params /")
    assert message(adam(n=0, ends=(0,))) == "ppo_clip_adam_step: n must be > 0 (got 0)"
    assert message(adam(num_segments=0)).startswith("ppo_clip_adam_step: num_segments 0 outside [1, ")
    assert message(adam(ends=(6, 4, 10))) == "ppo_clip_adam_step: seg_end decreases at segment 1"
    assert message(adam(ends=(4, 9))) == "ppo_clip_adam_step: the last seg_end (9) is not n (10)"
    with pytest.raises(_capi.UavenvError, match="error -1: ppo_normalize_advantages: n must be > 0"):
        _capi.check(L.ppo_normalize_advantages(p, 0, p, 0, None))


def test_config_mirror_reads_like_the_reference():
    cfg = ub.Config()
    assert cfg.UAV_GEN_X_RANGE == (60, 90) and cfg.GAMMA == 0.998 and cfg.GAE_LAMBDA == 0.95
    cfg.NUM_UAVS = 64            # attribute assignment before building an env, as with the reference singleton
    assert cfg.to_c().num_uavs == 64
    with pytest.raises(AttributeError):
        ub.Config(NOT_A_FIELD=1)
    hard = ub.Config(**ub.HARD_MODE)
    assert hard.PARAM_K == 5.0 and hard.NUM_NFZ == 2


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "target-allocation-ppo-transformer_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "uavenv_oracle" not in src, f
                assert "/root/reference" not in src, f


def test_lazy_exports_resolve_to_the_same_objects_every_time():
    for name in ("train", "PPOAgent", "FusedTrunks", "compute_gae", "TransformerActorCritic", "analyze_environment_difficulty",
                 "record_decisions"):
        first, second = getattr(ub, name), getattr(ub, name)
        assert callable(first) and first is second, name


def test_training_path_refuses_to_run_without_cuda():
    """No CPU fallback anywhere on the product path: the update's library handle cannot be created on a CPU device."""
    with pytest.raises(RuntimeError):
        ub.FusedTrunks(8, "cpu")
    with pytest.raises(RuntimeError):
        ub.FusedPolicyForward(8, "cpu")
