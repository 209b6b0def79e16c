"""Build the sm_100a shared library (C ABI of include/uavenv_b200.h) in-tree with nvcc.

Output: target-allocation-ppo-transformer_b200/lib/libuavenv_b200.so (git-ignored, travels with gpurun).
nvcc cross-compiles without a GPU, so this also is the repo's "does it build" check
(__graft_entry__.build()).
"""
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_DIR = os.path.join(PKG_DIR, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libuavenv_b200.so")            # the env + GAE (include/uavenv_b200.h)
POLICY_LIB_PATH = os.path.join(LIB_DIR, "libuavpolicy_b200.so")   # the policy rollout forward (include/uavpolicy_b200.h)
OBJ_DIR = os.path.join(LIB_DIR, "obj")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-I", os.path.join(ROOT, "include"), "-I", CSRC]


# library -> [(source, extra flags, headers it depends on)].  The env kernels reproduce the reference's fp64
# operation order: no FMA contraction there.
LIBS = {
    LIB_PATH: [
        ("uavenv_capi.cu", ["-fmad=false"], ["handle.cuh", "philox.cuh", "uavenv_device.cuh", "uavenv_kernels.cuh",
                                             "../../include/uavenv_b200.h"]),
        ("ppo_gae.cu", [], ["handle.cuh", "../../include/uavenv_b200.h"]),
        ("ppo_attn.cu", [], ["handle.cuh", "../../include/uavenv_b200.h"]),
        ("ppo_optim.cu", [], ["handle.cuh", "../../include/uavenv_b200.h"]),
        ("uavenv_episodes.cu", [], ["handle.cuh", "../../include/uavenv_b200.h"]),
    ],
    POLICY_LIB_PATH: [
        ("policy_dense.cu", [], ["policy_gemm.cuh", "tcgen05_util.cuh", "../../include/uavpolicy_b200.h"]),
        ("policy_forward.cu", [], ["handle.cuh", "philox.cuh", "policy_kernels.cuh", "policy_weights.cuh", "tcgen05_util.cuh",
                                   "../../include/uavpolicy_b200.h", "../../include/uavpolicy_eval_b200.h"]),
        ("policy_train.cu", [], ["handle.cuh", "policy_gemm.cuh", "policy_kernels.cuh", "policy_weights.cuh", "../../include/uavpolicy_b200.h"]),
        ("policy_wgrad.cu", [], ["policy_gemm.cuh", "tcgen05_util.cuh", "policy_weights.cuh", "../../include/uavpolicy_b200.h"]),
        ("policy_fused.cu", [], ["policy_kernels.cuh", "tcgen05_util.cuh", "policy_weights.cuh", "../../include/uavpolicy_b200.h"]),
    ],
}


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")


def _digest(paths, extra=""):
    """Content hash of the given files (+ flags): staleness does not depend on mtimes, which a snapshot / checkout to
    another box does not preserve."""
    import hashlib
    h = hashlib.sha256(extra.encode())
    for p in paths:
        h.update(os.path.relpath(p, ROOT).encode())      # relative: the tree is checked out at different places
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _stamp_ok(target, digest):
    try:
        return os.path.isfile(target) and open(target + ".srchash").read().strip() == digest
    except OSError:
        return False


def _write_stamp(target, digest):
    tmp = "%s.srchash.%d" % (target, os.getpid())
    with open(tmp, "w") as f:
        f.write(digest)
    os.replace(tmp, target + ".srchash")


def _unit_deps(src, headers):
    return [os.path.join(CSRC, src)] + [os.path.normpath(os.path.join(CSRC, h)) for h in headers]


def _unit_flags(extra):
    return list(extra) + os.environ.get("UAVENV_EXTRA_NVCC_FLAGS", "").split()


def _lib_digest(lib):
    deps, flags = [], []
    for src, extra, headers in LIBS[lib]:
        deps += _unit_deps(src, headers)
        flags.append(" ".join(extra))
    return _digest(sorted(set(deps)), " ".join(ARCH + COMMON[:4] + flags) + os.environ.get("UAVENV_EXTRA_NVCC_FLAGS", ""))


def source_digest(lib=LIB_PATH):
    """Hash of everything `lib` is built from (recorded next to the .so as <lib>.srchash when it is built)."""
    return _lib_digest(lib)


def up_to_date(lib=LIB_PATH):
    """True when `lib` exists and was built from exactly the sources now in the tree."""
    return _stamp_ok(lib, _lib_digest(lib))


class _BuildLock:
    """Inter-process lock: under torchrun every rank may find the library stale at the same time; one builds, the
    others wait and then see it up to date."""

    def __enter__(self):
        import fcntl
        os.makedirs(LIB_DIR, exist_ok=True)
        self.f = open(os.path.join(LIB_DIR, ".build.lock"), "w")
        fcntl.flock(self.f, fcntl.LOCK_EX)
        return self

    def __exit__(self, *exc):
        import fcntl
        fcntl.flock(self.f, fcntl.LOCK_UN)
        self.f.close()


def build(force=False, verbose=False, lib=None):
    """Compile what is stale.  lib=None builds both libraries; returns the env library's path."""
    targets = [lib] if lib else list(LIBS)
    if not force and all(up_to_date(t) for t in targets):
        return LIB_PATH
    with _BuildLock():
        for target in targets:
            if not force and up_to_date(target):       # re-checked under the lock: another rank may have built it
                continue
            nvcc = _nvcc()
            os.makedirs(OBJ_DIR, exist_ok=True)
            objs, jobs = [], []
            for src, extra, headers in LIBS[target]:
                obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
                objs.append(obj)
                flags = _unit_flags(extra)
                dg = _digest(_unit_deps(src, headers), " ".join(ARCH + COMMON[:4] + flags))
                if not force and _stamp_ok(obj, dg):
                    continue
                tmp_obj = "%s.%d.tmp" % (obj, os.getpid())
                jobs.append((src, [nvcc] + ARCH + COMMON + flags + (["-Xptxas", "-v"] if verbose else []) + [
                    "-c", os.path.join(CSRC, src), "-o", tmp_obj], tmp_obj, obj, dg))
            # compile the translation units side by side
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as pool:
                results = list(pool.map(lambda j: (j, subprocess.run(j[1], capture_output=True, text=True)), jobs))
            for (src, _, tmp_obj, obj, dg), r in results:
                if verbose or r.returncode != 0:
                    sys.stderr.write(r.stdout + r.stderr)
                if r.returncode != 0:
                    raise RuntimeError("nvcc failed on %s" % src)
                os.replace(tmp_obj, obj)
                _write_stamp(obj, dg)
            tmp = "%s.%d.tmp" % (target, os.getpid())
            r = subprocess.run([nvcc] + ARCH + ["-shared", "-o", tmp] + objs, capture_output=True, text=True)
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError("nvcc link failed")
            os.replace(tmp, target)
            _write_stamp(target, _lib_digest(target))
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
