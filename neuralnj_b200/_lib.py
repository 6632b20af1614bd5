"""ctypes binding of libnnj (include/nnj.h).  PyTorch is plumbing only: device memory,
streams and pointers.  There is no CPU or eager fallback — if the CUDA library is missing
or fails, the call raises."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnnj.so")
SOURCES = ["nnj_api.cu", "nnj_encoder.cu", "nnj_encoder_tc.cu", "nnj_njloop.cu", "nnj_tc.cu", "nnj_score_tc.cu", "nnj_score_inc.cu", "nnj_alpha_tc.cu", "nnj_score_big.cu", "nnj_llh.cu", "nnj_score_small.cu", "nnj_alpha_small.cu", "nnj_rankloss.cu", "nnj_support.cu", "nnj_llh_nni.cu", "nnj_llh_topo.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-cudart", "static"]

EXPORTS = ["nnj_last_error", "nnj_abi_version", "nnj_model_create", "nnj_model_destroy", "nnj_workspace_bytes",
           "nnj_encode", "nnj_pair_scores_full", "nnj_pair_scores_list", "nnj_pair_scores_incr", "nnj_aggregate",
           "nnj_merge", "nnj_rollout", "nnj_rollout_from_state", "nnj_rollout_host", "nnj_launch_count",
           "nnj_profile_enable", "nnj_profile_classes", "nnj_profile_name", "nnj_profile_read", "nnj_gemm_split_bf16", "nnj_tc_selftest",
           "nnj_llh_workspace_bytes", "nnj_llh_eval", "nnj_llh_optimize_brlen", "nnj_llh_optimize_all", "nnj_gamma_rates",
           "nnj_llh_support_workspace_bytes", "nnj_llh_branch_support", "nnj_llh_topotest_workspace_bytes", "nnj_llh_topology_test",
           "nnj_rank_loss_workspace_bytes", "nnj_rank_loss",
           "nnj_bootstrap_columns", "nnj_split_distances"]


class NnjError(RuntimeError):
    pass


class nnj_config(C.Structure):
    _fields_ = [("embed_dim", C.c_int32), ("num_heads", C.c_int32), ("num_layers", C.c_int32),
                ("vocab_size", C.c_int32), ("patch_size", C.c_int32), ("precision", C.c_int32)]


OBJ_DIR = os.path.join(_HERE, "_build")


def _headers():
    src_dir = os.path.join(_HERE, "csrc")
    return [os.path.join(src_dir, f) for f in os.listdir(src_dir) if f.endswith((".h", ".cuh"))] + [os.path.join(_HERE, "..", "include", "nnj.h")]


def _mtime(path: str) -> float:
    return os.path.getmtime(path) if os.path.exists(path) else -1.0


def _source_hash(flags_now: str) -> str:
    """sha256 over the compile flags and the bytes of every source and header: what libnnj.so was built from."""
    import hashlib
    h = hashlib.sha256(flags_now.encode())
    for path in sorted([os.path.join(_HERE, "csrc", s) for s in SOURCES] + [os.path.abspath(x) for x in _headers()]):
        h.update(os.path.basename(path).encode())
        with open(path, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _read(path: str) -> str:
    try:
        with open(path) as f:
            return f.read()
    except OSError:
        return ""


HASH_TAG = LIB_PATH + ".srchash"      # travels with the .so (git-ignored as a built artefact, not gpurun-ignored)


def build(force: bool = False, verbose: bool = False, jobs: int = 0) -> str:
    """Compile csrc/*.cu for sm_100a into neuralnj_b200/libnnj.so (in-tree, travels with the repo).

    Up to date means: libnnj.so exists and the hash of flags + sources + headers recorded beside it (libnnj.so.srchash) equals
    the tree's - file times do not survive a snapshot copy, contents do.  Otherwise every source becomes an object under
    neuralnj_b200/_build/ (compiled in parallel, rebuilt when the source or any header is newer - or always with force=True /
    NNJ_FORCE_BUILD=1), then the objects are linked.  The whole rebuild holds an exclusive file lock and the library is moved into
    place atomically, so the ranks of one torchrun job (bench.py calls build() on every rank) neither compile into each other's
    objects nor load a half-written library: the first rank builds, the others wait and find it up to date.
    nvcc cross-compiles without a GPU."""
    import fcntl
    from concurrent.futures import ThreadPoolExecutor
    nvcc = os.environ.get("NVCC", "nvcc")
    extra = os.environ.get("NNJ_EXTRA_NVCC_FLAGS", "").split()
    flags_now = " ".join(NVCC_FLAGS + extra)
    want = _source_hash(flags_now)

    def up_to_date() -> bool:
        return os.path.exists(LIB_PATH) and _read(HASH_TAG) == want

    if not force and up_to_date():
        return LIB_PATH
    os.makedirs(OBJ_DIR, exist_ok=True)
    with open(os.path.join(OBJ_DIR, "build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and up_to_date():      # another process finished the same build while this one waited
                return LIB_PATH
            flags_tag = os.path.join(OBJ_DIR, "flags.txt")
            if _read(flags_tag) != flags_now:
                force = True
            hdr_t = max(_mtime(h) for h in _headers())
            todo, objs = [], []
            for src in SOURCES:
                sp, op = os.path.join(_HERE, "csrc", src), os.path.join(OBJ_DIR, src[:-3] + ".o")
                objs.append(op)
                if force or _mtime(op) < max(_mtime(sp), hdr_t):
                    todo.append((sp, op))
            compile_flags = [f for f in NVCC_FLAGS if f not in ("-shared", "-cudart", "static")]

            def cc(job):
                sp, op = job
                cmd = [nvcc] + compile_flags + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", sp, "-o", op]
                r = subprocess.run(cmd, capture_output=True, text=True)
                return sp, r

            if todo:
                with ThreadPoolExecutor(max_workers=jobs or min(len(todo), os.cpu_count() or 4)) as ex:
                    for sp, r in ex.map(cc, todo):
                        if r.returncode != 0:
                            raise NnjError(f"nvcc failed on {sp}:\n" + r.stdout + r.stderr)
                        if verbose:
                            sys.stderr.write(r.stderr)
            if todo or _mtime(LIB_PATH) < max(_mtime(o) for o in objs):
                tmp = LIB_PATH + f".tmp{os.getpid()}"
                r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static", "-o", tmp] + objs,
                                   capture_output=True, text=True)
                if r.returncode != 0:
                    if os.path.exists(tmp):
                        os.remove(tmp)
                    raise NnjError("nvcc link failed:\n" + r.stdout + r.stderr)
                os.replace(tmp, LIB_PATH)
                with open(flags_tag, "w") as f:
                    f.write(flags_now)
            with open(HASH_TAG, "w") as f:
                f.write(want)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH


_lib = None


def lib() -> C.CDLL:
    """Load libnnj.so and declare the prototypes of include/nnj.h."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("NNJ_LIB_PATH") or LIB_PATH       # override: A/B runs against another build of the same sources
    if not os.path.exists(path):
        raise NnjError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU fallback for the NeuralNJ hot path)")
    L = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    L.nnj_last_error.restype = C.c_char_p
    L.nnj_abi_version.restype = i32
    L.nnj_model_create.argtypes = [C.POINTER(vp), C.POINTER(nnj_config), C.POINTER(vp), C.POINTER(i64), i32, i32]
    L.nnj_model_destroy.argtypes = [vp]
    L.nnj_model_destroy.restype = None
    L.nnj_workspace_bytes.argtypes = [vp, i32, i32, i32, i32]
    L.nnj_workspace_bytes.restype = i64
    L.nnj_encode.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, i64, vp]
    L.nnj_pair_scores_full.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, i64, vp]
    L.nnj_pair_scores_list.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, i32, vp, vp, i64, vp]
    L.nnj_pair_scores_incr.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, i64, vp]
    L.nnj_aggregate.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, vp]
    L.nnj_merge.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, vp]
    L.nnj_rollout.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, i64, vp]
    L.nnj_rollout_from_state.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, i64, vp]
    L.nnj_rollout_host.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp, vp, vp]
    L.nnj_gemm_split_bf16.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp, i64, vp]
    L.nnj_gemm_split_bf16.restype = i32
    L.nnj_tc_selftest.argtypes = [vp, vp, vp, i32, vp]
    L.nnj_tc_selftest.restype = i32
    dp = C.POINTER(C.c_double)
    L.nnj_llh_workspace_bytes.argtypes = [i32, i32, i32]
    L.nnj_llh_workspace_bytes.restype = i64
    L.nnj_llh_eval.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, vp, vp, i64, vp]
    L.nnj_llh_eval.restype = i32
    L.nnj_llh_optimize_brlen.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, C.c_double, vp, vp, vp, i64, vp]
    L.nnj_llh_optimize_brlen.restype = i32
    L.nnj_llh_optimize_all.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, C.c_double, C.c_double, i32, vp, vp, vp, i64, vp]
    L.nnj_llh_optimize_all.restype = i32
    L.nnj_llh_support_workspace_bytes.argtypes = [i32, i32, i32, i32]
    L.nnj_llh_support_workspace_bytes.restype = i64
    L.nnj_llh_branch_support.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, C.c_uint64, i64, i32, vp, vp, vp, vp, vp, vp, vp, i64, vp]
    L.nnj_llh_branch_support.restype = i32
    L.nnj_llh_topotest_workspace_bytes.argtypes = [i32, i32, i32, i32]
    L.nnj_llh_topotest_workspace_bytes.restype = i64
    L.nnj_llh_topology_test.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, C.c_uint64, i32, vp, vp, vp, vp, vp, vp, vp, i64, vp]
    L.nnj_llh_topology_test.restype = i32
    L.nnj_gamma_rates.argtypes = [C.c_double, i32, dp]
    L.nnj_gamma_rates.restype = i32
    L.nnj_rank_loss_workspace_bytes.argtypes = [i32, i32]
    L.nnj_rank_loss_workspace_bytes.restype = i64
    L.nnj_rank_loss.argtypes = [vp, vp, i32, i32, C.c_float, C.c_double, vp, vp, i64, vp]
    L.nnj_rank_loss.restype = i32
    L.nnj_bootstrap_columns.argtypes = [vp, i32, i32, i32, C.c_uint64, i64, i32, vp, vp]
    L.nnj_bootstrap_columns.restype = i32
    L.nnj_split_distances.argtypes = [vp, i32, i32, vp, i32, vp, vp]
    L.nnj_split_distances.restype = i32
    L.nnj_launch_count.argtypes = [i32]
    L.nnj_launch_count.restype = i64
    L.nnj_profile_enable.argtypes = [i32]
    L.nnj_profile_name.argtypes = [i32]
    L.nnj_profile_name.restype = C.c_char_p
    L.nnj_profile_read.argtypes = [i32, C.POINTER(C.c_double), C.POINTER(i64)]
    for name in ("nnj_model_create", "nnj_encode", "nnj_pair_scores_full", "nnj_pair_scores_list", "nnj_pair_scores_incr",
                 "nnj_aggregate", "nnj_merge", "nnj_rollout", "nnj_rollout_from_state", "nnj_rollout_host"):
        getattr(L, name).restype = i32
    if L.nnj_abi_version() != 1:
        raise NnjError("libnnj ABI version mismatch")
    _lib = L
    return L


def check(rc: int, what: str = "libnnj") -> None:
    if rc != 0:
        raise NnjError(f"{what} failed ({rc}): {lib().nnj_last_error().decode()}")
