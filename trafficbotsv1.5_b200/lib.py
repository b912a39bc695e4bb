"""ctypes binding of libtbknarpe.so (C ABI declared in include/tb_knarpe.h) + in-tree nvcc build.

The product path fails loudly when the library is missing: there is no CPU / PyTorch fallback.
"""
import ctypes
import glob
import os
import subprocess
from ctypes import c_float, c_int, c_void_p

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
SO_PATH = os.environ.get("TB_LIB", os.path.join(_PKG, "libtbknarpe.so"))
_SOURCES = ["api.cu", "knn_select.cu", "knarpe_attn.cu", "knarpe_attn_mma.cu", "knarpe_attn_bwd.cu", "linear_f32.cu", "linear_tc.cu", "elementwise.cu", "post_process.cu", "ag_frontend.cu", "mlp_chain.cu",
            "rollout_step.cu", "rule_check.cu", "train_bwd.cu", "wgrad_tc.cu"]
_lib = None

EXPORTS = ["tb_strerror", "tb_version", "tb_knn_select", "tb_knarpe_attn", "tb_linear", "tb_linear_ln", "tb_layernorm",
           "tb_pointnet_pool", "tb_pose_emb", "tb_ag_featurize", "tb_tl_featurize", "tb_dyn_step", "tb_tl_step",
           "tb_step_advance", "tb_gather_rows", "tb_action_mean", "tb_rule_check", "tb_future_filter",
           "tb_traj_global", "tb_womd_post", "tb_ag_frontend", "tb_ag_frontend_blob_halves", "tb_knarpe_attn_bwd", "tb_set_fp16_flag", "tb_dyn_step_ex", "tb_tl_step_ex",
           "tb_dyn_update", "tb_chain_program_bytes", "tb_chain_encode", "tb_chain_run", "tb_layernorm_bwd", "tb_linear_wgrad", "tb_grad_mask",
           "tb_group_sum", "tb_pointnet_pool_bwd", "tb_il_loss_fwd", "tb_il_loss_bwd", "tb_tl_nll", "tb_softmax_nll", "tb_ag_featurize_ex",
           "tb_tl_featurize_ex", "tb_colsum", "tb_ag_frontend_ex", "tb_tf32_split3", "tb_dyn_step_player"]


def build(force: bool = False, verbose: bool = False) -> str:
    """nvcc -gencode arch=compute_100a,code=sm_100a -> trafficbotsv1.5_b200/libtbknarpe.so (cross-compiles on CPU).
    Every csrc/*.cu is compiled to its own object (in parallel, rebuilt only when it or a header changed; objects live
    under csrc/_obj, git- and gpurun-ignored) and the objects are linked into the one shared library."""
    from concurrent.futures import ThreadPoolExecutor
    csrc = os.path.join(_PKG, "csrc")
    hdrs = glob.glob(os.path.join(csrc, "*.cuh")) + [os.path.join(_ROOT, "include", "tb_knarpe.h")]
    hdr_t = max(os.path.getmtime(h) for h in hdrs)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    flags = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
             "-I", os.path.join(_ROOT, "include")]
    if verbose:
        flags.insert(0, "-Xptxas=-v")
    extra = os.environ.get("TB_NVCC_FLAGS")  # tuning experiments only (e.g. -DTB_ATTN_G=2)
    if extra:
        flags[0:0] = extra.split()
        force = True
    objdir = os.path.join(csrc, "_obj")
    os.makedirs(objdir, exist_ok=True)
    jobs, objs = [], []
    for name in _SOURCES:
        src, obj = os.path.join(csrc, name), os.path.join(objdir, name[:-3] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_t):
            jobs.append([nvcc] + flags + ["-c", src, "-o", obj])
    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for r in ex.map(lambda c: subprocess.run(c, capture_output=not verbose, text=True), jobs):
                if r.returncode != 0:
                    raise RuntimeError(f"nvcc failed: {' '.join(r.args)}\n{r.stdout or ''}{r.stderr or ''}")
    if jobs or not os.path.exists(SO_PATH) or any(os.path.getmtime(o) > os.path.getmtime(SO_PATH) for o in objs):
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", SO_PATH] + objs + ["-lcuda"], check=True)
    return SO_PATH


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(f"{SO_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'`. "
                           "There is no CPU fallback for the CUDA hot path.")
    lib = ctypes.CDLL(SO_PATH)
    lib.tb_strerror.restype = ctypes.c_char_p
    lib.tb_strerror.argtypes = [c_int]
    P, I, F = c_void_p, c_int, c_float
    sig = {
        "tb_knn_select": [P, P, P, P, I, I, I, I, I, F, P, P, P, I, I, P, P, I, P],
        "tb_knarpe_attn": [P, I, P, I, P, I, I, I, I, P, I, I, I, I, P, P, P, P, P, I, I, I, I, P, P, I, P, I, P],
        "tb_linear": [P, I, P, P, I, P, I, I, I, I, I, P, P, I, P, I, P, I, I, P],
        "tb_linear_ln": [P, I, P, P, P, I, I, I, I, P, P, I, P, I, P, P, P, I, P],
        "tb_layernorm": [P, I, P, P, P, I, I, I, I, P],
        "tb_pointnet_pool": [P, I, P, I, I, I, I, P, I, P],
        "tb_layernorm_bwd": [P, I, P, P, I, P, I, P, P, I, I, P],
        "tb_linear_wgrad": [P, I, P, I, I, I, I, P, I, P, I, P],
        "tb_colsum": [P, I, I, I, P, P],
        "tb_tf32_split3": [P, I, I, I, P, I, P],
        "tb_grad_mask": [P, I, P, I, P, P, I, I, P, I, P],
        "tb_group_sum": [P, I, I, I, I, P, I, P],
        "tb_pointnet_pool_bwd": [P, I, P, I, I, I, I, P, I, P, I, P],
        "tb_il_loss_fwd": [P, P, P, P, F, P, P, P, P, P, P, P, P, I, I, I, I, I, I, F, F, F, P, P, P],
        "tb_il_loss_bwd": [P, P, P, P, F, P, P, P, P, P, P, I, I, I, I, I, I, F, F, F, P, P, P, P],
        "tb_tl_nll": [P, P, P, I, I, I, P, P, P, P],
        "tb_softmax_nll": [P, I, P, P, I, I, P, P, P, I, P],
        "tb_pose_emb": [P, P, I, P, I, I, P, I, P],
        "tb_ag_featurize": [P, P, P, P, P, P, I, I, I, P, P, P, P, I, P, I, P],
        "tb_tl_featurize": [P, P, P, I, I, I, P, I, P, P],
        "tb_ag_featurize_ex": [P, P, P, P, P, I, P, I, I, I, P, P, P, P, I, P, I, P],
        "tb_tl_featurize_ex": [P, P, P, I, I, I, I, P, I, P, P],
        "tb_dyn_step": [P, P, P, P, F, P, P, P, P, P, P, P, P, P, P, I, I, P, P, P, P, P, P, I, I, F, F, F, P, I, I, I,
                        I, P, P, P, P, P, P, P],
        "tb_dyn_step_ex": [P, P, P, P, F, P, P, P, P, P, P, P, P, P, P, I, I, P, P, P, P, P, P, I, I, F, F, F, P, I, I,
                           I, I, P, P, P, P, P, P, P, P, P],
        "tb_dyn_step_player": [P, P, P, P, F, P, P, P, P, P, P, P, P, P, P, I, I, P, P, P, P, P, P, I, I, F, F, F, P, I,
                               I, I, I, P, P, P, P, P, P, P, P, P, P, P],
        "tb_tl_step": [P, P, P, I, P, I, I, I, I, P, P, P],
        "tb_tl_step_ex": [P, P, P, I, P, I, I, I, I, P, P, P, P],
        "tb_dyn_update": [P, P, P, P, P, P, P, F, I, P, P, P, P, P, P],
        "tb_step_advance": [P, P],
        "tb_chain_program_bytes": [],
        "tb_chain_encode": [P, I, I, P],
        "tb_chain_run": [P, P, P, I, I, P],
        "tb_gather_rows": [P, I, I, P, I, I, I, I, P, I, P],
        "tb_action_mean": [P, P, P, I, P, P],
        "tb_rule_check": [P, P, P, P, P, P, P, P, P, P, P, P, I, I, P, P, P, P, P, P, P, I, I, I, I, I, I, I, F, P],
        "tb_future_filter": [P, P, P, I, I, I, I, I, F, I, P, P, P],
        "tb_traj_global": [P, P, P, P, I, I, I, I, I, I, P, P, P],
        "tb_womd_post": [P, P, P, I, I, I, I, I, I, I, F, F, F, F, I, I, I, P, P, P, P],
        "tb_ag_frontend": [P, P, P, P, P, P, I, I, I, P, P, P, I, P, P, P, P, P, I, P],
        "tb_ag_frontend_ex": [P, P, P, P, P, I, P, I, I, I, P, P, P, I, P, P, P, P, P, I, P],
        "tb_ag_frontend_blob_halves": [],
        "tb_set_fp16_flag": [P],
        "tb_knarpe_attn_bwd": [P, I, P, I, P, I, I, I, I, P, I, I, I, I, P, P, P, P, I, I, I, I, P, P, I, P, I, P, P, P],
    }
    for name, args in sig.items():
        fn = getattr(lib, name)
        fn.restype = c_int
        fn.argtypes = args
    lib.tb_version.restype = c_int
    _lib = lib
    return lib


def check(code: int, what: str) -> None:
    if code != 0:
        raise RuntimeError(f"{what} failed: {load().tb_strerror(code).decode()} ({code})")


def ptr(t):
    """device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream
