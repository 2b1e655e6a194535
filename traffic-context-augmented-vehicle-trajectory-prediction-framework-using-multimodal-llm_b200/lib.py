"""Build + load of libtcavp.so (the C-ABI shared library declared in include/tcavp.h).

The library is compiled in-tree with nvcc for sm_100a only and loaded through ctypes; there is no CPU
fallback — every op raises if the library is missing or a call fails."""
import ctypes
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libtcavp.so")
INCLUDE = os.path.join(_ROOT, "include")
SOURCES = ["api.cu", "gemm.cu", "attention.cu", "attention_tc.cu", "attention_tm.cu", "attention_x.cu", "attention_xt.cu", "norm.cu", "elementwise.cu", "ltsf.cu", "backward.cu", "attention_bwd_tc.cu", "dw_tc.cu", "lora_drop.cu", "ffn_tm.cu", "ce.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-I", INCLUDE]

EXPORTS = [
    "tcavp_last_error", "tcavp_version", "tcavp_device_info", "tcavp_launch_count", "tcavp_last_kernel", "tcavp_clock_probe", "tcavp_gemm_tile_order", "tcavp_gemm_wide_min_k", "tcavp_gemm", "tcavp_attention",
    "tcavp_layernorm", "tcavp_rmsnorm", "tcavp_row_rstd", "tcavp_rope", "tcavp_rope_table", "tcavp_embed_text", "tcavp_add_rowvec",
    "tcavp_cast", "tcavp_split_bf16x3", "tcavp_poly_embed", "tcavp_masked_mean", "tcavp_ltsf_encode", "tcavp_nlinear_decode",
    "tcavp_fusion_head", "tcavp_fusion_head_tc", "tcavp_ffn64_ln", "tcavp_traj_metrics", "tcavp_best_of_k", "tcavp_dropout",
    # fine-tune step
    "tcavp_transpose", "tcavp_period_sum", "tcavp_relu_bwd", "tcavp_axpby", "tcavp_swiglu", "tcavp_swiglu_bwd", "tcavp_layernorm_bwd",
    "tcavp_rmsnorm_bwd", "tcavp_rope_adjacent", "tcavp_copy_rows", "tcavp_masked_mean_bwd", "tcavp_nlinear_bwd", "tcavp_head_assemble",
    "tcavp_traj_loss_bwd", "tcavp_skinny_dw", "tcavp_dw", "tcavp_attention_bwd", "tcavp_attention_bwd_owned", "tcavp_adamw",
    "tcavp_lora_a_drop", "tcavp_lora_dx_drop", "tcavp_lora_da_drop", "tcavp_ce_loss", "tcavp_gelu_tanh", "tcavp_gelu_tanh_bwd", "tcavp_layernorm_bwd_dx", "tcavp_layernorm_strided",
    # gradient clipping / non-finite step skipping
    "tcavp_clip_prologue", "tcavp_adamw_clipped", "tcavp_mark_nonfinite",
    # fp8 serving mode
    "tcavp_quant_e4m3_rows",
]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "tcavp.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compiles csrc/*.cu -> libtcavp.so (sm_100a).  Cross-compiles fine on a box without a GPU."""
    if not force and not _stale():
        return LIB_PATH
    # one builder at a time (torchrun starts N ranks at once): the others wait on the lock and then find a fresh library
    import fcntl
    os.makedirs(os.path.join(_HERE, "build"), exist_ok=True)
    with open(os.path.join(_HERE, "build", ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale():
                return LIB_PATH
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose):
    objdir = os.path.join(_HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out:
            print(out)
        objs.append(obj)
    tmp = LIB_PATH + f".tmp{os.getpid()}"
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp, *objs]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(tmp, LIB_PATH)       # atomic: a concurrent loader never sees a half-written library
    return LIB_PATH


_lib = None
_lock = threading.Lock()


def load():
    """Returns the ctypes handle, raising loudly if the library has not been built."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                   "(there is no CPU fallback)")
            lib = ctypes.CDLL(LIB_PATH)
            lib.tcavp_last_error.restype = ctypes.c_char_p
            lib.tcavp_launch_count.restype = ctypes.c_longlong
            lib.tcavp_last_kernel.restype = ctypes.c_char_p
            for name in EXPORTS:
                getattr(lib, name)   # AttributeError if a declared symbol is not exported
            _lib = lib
    return _lib


class TcavpError(RuntimeError):
    pass


def check(rc, what=""):
    if rc != 0:
        msg = load().tcavp_last_error().decode(errors="replace")
        raise TcavpError(f"{what} failed ({rc}): {msg}")
