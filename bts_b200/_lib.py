"""Loader (and in-tree builder) of libbts_b200.so -- the C-ABI declared in include/bts_b200.h.

The product path has NO fallback: if the library is missing or a symbol cannot be resolved, import of the
ops raises, and every op raises on non-CUDA tensors.  Nothing here imports oracle/.
"""
import ctypes
import glob
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.path.join(_HERE, "libbts_b200.so")
CSRC = os.path.join(_HERE, "csrc")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def needs_build():
    if not os.path.isfile(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(_ROOT, "include", "*.h"))
    return any(os.path.getmtime(f) > t for f in deps)


def build(force=False, verbose=False):
    """nvcc cross-compiles every kernel for sm_100a into bts_b200/libbts_b200.so (works without a GPU)."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    os.makedirs(os.path.join(_HERE, "build"), exist_ok=True)
    for src in sources():
        obj = os.path.join(_HERE, "build", os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        cmd = [nvcc] + NVCC_FLAGS + ["-c", src, "-o", obj]
        if verbose:
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out.decode()))
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH] + objs
    subprocess.check_call(cmd)
    return LIB_PATH


_lib = None

_f = ctypes.c_float
_i = ctypes.c_int
_p = ctypes.c_void_p
_ll = ctypes.c_longlong

# name -> argtypes; must list every symbol include/bts_b200.h declares (tests/test_abi.py checks this)
SIGNATURES = {
    "bts_version": [ctypes.c_char_p, _i],
    "bts_lpg_fwd": [_p, _p, _i, _i, _i, _i, _i, _p],
    "bts_lpg_fwd_fused": [_p, _p, _p, _p, _f, _i, _i, _i, _i, _i, _i, _p],
    "bts_lpg_bwd": [_p, _p, _p, _i, _i, _i, _i, _i, _i, _p],
    "bts_lpg_bwd_fused": [_p, _p, _p, _f, _i, _p, _p, _i, _i, _i, _i, _i, _i, _p],
    "bts_lpg_fwd_h": [_p, _p, _i, _i, _i, _i, _i],
    "bts_lpg_bwd_h": [_p, _p, _p, _i, _i, _i, _i, _i, _i],
    "bts_silog_fwd": [_p, _p, _p, _ll, _f, _p, _p, _p],
    "bts_silog_bwd": [_p, _p, _p, _ll, _f, _p, _p, _p, _p],
    "bts_plane_head_fwd": [_p, _p, _p, _p, _f, _i, _i, _i, _i, _i, _p],
    "bts_plane_head_bwd": [_p, _p, _p, _p, _f, _i, _i, _i, _i, _i, _p],
    "bts_conv_n_tile": [_i],
    "bts_conv_packed_floats": [_i, _i, _i, _i],
    "bts_conv_pack_weights": [_p, _ll, _ll, _ll, _ll, _i, _i, _i, _i, _i, _i, _p, _p],
    "bts_conv_fwd": [_p, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p, _p, _i, _p, _ll, _i, _i, _p],
    "bts_conv_fwd_stats": [_p, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p, _p, _i, _p, _ll, _i, _i, _p, _p, _p],
    "bts_conv_fwd_ex": [_p, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p, _p, _i, _p, _ll, _i, _i, _p,
                        _p, _i, _p],
    "bts_conv_fwd_bnbwd": [_p, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p, _ll, _i, _p, _ll, _p, _i,
                           _p, _p, _i, _p],
    "bts_bn_bwd_coef": [_p, _p, _ll, _i, _p, _p, _p, _p, _p],
    "bts_conv_set_tma": [_i],
    "bts_conv_get_tma": [],
    "bts_conv_set_issue_mode": [_i],
    "bts_conv_set_producer_groups": [_i],
    "bts_conv_group_window": [_i, _i],
    "bts_conv_packed_floats_grouped": [_i, _i, _i, _i],
    "bts_conv_pack_weights_grouped": [_p, _ll, _ll, _ll, _ll, _i, _i, _i, _i, _i, _i, _p, _p],
    "bts_conv_wgrad_grouped_plan": [_i, _i, _i, _i, _i, _i, _i, _p, _p],
    "bts_conv_wgrad_grouped": [_p, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _ll, _p, _i, _p, _ll, _ll, _ll, _ll, _i, _p],
    "bts_conv_wgrad_plan": [_i, _i, _i, _i, _i, _i, _i, _i, _p, _p],
    "bts_conv_wgrad": [_p, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p, _i, _p, _ll, _i, _p, _i, _p, _ll, _ll,
                       _ll, _ll, _i, _p],
    "bts_conv_c1_workspace_floats": [_i, _i],
    "bts_conv_c1_fwd": [_p, _ll, _i, _i, _i, _i, _i, _p, _ll, _ll, _ll, _i, _p, _p],
    "bts_conv_c1_dgrad": [_p, _p, _i, _i, _i, _i, _i, _p, _ll, _ll, _ll, _p, _ll, _p],
    "bts_conv_c1_wgrad": [_p, _ll, _p, _p, _i, _i, _i, _i, _i, _p, _p, _ll, _ll, _ll, _p],
    "bts_bn_stats": [_p, _ll, _ll, _i, _p, _p, _p],
    "bts_bn_finalize": [_p, _p, _ll, _i, _p, _p, _f, _f, _p, _p, _p, _p, _p, _p, _p],
    "bts_bn_finalize_track": [_p, _p, _ll, _i, _p, _p, _f, _f, _p, _p, _p, _p, _p, _p, _p, _p],
    "bts_bn_fold": [_i, _p, _p, _f, _p, _p, _p, _p, _p, _p, _p],
    "bts_bn_relu_bwd_reduce": [_p, _ll, _p, _ll, _ll, _i, _p, _p, _p, _p, _p, _p, _p, _p],
    "bts_bn_relu_bwd_apply": [_p, _ll, _p, _ll, _ll, _i, _p, _p, _p, _p, _ll, _i, _p],
    "bts_wgrad2_set_tma": [_i],
    "bts_wgrad2_set_min_pixels": [_ll],
    "bts_wgrad2_set_min_kblocks": [_i],
    "bts_wgrad2_set_pointwise": [_i],
    "bts_bn_relu_bwd_fused": [_p, _ll, _p, _ll, _ll, _i, _p, _p, _p, _p, _p, _p, _p, _ll, _p, _p, _p],
    "bts_bn_bwd_correct": [_p, _ll, _ll, _i, _p, _p, _p, _ll, _p],
    "bts_bn_bwd_reduce": [_p, _ll, _p, _ll, _ll, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p],
    "bts_bn_bwd_apply": [_p, _ll, _p, _ll, _ll, _i, _p, _p, _p, _i, _p, _ll, _i, _p],
    "bts_bn_apply": [_p, _ll, _ll, _i, _p, _p, _i, _p, _ll, _p],
    "bts_elu_bwd": [_p, _ll, _p, _ll, _ll, _i, _p, _ll, _p],
    "bts_upsample2_sum": [_p, _ll, _i, _i, _i, _i, _p, _ll, _p, _ll, _p],
    "bts_copy_channels": [_p, _ll, _ll, _i, _p, _ll, _i, _p],
    "bts_zero_channels": [_p, _ll, _ll, _i, _i, _p],
    "bts_avgpool2_fwd": [_p, _ll, _i, _i, _i, _i, _p, _ll, _p],
    "bts_avgpool2_bwd": [_p, _ll, _i, _i, _i, _i, _p, _ll, _p],
    "bts_bn_add_relu": [_p, _ll, _ll, _i, _p, _p, _p, _ll, _p, _ll, _p],
    "bts_bn_add": [_p, _ll, _ll, _i, _p, _p, _p, _ll, _p, _ll, _p],
    "bts_relu_bwd": [_p, _ll, _p, _ll, _ll, _i, _p, _ll, _p],
    "bts_maxpool3s2_fwd": [_p, _ll, _i, _i, _i, _i, _p, _ll, _p, _p],
    "bts_maxpool3s2_bwd": [_p, _ll, _p, _i, _i, _i, _i, _p, _ll, _p],
    "bts_fill_zero_f32": [_p, _ll, _p],
    "bts_input_prep": [_p, _i, _i, _p, _f, _p, _i, _i, _i, _p, _ll, _p, _p],
    "bts_eval_errors": [_p, _p, _i, _i, _f, _f, _i, _i, _i, _i, _p, _p, _p],
    "bts_depth_to_u16": [_p, _f, _ll, _p, _p],
    "bts_adamw_chunk": [],
    "bts_adamw_multi": [_p, _p, _p, _i, _p, _p, _i, _p, _i, _p],
    "bts_conv_pack_weights_multi": [_p, _i, _ll, _p],
    "bts_conv_pw_wgrad_eligible": [_i, _i],
    "bts_conv_pw_wgrad_workspace_floats": [_i, _i],
    "bts_conv_pw_fwd_eligible": [_i, _i],
    "bts_conv_pw_fwd": [_p, _ll, _ll, _i, _p, _ll, _ll, _i, _i, _p, _ll, _p],
    "bts_conv_pw_wgrad": [_p, _ll, _p, _ll, _ll, _i, _i, _p, _p, _ll, _ll, _p],
    "bts_dw_partials": [_i, _i, _i, _i, _i],
    "bts_dw_fwd": [_p, _ll, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _ll, _p, _p, _p],
    "bts_dw_dgrad": [_p, _ll, _i, _i, _i, _i, _i, _p, _p, _ll, _p],
    "bts_dw_wgrad": [_p, _ll, _i, _i, _i, _i, _i, _p, _p, _p, _ll, _p, _p, _ll, _ll, _ll, _p],
}
RESTYPES = {"bts_conv_packed_floats": ctypes.c_longlong, "bts_conv_packed_floats_grouped": ctypes.c_longlong, "bts_conv_pw_wgrad_workspace_floats": ctypes.c_longlong,
            "bts_dw_partials": ctypes.c_longlong}


def lib():
    """Returns the loaded library; raises (never falls back) if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                "bts_b200: %s not found -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU / eager fallback)" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError if the symbol is missing
            fn.argtypes = args
            fn.restype = RESTYPES.get(name, ctypes.c_int)
        _lib = L
    return _lib


class BtsNativeError(RuntimeError):
    pass


def check(rc, what):
    if rc != 0:
        if rc == -1:
            raise ValueError("%s: invalid argument (BTS_EINVAL)" % what)
        if rc == -2:
            raise ValueError("%s: misaligned pointer (BTS_EALIGN)" % what)
        raise BtsNativeError("%s failed with code %d" % (what, rc))


# launch counter: bench.py reports how many of OUR kernels ran inside the timed region
launches = 0


def count(n=1):
    global launches
    launches += n
