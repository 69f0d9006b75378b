"""ctypes binding of libcidb200.so (include/cidb200.h).

The library is the product: there is NO fallback.  If it has not been built
(``python -c "import __graft_entry__ as g; g.build()"``) importing this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CID_LIB_PATH") or os.path.join(_HERE, "libcidb200.so")     # CID_LIB_PATH: A/B builds of the same ABI (tools/build_variant.sh)

F16, BF16 = 0, 1
EPI_STORE, EPI_GEGLU, EPI_QKV, EPI_GELU, EPI_QUICK_GELU = 0, 1, 2, 3, 4


class CidError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA library has not been built. Run __graft_entry__.build() "
            "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU/eager fallback by design.")
    return C.CDLL(LIB_PATH)


_lib = _load()

_vp, _ll, _i, _f = C.c_void_p, C.c_longlong, C.c_int, C.c_float
_SIGS = {
    "cid_version": ([], _i),
    "cid_last_error": ([], C.c_char_p),
    "cid_gemm_tile_n": ([_i, _i], _i),
    "cid_set_splitk": ([_i, _i], _i),
    "cid_gemm": ([_vp, _ll, _vp, _ll, _i, _i, _vp, _vp, _ll, _i, _i, _vp, _vp, _ll, _vp, _i, _ll, _i, _vp, _i, _i, _i, _i, _f, _i, _vp, C.c_ulonglong, _vp, _i, _vp, _vp, _vp, _f, _vp], _i),
    "cid_conv3x3": ([_vp, _vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _vp, _vp, _ll, _vp, _ll, _f, _i, _vp, C.c_ulonglong, _vp, _vp], _i),
    "cid_attn_self": ([_vp, _ll, _vp, _ll, _vp, _vp, _ll, _i, _i, _i, _i, _i, _vp], _i),
    "cid_attn_self_ragged": ([_vp, _ll, _vp, _ll, _vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _vp], _i),
    "cid_attn_cross": ([_vp, _ll, _vp, _vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _f, _i, _vp], _i),
    "cid_pack_cross_kv": ([_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp], _i),
    "cid_gn_stats": ([_vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _i, _vp], _i),
    "cid_gn_apply": ([_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _f, _i, _vp, _vp, _i, _vp], _i),
    "cid_gn_apply_ch": ([_vp, _i, _vp, _vp, _i, _vp, _i, _i, _i, _vp, _vp, _f, _i, _vp, _i, _vp], _i),
    "cid_gn_small": ([_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _f, _i, _vp, _i, _vp], _i),
    "cid_layernorm": ([_vp, _vp, _vp, _vp, _ll, _i, _f, _i, _vp], _i),
    "cid_upsample2x": ([_vp, _vp, _i, _i, _i, _i, _vp], _i),
    "cid_phase_split": ([_vp, _vp, _i, _i, _i, _i, _vp], _i),
    "cid_nchw_to_nhwc_pad": ([_vp, _vp, _i, _i, _i, _i, _vp, _i, _vp], _i),
    "cid_rows_to_nchw": ([_vp, _i, _vp, _i, _i, _i, _vp], _i),
    "cid_add_inplace": ([_vp, _vp, _ll, _i, _vp], _i),
    "cid_timestep_embed": ([_vp, _i, _i, _i, _vp, _ll, _i, _i, _vp], _i),
    "cid_skinny_linear": ([_vp, _ll, _vp, _vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _vp], _i),
    "cid_cfg_sched_step": ([_vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp, _vp, _i, _vp], _i),
    "cid_advance_step": ([_vp, _vp, _vp, _i, _vp], _i),
    "cid_latents_to_input": ([_vp, _vp, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp], _i),
    "cid_silu_inplace": ([_vp, _ll, _i, _vp], _i),
    "cid_inpaint_blend": ([_vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _i, _vp], _i),
    "cid_layernorm_rows": ([_vp, _ll, _ll, _ll, _vp, _vp, _vp, _ll, _ll, _ll, _ll, _ll, _i, _f, _i, _vp], _i),
    "cid_perceiver_attn": ([_vp, _ll, _vp, _ll, _vp, _ll, _i, _i, _i, _i, _i, _i, _vp], _i),
    "cid_softmax_rows": ([_vp, _ll, _ll, _i, _i, _vp], _i),
    "cid_attn_self_causal": ([_vp, _ll, _vp, _ll, _vp, _vp, _ll, _i, _i, _i, _i, _i, _vp], _i),
    "cid_embed_tokens": ([_vp, _i, _i, _i, _vp, _ll, _vp, _vp, _i, _i, _vp], _i),
}
EXPORTS = tuple(_SIGS)
for _name, (_args, _res) in _SIGS.items():
    _fn = getattr(_lib, _name)          # AttributeError here == header / library mismatch
    _fn.argtypes, _fn.restype = _args, _res


def last_error() -> str:
    return _lib.cid_last_error().decode()


LAUNCHES = 0          # number of kernel-launching entry-point calls issued by this process (bench "gpu_launches")


def call(name, *args):
    """Invoke a status-returning entry point; raise CidError with the library's message on failure."""
    global LAUNCHES
    LAUNCHES += 1
    rc = getattr(_lib, name)(*args)
    if rc != 0:
        raise CidError(f"{name} failed ({rc}): {last_error()}")


def version() -> int:
    return _lib.cid_version()


def set_splitk(max_split: int = -1, min_kblocks: int = -1) -> None:
    """GEMM/conv tail-balancing policy (cid_set_splitk); defaults restore the library's measured settings."""
    if _lib.cid_set_splitk(max_split, min_kblocks) != 0:
        raise CidError(last_error())


def gemm_tile_n(n: int, epi: int) -> int:
    return _lib.cid_gemm_tile_n(n, epi)
