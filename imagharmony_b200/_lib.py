"""ctypes loader for libimagharmony_sm100.so (the C ABI declared in include/ih_api.h).

The product path has no CPU / PyTorch fallback: if the shared library is missing or a symbol is absent this module
raises, and every op raises ``IHError`` on a non-zero return code.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_longlong, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libimagharmony_sm100.so"
LIB_PATH = os.path.join(_HERE, LIB_NAME)


HASH_PATH = LIB_PATH + ".srchash"
_SRC_DIRS = (os.path.join(_HERE, "csrc"), os.path.join(os.path.dirname(_HERE), "include"))


class IHError(RuntimeError):
    pass


def source_hash() -> str:
    """sha256 over the CUDA / header sources the library is built from (name + content, sorted)."""
    import hashlib
    h = hashlib.sha256()
    for d in _SRC_DIRS:
        for name in sorted(os.listdir(d)):
            if name.endswith((".cu", ".cuh", ".h")) or name == "Makefile":
                h.update(name.encode())
                with open(os.path.join(d, name), "rb") as f:
                    h.update(f.read())
    return h.hexdigest()


def write_source_hash() -> None:
    """Called by __graft_entry__.build() after a successful `make`: records which sources the binary was built from."""
    with open(HASH_PATH, "w") as f:
        f.write(source_hash())


def _check_fresh() -> None:
    """A stale binary must never be tested or benchmarked: the library is refused unless it was built from exactly the
    sources in the tree (IH_SKIP_SRCHASH=1 overrides, for debugging only)."""
    if os.environ.get("IH_SKIP_SRCHASH", "0") == "1":
        return
    if not os.path.exists(HASH_PATH):
        raise IHError(f"{LIB_NAME} has no source hash next to it: rebuild with `python -c 'import __graft_entry__ as g; "
                      "g.build()'`")
    built = open(HASH_PATH).read().strip()
    if built != source_hash():
        raise IHError(f"{LIB_NAME} is STALE: csrc/ or include/ changed since it was built; rebuild with "
                      "`python -c 'import __graft_entry__ as g; g.build()'`")


# name -> (restype, argtypes); must list every symbol of include/ih_api.h (tests/test_abi.py checks this)
SIGNATURES = {
    "ih_last_error": (c_char_p, []),
    "ih_version": (c_int, []),
    "ih_launch_count": (c_longlong, []),
    "ih_launch_count_reset": (None, []),
    "ih_gemm_f16": (c_int, [c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_void_p,
                            c_longlong, c_void_p, c_longlong, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "ih_gemm_ln_f16": (c_int, [c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_void_p,
                               c_longlong, c_void_p, c_longlong, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int,
                               c_float, c_void_p, c_void_p]),
    "ih_gemm_scaled_f16": (c_int, [c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p, c_longlong,
                                   c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "ih_conv2d_scaled_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                     c_int, c_float, c_void_p]),
    "ih_conv2d_shortcut_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p, c_int, c_void_p, c_int,
                                       c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "ih_conv2d_s2_padbr_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                       c_void_p]),
    "ih_gemm_set_trace": (None, [c_void_p]),
    "ih_gemm_prefetch_next": (None, [c_void_p, c_longlong]),
    "ih_conv2d_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_int, c_int,
                              c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "ih_attention_f16": (c_int, [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_void_p,
                                 c_longlong, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "ih_attention_ws_f16": (c_int, [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_void_p,
                                    c_longlong, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_longlong,
                                    c_void_p]),
    "ih_xattn_q_fused_f16": (c_int, [c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_int, c_float, c_void_p,
                                     c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_int, c_int, c_int, c_int,
                                     c_int, c_float, c_int, c_void_p]),
    "ih_attention_workspace_bytes": (c_longlong, [c_int, c_int, c_int, c_int, c_int]),
    "ih_softmax_rows_f16": (c_int, [c_void_p, c_longlong, c_longlong, c_int, c_void_p]),
    "ih_softmax_rows_masked_f16": (c_int, [c_void_p, c_longlong, c_longlong, c_int, c_int, c_void_p]),
    "ih_attention_set_split_policy": (None, [c_int]),
    "ih_attention_set_trace": (None, [c_void_p]),
    "ih_groupnorm_f16": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                 c_int, c_int, c_float, c_int, c_void_p]),
    "ih_groupnorm_workspace_bytes": (c_longlong, [c_int, c_int]),
    "ih_layernorm_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p]),
    "ih_linear_small_f16": (c_int, [c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p,
                                    c_longlong, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "ih_attention_small_f16": (c_int, [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_void_p,
                                       c_longlong, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "ih_add_bcast_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_longlong, c_longlong, c_void_p]),
    "ih_mean_tokens_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "ih_sinusoid_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p]),
    "ih_upsample2x_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "ih_concat_f16": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_longlong, c_void_p]),
    "ih_conv_in_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "ih_conv_out_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "ih_im2col3x3_nchw_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "ih_image_im2col3x3_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "ih_vae_sample_add_noise_f16": (c_int, [c_void_p, c_longlong, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                            c_int, c_int, c_int, c_float, c_float, c_void_p]),
    "ih_vae_sample_inpaint_f16": (c_int, [c_void_p, c_longlong, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                          c_int, c_int, c_int, c_int, c_float, c_float, c_int, c_void_p]),
    "ih_latent_mask_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "ih_nhwc_to_nchw_f16": (c_int, [c_void_p, c_longlong, c_void_p, c_int, c_longlong, c_int, c_void_p]),
    "ih_euler_cfg_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_longlong, c_int,
                                  c_void_p]),
    "ih_attention_generic_f16": (c_int, [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p, c_longlong, c_void_p,
                                         c_longlong, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p]),
    "ih_embed_tokens_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "ih_resize_patchify_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                       ctypes.POINTER(c_float), ctypes.POINTER(c_float), c_void_p]),
    "ih_euler_step_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float, c_longlong, c_int,
                                 c_int, c_void_p]),
    "ih_euler_step_inpaint": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float, c_longlong,
                                      c_int, c_int, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p,
                                      c_void_p]),
    "ih_scale_model_input": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p]),
    "ih_scale_model_input_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_void_p]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library (once). Raises IHError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise IHError(
            f"{LIB_NAME} not found at {LIB_PATH}: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C imagharmony_b200/csrc` (there is no CPU fallback)")
    _check_fresh()
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:  # pragma: no cover
            raise IHError(f"{LIB_NAME} does not export {name}") from e
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().ih_last_error()
        raise IHError(f"{what} failed with code {rc}: {msg.decode() if msg else '?'}")
