"""ctypes binding of libbdetr.so (include/bdetr.h).  There is NO fallback: if the CUDA library is
missing or a call fails, the product path raises."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_float, c_int, c_int32, c_longlong, c_size_t, c_uint32, c_ulonglong, c_void_p, c_char_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libbdetr.so")

BDETR_OK = 0
BDETR_E_BAD_SHAPE, BDETR_E_CUDA, BDETR_E_INVALID_COST, BDETR_E_INFEASIBLE, BDETR_E_NULL, BDETR_E_UNSUPPORTED = -1, -2, -3, -4, -5, -6
BDETR_E_NCCL = -7
MODE_FP32, MODE_TF32, MODE_FP16 = 0, 1, 2


class BdetrError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libbdetr status {code}: {msg}")
        self.code = code


def _ptr_struct(name, fields):
    return type(name, (Structure,), {"_fields_": [(f, c_void_p) for f in fields]})


AttnParams = _ptr_struct("AttnParams", ["wq", "bq", "wk", "bk", "wv", "bv", "wo", "bo", "ln_gamma", "ln_beta"])
AttnSaved = _ptr_struct("AttnSaved", ["qp", "kp", "vp", "o", "lse", "z", "mean", "rstd", "ws16"])
AttnScratch = _ptr_struct("AttnScratch", ["d_qp", "d_kp", "d_vp", "d_o", "d_z", "delta"])
FfnParams = _ptr_struct("FfnParams", ["w1", "b1", "w2", "b2", "ln_gamma", "ln_beta"])
FfnSaved = _ptr_struct("FfnSaved", ["h", "z", "mean", "rstd"])
FfnScratch = _ptr_struct("FfnScratch", ["d_z", "d_h"])
HeadParams = _ptr_struct("HeadParams", ["w1", "b1", "bn_gamma", "bn_beta", "bn_moving_mean", "bn_moving_var", "w2", "b2"])
HeadSaved = _ptr_struct("HeadSaved", ["h", "hn", "bn_mean", "bn_rstd", "bn_acc", "act"])
HeadScratch = _ptr_struct("HeadScratch", ["d_logits", "d_hn", "d_h"])
HeadsSaved = _ptr_struct("HeadsSaved", ["h", "bn_mean", "bn_rstd", "w2f", "b2f", "bn_part", "act0", "act1", "act2"])
HeadsScratch = _ptr_struct("HeadsScratch", ["d_logits", "hTd", "colsum_d", "bn_s", "d_h"])
NeckParams = _ptr_struct("NeckParams", ["bn1_gamma", "bn1_beta", "bn1_moving_mean", "bn1_moving_var", "conv_w", "conv_b",
                                         "bn2_gamma", "bn2_beta", "bn2_moving_mean", "bn2_moving_var"])
NeckSaved = _ptr_struct("NeckSaved", ["t", "wf", "bf", "part", "stat1", "stat2"])
PTR3 = c_void_p * 3
INT3 = c_int * 3


class PosFold(Structure):
    _fields_ = [("pos", c_void_p), ("tab_q", c_void_p), ("tab_k", c_void_p), ("resid_pos", c_int), ("pos_tc", c_void_p)]

P = c_void_p
I = c_int
F = c_float

# name -> (restype, argtypes); must list every function declared in include/bdetr.h
PROTOTYPES = {
    "bdetr_version": (c_int, []),
    "bdetr_last_error": (c_char_p, []),
    "bdetr_set_mode": (c_int, [I]),
    "bdetr_get_mode": (c_int, []),
    "bdetr_attention_f16_workspace_bytes": (c_size_t, [I, I, I, I, I]),
    "bdetr_attention_core_fwd_f16": (c_int, [I, I, I, I, I, P, P, P, P, P, P, P]),
    "bdetr_set_pdl": (c_int, [I]),
    "bdetr_set_concurrency": (c_int, [I]),
    "bdetr_get_concurrency": (c_int, []),
    "bdetr_set_deferred_join": (c_int, [I]),
    "bdetr_join": (c_int, [P]),
    "bdetr_join_into": (c_int, [P, P]),
    "bdetr_get_pdl": (c_int, []),
    "bdetr_launch_count": (c_longlong, []),
    "bdetr_reset_launch_count": (None, []),
    "bdetr_cost_matrix_fwd": (c_int, [I, I, I, I, I, P, P, P, P, P, P, F, F, F, P, P]),
    "bdetr_cost_targets_bytes": (c_size_t, [I, I, I, I]),
    "bdetr_cost_targets_prepare": (c_int, [I, I, I, I, P, P, P, P, P]),
    "bdetr_cost_matrix_prepared": (c_int, [I, I, I, I, I, P, P, P, P, F, F, F, P, P]),
    "bdetr_lsap_assign": (c_int, [I, I, I, P, P, P, P, P, P, P, P]),
    "bdetr_lsap_smem_bytes": (c_size_t, [I, I]),
    "bdetr_matched_loss_fwd": (c_int, [I, I, I, I, I, P, P, P, P, P, P, P, P, P, F, F, F, F, P, P, P]),
    "bdetr_matched_loss_bwd": (c_int, [I, I, I, I, I, P, P, P, P, P, P, P, P, P, F, F, F, F, F, P, P, P, P]),
    "bdetr_attention_block_fwd": (c_int, [I, I, I, I, I, P, P, P, POINTER(AttnParams), F, c_uint32, P, F, P,
                                          POINTER(AttnSaved), P]),
    "bdetr_attention_core_fwd": (c_int, [I, I, I, I, I, P, P, P, P, P, P]),
    "bdetr_attention_core_bwd": (c_int, [I, I, I, I, I, P, P, P, P, P, P, P, P, P, P, P]),
    "bdetr_attention_block_bwd": (c_int, [I, I, I, I, I, P, P, P, POINTER(AttnParams), F, c_uint32, P,
                                          POINTER(AttnSaved), P, P, P, P, I, POINTER(AttnParams),
                                          POINTER(AttnScratch), P]),
    "bdetr_ffn_block_fwd": (c_int, [I, I, P, POINTER(FfnParams), F, c_uint32, P, F, P, POINTER(FfnSaved), P]),
    "bdetr_ffn_block_bwd": (c_int, [I, I, P, POINTER(FfnParams), F, c_uint32, P, POINTER(FfnSaved), P, P, I,
                                    POINTER(FfnParams), POINTER(FfnScratch), P]),
    "bdetr_add_positional_fwd": (c_int, [I, I, I, P, P, P, P]),
    "bdetr_add_positional_bwd": (c_int, [I, I, I, P, P, P]),
    "bdetr_tile_queries_fwd": (c_int, [I, I, I, P, P, P]),
    "bdetr_accumulate": (c_int, [c_size_t, P, P, P]),
    "bdetr_suffix_sum": (c_int, [I, c_size_t, P, P]),
    "bdetr_sgd_step": (c_int, [I, P, P, P, P, P, F, P, F, I, F, P]),
    "bdetr_round_tf32": (c_int, [c_size_t, P, P, P]),
    "bdetr_debug_set_timeline": (c_int, [P]),
    "bdetr_debug_force_attention_kernel": (c_int, [I]),
    "bdetr_head_fwd": (c_int, [I, I, I, I, I, I, F, P, POINTER(HeadParams), F, F, P, I, POINTER(HeadSaved), P]),
    "bdetr_head_bwd": (c_int, [I, I, I, I, I, I, F, P, POINTER(HeadParams), F, POINTER(HeadSaved), P, P, I,
                               POINTER(HeadParams), POINTER(HeadScratch), P]),
    "bdetr_pairwise_iou": (c_int, [I, I, I, P, P, P, P, P]),
    "bdetr_attention_block_saved_bytes": (c_size_t, [I, I, I, I, I, I]),
    "bdetr_attention_block_scratch_bytes": (c_size_t, [I, I, I, I, I]),
    "bdetr_ffn_block_saved_bytes": (c_size_t, [I, I, I]),
    "bdetr_ffn_block_scratch_bytes": (c_size_t, [I, I]),
    "bdetr_heads_saved_bytes": (c_size_t, [I, I, I, I]),
    "bdetr_heads_scratch_bytes": (c_size_t, [I, I, I, I]),
    "bdetr_backbone_neck_fwd": (c_int, [I, I, I, P, POINTER(NeckParams), F, F, I, P, POINTER(NeckSaved), I, P]),
    "bdetr_backbone_neck_bwd": (c_int, [I, I, I, P, POINTER(NeckParams), I, POINTER(NeckSaved), P, POINTER(NeckParams), P, P, P]),
    "bdetr_inverse_tokenize": (c_int, [I, I, I, I, P, P, P, P, P, P, F, P]),
    "bdetr_exit_graph_create": (c_int, [I, POINTER(c_void_p), POINTER(c_ulonglong)]),
    "bdetr_exit_graph_build": (c_int, [P, POINTER(c_void_p), I]),
    "bdetr_exit_graph_launch": (c_int, [P, P]),
    "bdetr_exit_graph_destroy": (c_int, [P]),
    "bdetr_early_exit_decide": (c_int, [I, I, I, P, P, P, P, c_ulonglong, P, P, P]),
    "bdetr_select_exit_predictions": (c_int, [I, I, I, I, I, POINTER(c_void_p), P, P, P, P, P]),
    "bdetr_image_exit_state_bytes": (c_size_t, [I, I]),
    "bdetr_image_exit_plan": (c_int, [I, I, I, I, I, P, P, P, P, c_ulonglong, P, P]),
    "bdetr_image_exit_compact": (c_int, [I, I, I, I, I, I, I, c_longlong, P, POINTER(PTR3), P, POINTER(PTR3), POINTER(PTR3), P, P]),
    "bdetr_switch_graph_create": (c_int, [I, I, POINTER(c_void_p), POINTER(c_ulonglong)]),
    "bdetr_switch_graph_build": (c_int, [P, POINTER(c_void_p), I]),
    "bdetr_comm_unique_id": (c_int, [P]),
    "bdetr_comm_init": (c_int, [POINTER(c_void_p), I, I, P]),
    "bdetr_comm_destroy": (c_int, [P]),
    "bdetr_comm_info": (c_int, [P, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "bdetr_allreduce": (c_int, [P, P, c_size_t, P]),
    "bdetr_broadcast": (c_int, [P, P, c_size_t, I, P]),
    "bdetr_gemm": (c_int, [I, I, I, P, I, P, I, P, I, I, P, P]),
    "bdetr_pos_projection": (c_int, [I, I, P, I, POINTER(PTR3), POINTER(PTR3), POINTER(PTR3), P]),
    "bdetr_attention_fused_fwd": (c_int, [I, I, I, I, I, P, P, POINTER(PosFold), POINTER(AttnParams), F, c_uint32, P, F, I, P,
                                          POINTER(AttnSaved), P]),
    "bdetr_attention_fused_bwd": (c_int, [I, I, I, I, I, P, P, POINTER(PosFold), POINTER(AttnParams), F, c_uint32, P,
                                          POINTER(AttnSaved), P, P, P, I, P, POINTER(AttnParams), POINTER(AttnScratch), P, P, P]),
    "bdetr_ffn_fused_fwd": (c_int, [I, I, P, POINTER(FfnParams), F, c_uint32, P, F, I, P, POINTER(FfnSaved), P]),
    "bdetr_ffn_fused_bwd": (c_int, [I, I, P, POINTER(FfnParams), F, c_uint32, P, POINTER(FfnSaved), P, P, I,
                                    POINTER(FfnParams), POINTER(FfnScratch), P]),
    "bdetr_decoder_self_fwd": (c_int, [I, I, I, I, P, P, POINTER(AttnParams), F, c_uint32, P, F, I, P, POINTER(AttnSaved), P, P]),
    "bdetr_decoder_self_bwd": (c_int, [I, I, I, I, P, P, POINTER(AttnParams), F, c_uint32, P, POINTER(AttnSaved), P, P,
                                       POINTER(AttnParams), POINTER(AttnScratch), P, P, P]),
    "bdetr_heads_fwd": (c_int, [I, I, I, I, I, P, POINTER(HeadParams), POINTER(INT3), F, F, F, POINTER(PTR3), POINTER(PTR3),
                                POINTER(HeadsSaved), P]),
    "bdetr_heads_bwd": (c_int, [I, I, I, I, I, P, POINTER(HeadParams), POINTER(INT3), F, POINTER(HeadsSaved), POINTER(PTR3), P, I,
                                POINTER(PTR3), POINTER(HeadsScratch), P]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Loads libbdetr.so (built by boosted_detr_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: run `python -m boosted_detr_b200.build` (or __graft_entry__.build()). "
            "There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    # A/B switches for debugging / timing (defaults: both on)
    if os.environ.get("BDETR_PDL") is not None:
        lib.bdetr_set_pdl(int(os.environ["BDETR_PDL"]))
    if os.environ.get("BDETR_CONCURRENCY") is not None:
        lib.bdetr_set_concurrency(int(os.environ["BDETR_CONCURRENCY"]))
    _lib = lib
    return lib


def tc_mode() -> bool:
    """True in the tensor-core modes (BDETR_MODE_TF32, and BDETR_MODE_FP16 = the same with fp16 attention operands)."""
    return load().bdetr_get_mode() in (MODE_TF32, MODE_FP16)


def check(code: int) -> None:
    if code != BDETR_OK:
        raise BdetrError(code, load().bdetr_last_error().decode())


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args))
