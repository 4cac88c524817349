"""ctypes loader for the C-ABI shared library (include/sealfm.h, include/sealdec.h).

The library is the product; there is NO Python/CPU fallback.  If libsealb200.so is missing or a
symbol cannot be resolved, importing this module raises — loudly, on purpose.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsealb200.so")

u64 = C.c_uint64
u32 = C.c_uint32
i32 = C.c_int
vp = C.c_void_p
cp = C.c_char_p


class SealB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[sealb200 {code}] {msg}")
        self.code = code


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C seal_b200/csrc`. seal_b200 has no CPU fallback.")
    return C.CDLL(LIB_PATH)


lib = _load()

# name -> (restype, argtypes); mirrors include/sealfm.h one to one
_FM_SIGS = {
    "sealfm_last_error": (cp, []),
    "sealfm_abi_version": (i32, []),
    "sealfm_build": (i32, [vp, u64, C.POINTER(vp)]),
    "sealfm_build_gpu": (i32, [vp, u64, i32, C.POINTER(vp)]),
    "sealfm_save_sdsl": (i32, [vp, cp]),
    "sealfm_from_sections": (i32, [u64, u32, u64, vp, u64, vp, vp, vp, u64, vp, u64, C.POINTER(vp)]),
    "sealfm_build_from_file": (i32, [cp, i32, C.POINTER(vp)]),
    "sealfm_load": (i32, [cp, C.POINTER(vp)]),
    "sealfm_save": (i32, [vp, cp]),
    "sealfm_free": (None, [vp]),
    "sealfm_size": (u64, [vp]),
    "sealfm_sigma": (u64, [vp]),
    "sealfm_max_level": (u32, [vp]),
    "sealfm_section": (i32, [vp, i32, C.POINTER(C.POINTER(u64)), C.POINTER(u64)]),
    "sealfm_to_device": (i32, [vp, i32]),
    "sealfm_device": (i32, [vp]),
    "sealfm_device_bytes": (u64, [vp]),
    "sealfm_set_beginnings": (i32, [vp, vp, u64]),
    "sealfm_backward_search_step": (i32, [vp, u64, vp, vp, vp, vp, vp]),
    "sealfm_backward_search_multi": (i32, [vp, u64, vp, vp, vp, vp]),
    "sealfm_distinct_count_multi": (i32, [vp, u64, vp, vp, vp, vp, u64]),
    "sealfm_locate": (i32, [vp, u64, vp, vp]),
    "sealfm_doc_index_from_rows": (i32, [vp, u64, vp, vp]),
    "sealfm_extract_text": (i32, [vp, u64, vp, vp, vp, vp, u64]),
    "sealfm_backward_search_step_d": (i32, [vp, vp, u64, vp, vp, vp, vp, vp]),
    "sealfm_expand_mask_d": (i32, [vp, vp, u64, vp, vp, vp, u32, u32, u32]),
    "sealfm_debug_sector_probe": (i32, [u64, u64, i32, C.POINTER(C.c_double)]),
}


f32p = C.POINTER(C.c_float)


class ProcessorCfg(C.Structure):          # sealdec_processor_cfg_t
    _fields_ = [("num_beams", C.c_int32), ("pad_token_id", C.c_int32), ("eos_token_id", C.c_int32),
                ("stop_at_count", C.c_int32), ("always_allow_eos", C.c_int32), ("forced_bos_token_id", C.c_int32),
                ("n_force_decoding_from", C.c_int32), ("force_decoding_from", C.POINTER(C.c_int64)),
                ("shift", C.c_int32)]


class BartConfig(C.Structure):            # sealbart_config_t
    _fields_ = [("vocab_size", C.c_int32), ("d_model", C.c_int32), ("encoder_layers", C.c_int32),
                ("decoder_layers", C.c_int32), ("heads", C.c_int32), ("ffn_dim", C.c_int32),
                ("max_positions", C.c_int32), ("scale_embedding", C.c_int32), ("gemm_mode", C.c_int32)]


class DecParams(C.Structure):             # sealdec_params_t
    _fields_ = [("num_beams", C.c_int32), ("min_length", C.c_int32), ("max_length", C.c_int32),
                ("length_penalty", C.c_float), ("eos_token_id", C.c_int32), ("pad_token_id", C.c_int32),
                ("decoder_start_token_id", C.c_int32), ("model_eos_token_id", C.c_int32),
                ("forced_eos_token_id", C.c_int32), ("forced_bos_token_id", C.c_int32),
                ("stop_at_count", C.c_int32), ("always_allow_eos", C.c_int32), ("disable_fm_index", C.c_int32),
                ("remove_invalid_values", C.c_int32), ("n_force_decoding_from", C.c_int32),
                ("force_decoding_from", C.POINTER(C.c_int64)), ("shift", C.c_int32)]


_DEC_SIGS = {
    "sealdec_apply_index_mask_d": (i32, [vp, vp, C.POINTER(ProcessorCfg), vp, C.c_int64, C.c_int64, vp, vp, vp,
                                         C.c_int64, C.c_int64]),
    "sealbart_create": (i32, [C.POINTER(BartConfig), i32, C.POINTER(vp)]),
    "sealbart_free": (None, [vp]),
    "sealbart_set_tensor": (i32, [vp, cp, vp, u64]),
    "sealbart_finalize": (i32, [vp]),
    "sealbart_device_bytes": (u64, [vp]),
    "sealdec_hyps_per_query": (C.c_int64, [C.POINTER(DecParams)]),
    "sealdec_generate": (i32, [vp, vp, vp, C.POINTER(DecParams), vp, vp, C.c_int64, C.c_int64, vp, vp, vp, vp, vp, vp]),
    "sealdec_generate_d": (i32, [vp, vp, vp, C.POINTER(DecParams), vp, vp, C.c_int64, C.c_int64, vp, vp, vp, vp, vp,
                                 vp, vp, vp]),
    "sealdec_generate_dx": (i32, [vp, vp, vp, C.POINTER(DecParams), vp, vp, C.c_int64, C.c_int64, vp, vp, vp, vp, vp,
                                  vp, vp, vp, C.c_int64]),
    "sealbart_set_option": (i32, [vp, cp, C.c_int64]),
    "sealbart_get_stat": (C.c_int64, [vp, cp]),
    "sealdec_teacher_forced": (i32, [vp, vp, vp, C.c_int64, C.c_int64, vp, vp, C.c_int64, C.c_int64, C.c_float, vp,
                                     C.c_int64, vp]),
    "sealdec_debug_step_logits": (i32, [vp, vp, vp, C.c_int64, C.c_int64, C.c_int32, vp, C.c_int64, vp]),
    "sealdec_debug_gemm": (i32, [i32, C.c_int64, C.c_int32, C.c_int32, vp, vp, vp, vp, C.c_int32, C.c_int32,
                                 C.POINTER(C.c_double)]),
    "sealdec_debug_gemm_split": (i32, [i32, C.c_int64, C.c_int32, C.c_int32, vp, vp, vp, C.c_int32, vp, vp]),
    "sealdec_debug_gemm_trace": (i32, [i32, C.POINTER(C.c_int64)]),
    "sealev_first_stage": (i32, [C.c_int64, vp, vp, vp, vp, C.c_int64, vp, vp, vp, i32, i32, C.c_double, C.c_double, C.c_int64, vp, vp]),
    "sealev_score_docs": (i32, [C.c_int64, vp, vp, vp, vp, C.c_int64, C.c_int64, vp, vp, vp, C.c_int64, i32, i32, i32, i32,
                                C.c_double, C.c_double, vp, vp, vp, vp, vp, vp, C.c_int64]),
    "sealev_last_error": (C.c_char_p, []),
    "sealev_set_sum_mode": (None, [i32]),
    "sealdec_last_launch_count": (C.c_int64, [vp]),
    "sealdec_profile_gemm": (i32, [vp, i32, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_double)]),
    "sealdec_last_phase_us": (i32, [vp, C.POINTER(C.c_double)]),
}


def _bind(sigs):
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing: intended
        fn.restype = res
        fn.argtypes = args


_bind(_FM_SIGS)
_bind(_DEC_SIGS)


def check(code):
    if code != 0:
        raise SealB200Error(code, lib.sealfm_last_error().decode(errors="replace"))


def fm_symbols():
    return list(_FM_SIGS)
