"""ctypes binding of libzkp_b200.so (C ABI: include/zkp_b200.h).

There is NO CPU fallback: if the shared library is missing, or no sm_100 device is visible, the
first use raises ``ZkpB200Error``.  Nothing in this package imports ``oracle/``.
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libzkp_b200.so")

u8p = ctypes.POINTER(ctypes.c_uint8)
u64 = ctypes.c_uint64
u32 = ctypes.c_uint32
c_int = ctypes.c_int
intp = ctypes.POINTER(ctypes.c_int)
u64p = ctypes.POINTER(ctypes.c_uint64)
f32p = ctypes.POINTER(ctypes.c_float)
f64p = ctypes.POINTER(ctypes.c_double)
cbuf = ctypes.c_char_p  # bytes / bytearray-backed buffers are passed as c_char_p or c_void_p
vp = ctypes.c_void_p


class ZkpB200Error(RuntimeError):
    """Raised for every failure of the native layer (missing library, no GPU, CUDA error...)."""


class NotDivisibleError(ZkpB200Error):
    pass


# name -> (restype, argtypes); must list every symbol declared in include/zkp_b200.h
PROTOTYPES = {
    "zkp_init": (c_int, [c_int]),
    "zkp_shutdown": (c_int, []),
    "zkp_last_error": (ctypes.c_char_p, []),
    "zkp_device_info": (c_int, [ctypes.c_char_p, c_int, intp, intp, intp, intp]),
    "zkp_device_mem_info": (c_int, [u64p, u64p]),
    "zkp_device_pci_bus_id": (c_int, [ctypes.c_char_p, c_int]),
    "zkp_launch_count": (u64, []),
    "zkp_timer_start": (c_int, []),
    "zkp_timer_stop": (c_int, [f32p]),
    "zkp_sync": (c_int, []),
    "zkp_g1_msm": (c_int, [vp, vp, u64, vp, intp]),
    "zkp_g2_msm": (c_int, [vp, vp, u64, vp, intp]),
    "zkp_g1_table_load": (c_int, [vp, u64, u64p]),
    "zkp_g2_table_load": (c_int, [vp, u64, u64p]),
    "zkp_g1_table_precompute": (c_int, [u64, c_int]),
    "zkp_g2_table_precompute": (c_int, [u64, c_int]),
    "zkp_table_window_bits": (c_int, [u64, ctypes.POINTER(c_int)]),
    "zkp_scalars_load": (c_int, [vp, u64, u64p]),
    "zkp_free": (c_int, [u64]),
    "zkp_g1_msm_table": (c_int, [u64, u64, vp, u64, vp, intp]),
    "zkp_g2_msm_table": (c_int, [u64, u64, vp, u64, vp, intp]),
    "zkp_g1_msm_dev": (c_int, [u64, u64, u64, u64, u64, vp, intp]),
    "zkp_g2_msm_dev": (c_int, [u64, u64, u64, u64, u64, vp, intp]),
    "zkp_g1_msm_dev_batch": (c_int, [u64, u32, u64p, u64p, u64p, u64p, vp, intp]),
    "zkp_g1_msm_dev_many": (c_int, [u64, u64, u64, u32, u64, u64, vp, intp]),
    "zkp_g2_msm_dev_many": (c_int, [u64, u64, u64, u32, u64, u64, vp, intp]),
    "zkp_g1_msm_dev_partial": (c_int, [u64, u64, u64, u64, u64, vp]),
    "zkp_g1_combine_partials": (c_int, [vp, u32, vp, intp]),
    "zkp_msm_set_window_bits": (c_int, [c_int]),
    "zkp_msm_set_option": (c_int, [ctypes.c_char_p, c_int]),
    "zkp_comm_unique_id": (c_int, [vp]),
    "zkp_comm_init": (c_int, [c_int, c_int, vp]),
    "zkp_comm_info": (c_int, [intp, intp, intp]),
    "zkp_comm_barrier": (c_int, []),
    "zkp_comm_destroy": (c_int, []),
    "zkp_g1_msm_multi": (c_int, [u64, u64, u64, u64, u64, vp, intp]),
    "zkp_g1_msm_multi_table": (c_int, [u64, u64, vp, u64, vp, intp]),
    "zkp_g2_msm_multi": (c_int, [u64, u64, u64, u64, u64, vp, intp]),
    "zkp_g1_msm_dev_begin": (c_int, [u64, u64, u64, u64, u64]),
    "zkp_g1_msm_dev_end": (c_int, [vp, intp]),
    "zkp_g2_msm_dev_begin": (c_int, [u64, u64, u64, u64, u64]),
    "zkp_g2_msm_dev_end": (c_int, [vp, intp]),
    "zkp_g1_msm_multi_begin": (c_int, [u64, u64, u64, u64, u64]),
    "zkp_g1_msm_multi_end": (c_int, [vp, intp]),
    "zkp_g2_msm_multi_begin": (c_int, [u64, u64, u64, u64, u64]),
    "zkp_g2_msm_multi_end": (c_int, [vp, intp]),
    "zkp_fr_dot_dev": (c_int, [u64, u64, u64, u64, u64, vp]),
    "zkp_g1_fixed_base_mul": (c_int, [vp, vp, u64, u64p]),
    "zkp_g2_fixed_base_mul": (c_int, [vp, vp, u64, u64p]),
    "zkp_g1_fixed_base_mul_dev": (c_int, [vp, u64, u64, u64p]),
    "zkp_g1_table_scale": (c_int, [u64, u64, u64, u64, u64, u64p]),
    "zkp_g2_table_scale": (c_int, [u64, u64, u64, u64, u64, u64p]),
    "zkp_g1_table_validate": (c_int, [u64, u64, u64, u64p]),
    "zkp_g2_table_validate": (c_int, [u64, u64, u64, c_int, u64p]),
    "zkp_table_download": (c_int, [u64, u64, u64, vp]),
    "zkp_g1_table_load_compressed": (c_int, [vp, u64, u64p, u64p]),
    "zkp_g2_table_load_compressed": (c_int, [vp, u64, c_int, u64p, u64p]),
    "zkp_table_download_compressed": (c_int, [u64, u64, u64, vp]),
    "zkp_scalars_download": (c_int, [u64, u64, u64, vp]),
    "zkp_scalars_generate": (c_int, [u64, u64, u64p]),
    "zkp_fr_ntt": (c_int, [vp, u32, vp, c_int, vp]),
    "zkp_fr_ntt_dev": (c_int, [u64, u64, u32, vp, c_int, vp]),
    "zkp_fr_vec_op": (c_int, [c_int, vp, vp, u64, vp]),
    "zkp_fr_batch_inverse": (c_int, [vp, u64, vp]),
    "zkp_fr_prefix_product": (c_int, [vp, u64, vp]),
    "zkp_fr_poly_eval": (c_int, [vp, u64, vp, vp]),
    "zkp_fr_vec_matrix": (c_int, [vp, vp, u64, u64, vp]),
    "zkp_groth16_quotient": (c_int, [vp, vp, vp, u64, vp, u64, vp, vp]),
    "zkp_groth16_quotient_dev": (c_int, [u64, u64, u64, u64, u64, u64, u64p, u64p]),
    "zkp_groth16_quotient_batch_dev": (c_int, [u64, u64, u64, u64, u32, u64, u64, u64p]),
    "zkp_groth16_batch_scalars_dev": (c_int, [u64, u64, u64, u64, u64, u64, u32, vp, vp, u64p, u64p, u64p]),
    "zkp_scalars_alloc": (c_int, [u64, u64p]),
    "zkp_scalars_copy": (c_int, [u64, u64, u64, u64, u64]),
    "zkp_scalars_upload": (c_int, [u64, u64, vp, u64]),
    "zkp_scalars_scale": (c_int, [u64, u64, u64, vp]),
    "zkp_fr_poly_eval_dev": (c_int, [u64, u64, u64, vp, vp]),
    "zkp_g2_fixed_base_mul_dev": (c_int, [vp, u64, u64, u64p]),
    "zkp_fr_vec_op_dev": (c_int, [c_int, u64, u64, u64, u64, u64, u64, u64]),
    "zkp_fr_axpy_dev": (c_int, [u64, u64, vp, u64, u64, u64]),
    "zkp_scalars_add_const": (c_int, [u64, u64, u64, vp]),
    "zkp_scalars_fill_powers": (c_int, [u64, u64, u64, vp, vp]),
    "zkp_scalars_convert": (c_int, [u64, u64, u64, c_int]),
    "zkp_scalars_is_zero": (c_int, [u64, u64, u64, intp]),
    "zkp_fr_batch_inverse_dev": (c_int, [u64, u64, u64, c_int]),
    "zkp_fr_scan_dev": (c_int, [c_int, u64, u64, u64, u64, u64]),
    "zkp_groth16_msms_dev": (c_int, [u64, u64, u64, u64, u64, u64, u64, u64, u64, vp, vp, vp, ctypes.POINTER(c_int)]),
    "zkp_fr_poly_eval_multi_dev": (c_int, [u32, u64p, u64p, u64p, vp, vp]),
    "zkp_fr_lincomb_dev": (c_int, [u64, u64, u64, u32, u64p, u64p, u64p, vp]),
    "zkp_fr_div_linear_dev": (c_int, [u64, u64, u64, vp, u64, u64]),
    "zkp_plonk_perm_terms_dev": (c_int, [u64, u64, u64, u64, u64, u64, u64, vp, vp, vp, u64, u64]),
    "zkp_plonk_coset_setup_dev": (c_int, [u64, u32, vp, vp, vp, vp, u64, u64, u64]),
    "zkp_plonk_quotient_dev": (c_int, [u64p, u64, u32, u64, u64, u64, vp, vp, vp, u64]),
    "zkp_fr_ntt_many_dev": (c_int, [u64, u64, u32, vp, c_int, vp, u32]),
    "zkp_plonk_blind_many_dev": (c_int, [u64, u64, u64, u64, u32, vp, u32, u64, u64, u64]),
    "zkp_plonk_perm_terms_many_dev": (c_int, [u64, u64, u64, u64, u64, u64, u64, u64, u32, vp, vp, vp, u64, u64]),
    "zkp_fr_scan_many_dev": (c_int, [c_int, u64, u64, u64, u64, u64, u32]),
    "zkp_plonk_coset_inputs_many_dev": (c_int, [u64, u64, u64, u32, u32, u64]),
    "zkp_plonk_quotient_many_dev": (c_int, [u64, u64p, u64, u32, u32, u64, u64, u64, vp, vp, vp, u64]),
    "zkp_plonk_divisible_many_dev": (c_int, [u64, u64, u32, u32, u64p]),
    "zkp_plonk_split_t_many_dev": (c_int, [u64, u64, u32, u32, u64]),
    "zkp_fr_poly_eval_many_dev": (c_int, [u32, u64p, u64p, u64p, u64p, ctypes.POINTER(u32), u32, u32, vp, vp]),
    "zkp_fr_lincomb_many_dev": (c_int, [u64, u64, u64, u64, u32, u32, u64p, u64p, u64p, u64p, vp]),
    "zkp_fr_div_linear_many_dev": (c_int, [u64, u64, u64, u64, u32, vp, u64, u64, u64]),
    "zkp_plonk_pi_scatter_many_dev": (c_int, [u64, u64, u64, u64, u64, u32, u64, u64]),
    "zkp_plonk_coset_inputs_pi_many_dev": (c_int, [u64, u64, u64, u64, u64, u32, u32, u64]),
    "zkp_plonk_quotient_pi_many_dev": (c_int, [u64, u64p, u64, u32, u32, u64, u64, u64, vp, vp, vp, u64]),
    "zkp_plonk_pi_eval_many_dev": (c_int, [u64, u64, u64, u64, u64, u32, vp, vp, vp]),
    "zkp_sparse_load": (c_int, [vp, vp, vp, u64, u64, u64, u64p]),
    "zkp_sparse_matvec_dev": (c_int, [u64, u64, u64, u64, u64]),
    "zkp_fr_ap_interpolate_dev": (c_int, [u64, u64, u64, vp, u64, u64]),
    "zkp_sparse_matvec_many_dev": (c_int, [u64, u64, u64, u64, u64, u32]),
    "zkp_fr_ap_interpolate_many_dev": (c_int, [u64, u64, u64, u32, vp, u64, u64]),
    "zkp_fr_ap_vanishing_dev": (c_int, [u64, u64, u64]),
    "zkp_fr_ap_lagrange_dev": (c_int, [u64, vp, u64, u64]),
    "zkp_witness_program_load": (c_int, [vp, vp, vp, u64, vp, u64, vp, u64, vp, u64, u64, u64p]),
    "zkp_witness_solve_many_dev": (c_int, [u64, u64, u64, u32, u64, u64, u64p]),
    "zkp_fr_poly_mul": (c_int, [vp, u64, vp, u64, vp]),
    "zkp_fr_poly_divmod": (c_int, [vp, u64, vp, u64, vp, vp]),
    "zkp_msm_profile": (c_int, [c_int]),
    "zkp_msm_last_profile": (c_int, [ctypes.c_char_p, f32p]),
    "zkp_pinned_alloc": (c_int, [u64, ctypes.POINTER(ctypes.c_void_p)]),
    "zkp_pinned_free": (c_int, [vp]),
    "zkp_pairing": (c_int, [vp, vp, vp]),
    "zkp_pairing_check": (c_int, [vp, vp, vp, u64, c_int, intp]),
    "zkp_imad_peak": (c_int, [c_int, f64p, f64p]),
    "zkp_latency_probe": (c_int, [c_int, f64p]),
    "zkp_debug_check_guards": (c_int, [u64p, u64p]),
    "zkp_dbg_field_op": (c_int, [c_int, c_int, vp, vp, u64, vp]),
    "zkp_dbg_point_add": (c_int, [c_int, vp, vp, u64, vp]),
    "zkp_dbg_fp12_op": (c_int, [c_int, vp, vp, u64, vp]),
}

ZKP_ERR_NOT_DIVISIBLE = -5

_lock = threading.Lock()
_lib = None
_initialised = False


def load_library():
    """dlopen the library and bind every prototype (no device needed)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH) and os.environ.get("ZKP_B200_AUTOBUILD", "1") != "0":
            # a fresh checkout: compile the CUDA sources in-tree (this is the build, not a fallback --
            # without nvcc or without the sources it still fails loudly below)
            try:
                from . import build as _build
                _build.build()
            except Exception as e:
                raise ZkpB200Error("libzkp_b200.so is missing and building it failed: %s" % e) from e
        if not os.path.exists(LIB_PATH):
            raise ZkpB200Error(
                "libzkp_b200.so not found at %s: build it with "
                "`python -m interactive_zkp_study_b200.build` (there is no CPU fallback)" % LIB_PATH
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError as e:
                raise ZkpB200Error("libzkp_b200.so does not export %s" % name) from e
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def lib():
    """The initialised library (device selected); raises if no sm_100 GPU is usable."""
    global _initialised
    l = load_library()
    if not _initialised:
        with _lock:
            if not _initialised:
                dev = int(os.environ.get("ZKP_B200_DEVICE", "-1"))
                rc = l.zkp_init(dev)
                if rc != 0:
                    raise ZkpB200Error(
                        "zkp_init failed (%d): %s" % (rc, l.zkp_last_error().decode(errors="replace"))
                    )
                _initialised = True
    return l


def check(rc):
    if rc == 0:
        return
    msg = load_library().zkp_last_error().decode(errors="replace")
    if rc == ZKP_ERR_NOT_DIVISIBLE:
        raise NotDivisibleError(msg)
    raise ZkpB200Error("libzkp_b200 error %d: %s" % (rc, msg))


def buf(b):
    """ctypes view (void*) of a bytes / bytearray object without copying."""
    if b is None:
        return None
    if isinstance(b, bytearray):
        return ctypes.cast((ctypes.c_char * len(b)).from_buffer(b), ctypes.c_void_p) if len(b) else None
    if isinstance(b, bytes):
        return ctypes.cast(ctypes.c_char_p(b), ctypes.c_void_p)
    if isinstance(b, (int, ctypes.c_void_p)):  # raw address (pinned staging buffer)
        return b
    raise TypeError("expected bytes or bytearray")
