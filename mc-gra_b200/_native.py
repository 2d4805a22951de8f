"""ctypes binding of libmcgra_b200.so (the C ABI declared in include/mcgra.h).

There is no fallback: if the shared library is missing or a call fails this module raises.  The library
is built in-tree by `build_native.py` (nvcc, sm_100a); `__graft_entry__.build()` calls it.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmcgra_b200.so")

TILE = 128
HID = 16
MAXC = 32
ACC_N = 32
M_NONE, M_MSE, M_KL, M_HSIC, M_CKA, M_DP, M_PRE, M_KDE = 0, 1, 2, 3, 4, 5, 6, 7
ACC = dict(C1=1, C2=2, C6=3, C7=4, SUMCLAMP=8, SUMSQ=9, NLL=16, C9=17, C10=18, C1D=19, C2D=20, C6D=21, C7D=22)

c_fp = C.c_void_p     # device float* (passed as integer address)
i64 = C.c_int64


class ElemArgs(C.Structure):
    _fields_ = [("r", c_fp), ("Ftiles", c_fp), ("lseA", c_fp), ("lseF", c_fp), ("measure", C.c_int),
                ("k1", C.c_float), ("k6", C.c_float), ("acc", c_fp), ("eps_row", c_fp), ("dlse", c_fp)]


class NodeArgs(C.Structure):
    _fields_ = [("n", i64), ("nclass", C.c_int),
                ("W2", c_fp), ("b1", c_fp), ("b2", c_fp), ("Wl", c_fp), ("bl", c_fp),
                ("S1", c_fp), ("labels", c_fp), ("wmult", c_fp), ("HA", c_fp), ("YA", c_fp),
                ("d", c_fp), ("r", c_fp),
                ("B1", c_fp), ("Y1", c_fp), ("B2", c_fp), ("Y2", c_fp), ("B3", c_fp), ("Y3", c_fp),
                ("B4", c_fp), ("Y4", c_fp),
                ("S2", c_fp), ("T2", c_fp), ("H2", c_fp), ("dZ2", c_fp), ("dZ1", c_fp), ("dQ1", c_fp),
                ("dQ2", c_fp), ("demd", c_fp), ("zhat", c_fp), ("dzhat", c_fp),
                ("inv_norm", c_fp), ("masks", c_fp), ("masks2", c_fp), ("eps_row", c_fp), ("rho", c_fp),
                ("Wt", c_fp), ("Fdiag", c_fp), ("acc", c_fp),
                ("measure", C.c_int), ("weight_sup", C.c_float),
                ("k1", C.c_float), ("k2", C.c_float), ("k6", C.c_float), ("k7", C.c_float),
                ("w9", C.c_float), ("w10", C.c_float),
                ("npad", i64),
                ("d_next", c_fp), ("d_fill", C.c_float), ("acc_next", c_fp), ("minmax", c_fp),
                ("lseA", c_fp), ("lseF", c_fp), ("em", c_fp), ("dlse", c_fp), ("measure_nn", C.c_int)]


class FoldArgs(C.Structure):
    _fields_ = [("n", i64), ("npad", i64), ("Wt", c_fp), ("r", c_fp), ("rho", c_fp), ("Ftiles", c_fp),
                ("lseA", c_fp), ("lseF", c_fp), ("zhat", c_fp), ("measure", C.c_int),
                ("k1", C.c_float), ("k6", C.c_float), ("k2", C.c_float), ("norm_coef", C.c_float),
                ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float),
                ("step", C.c_int), ("acc_prev", c_fp), ("acc_next", c_fp), ("d_next", c_fp), ("store_clamped", C.c_int), ("Wk", c_fp), ("step_ptr", c_fp),
                ("plain_gd", C.c_int), ("Gtiles", c_fp)]


class NoisyArgs(C.Structure):
    """mcgra_noisy_args (include/mcgra.h): the --eps != 0 stages."""
    _fields_ = [("n", i64), ("npad", i64), ("tr0", C.c_int), ("tr1", C.c_int), ("tiles", c_fp), ("mu", c_fp),
                ("raw", C.c_int), ("noise", c_fp), ("eps", C.c_float), ("Lt", c_fp), ("Ut", c_fp), ("FLt", c_fp),
                ("FUt", c_fp), ("zhat", c_fp), ("r", c_fp), ("rho", c_fp), ("Wt", c_fp), ("k1", C.c_float),
                ("k2", C.c_float), ("k6", C.c_float), ("acc", c_fp), ("eps_row", c_fp), ("dzhat", c_fp), ("Gt", c_fp),
                ("gslab", c_fp), ("nb", C.c_int)]


PROD_DIRECT, PROD_MIRRORED, PROD_BOTH = 1, 2, 3


class Image(C.Structure):
    """mcgra_image: fp16x2 operand image of an fp32 matrix (include/mcgra.h)."""
    _fields_ = [("hi", c_fp), ("lo", c_fp), ("inv_scale", c_fp), ("rows", i64), ("cols", i64), ("ld", i64)]


class GemmEpilogue(C.Structure):
    _fields_ = [("C", c_fp), ("ldc", i64), ("alpha", C.c_float), ("beta", C.c_float), ("alpha_dev", c_fp),
                ("beta_dev", c_fp), ("u", c_fp), ("v", c_fp), ("coef", C.c_float), ("sumsq", c_fp), ("dot", c_fp),
                ("dot_with", C.POINTER(Image)), ("row0", i64), ("row1", i64)]


class Kl2Args(C.Structure):
    _fields_ = [("tiles", c_fp), ("mu", c_fp), ("raw", C.c_int), ("tr0", C.c_int), ("tr1", C.c_int), ("n", i64),
                ("Ftiles", c_fp), ("Fdiag_feat", c_fp), ("lseF", c_fp), ("zhat", c_fp), ("r", c_fp),
                ("seA", c_fp), ("seM", c_fp), ("lseA", c_fp), ("lseM", c_fp), ("klrow", c_fp), ("c1row", c_fp),
                ("EAt", c_fp), ("Ct", c_fp), ("k1c", C.c_double), ("k2c", C.c_double)]


class NdArgs(C.Structure):
    _fields_ = [("n", i64), ("nclass", C.c_int), ("measure", C.c_int), ("em", c_fp), ("HA", c_fp), ("YA", c_fp),
                ("Wl", c_fp), ("bl", c_fp), ("wmult", c_fp), ("m", C.c_double), ("w9", C.c_float), ("w10", C.c_float),
                ("p2", c_fp), ("mom", c_fp), ("coef", c_fp), ("demd", c_fp), ("acc", c_fp)]


ENSEMBLE_MAX = 8
TERM_GRAM, TERM_DENSE, TERM_LABEL = 0, 1, 2


class EnsembleTerm(C.Structure):
    _fields_ = [("kind", C.c_int), ("d", C.c_int), ("variant", C.c_int), ("pad_", C.c_int), ("Z", c_fp),
                ("rownorm", c_fp), ("dense", c_fp), ("labels", c_fp)]


class EnsembleArgs(C.Structure):
    _fields_ = [("nterms", C.c_int), ("pad_", C.c_int), ("t", EnsembleTerm * ENSEMBLE_MAX)]


_SIGS = {
    "mcgra_version": (C.c_int, []),
    "mcgra_set_engine": (C.c_int, [C.c_int, C.c_int]),
    "mcgra_tiles_in_rows": (i64, [C.c_int, C.c_int]),
    "mcgra_tril_to_tiles": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, c_fp]),
    "mcgra_tiles_to_tril": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, c_fp]),
    "mcgra_dense_to_tiles": (C.c_int, [c_fp, i64, i64, C.c_int, C.c_int, C.c_int, c_fp, c_fp, c_fp]),
    "mcgra_tiles_to_dense": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, i64, c_fp]),
    "mcgra_degree": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, c_fp]),
    "mcgra_propagate_ws_bytes": (i64, [i64, C.c_int]),
    "mcgra_propagate": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, C.c_int, c_fp, c_fp, c_fp]),
    "mcgra_propagate_sel": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, C.c_int, c_fp, c_fp, C.c_int,
                                      c_fp]),
    "mcgra_noise_stage": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, C.c_float, c_fp, c_fp, c_fp, c_fp,
                                    c_fp]),
    "mcgra_noise_tiles": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, C.c_float, c_fp, c_fp, c_fp, c_fp]),
    "mcgra_noise_diag": (C.c_int, [i64, c_fp, C.c_float, c_fp, c_fp, c_fp]),
    "mcgra_diag_axpy": (C.c_int, [c_fp, c_fp, C.c_int, i64, c_fp, c_fp]),
    "mcgra_noisy_terms": (C.c_int, [C.POINTER(NoisyArgs), c_fp]),
    "mcgra_noisy_grad": (C.c_int, [C.POINTER(NoisyArgs), c_fp]),
    "mcgra_node_rho_diag": (C.c_int, [C.POINTER(NodeArgs), c_fp, c_fp]),
    "mcgra_elem_stats": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, C.POINTER(ElemArgs), c_fp]),
    "mcgra_row_sumexp": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, c_fp, c_fp]),
    "mcgra_node_pre": (C.c_int, [C.POINTER(NodeArgs), c_fp]),
    "mcgra_node_mid": (C.c_int, [C.POINTER(NodeArgs), c_fp]),
    "mcgra_node_head": (C.c_int, [C.POINTER(NodeArgs), c_fp]),
    "mcgra_node_bwd2": (C.c_int, [C.POINTER(NodeArgs), c_fp]),
    "mcgra_node_bwd1": (C.c_int, [C.POINTER(NodeArgs), c_fp]),
    "mcgra_node_rho": (C.c_int, [C.POINTER(NodeArgs), c_fp]),
    "mcgra_pairs_ws_bytes": (i64, [i64]),
    "mcgra_pairs": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, c_fp, C.c_float, C.c_float,
                              c_fp, c_fp, c_fp, c_fp, c_fp, c_fp, c_fp]),
    "mcgra_fold_ws_bytes": (i64, [i64]),
    "mcgra_fold_adam": (C.c_int, [c_fp, c_fp, c_fp, C.c_int, C.c_int, c_fp, C.c_int, C.POINTER(FoldArgs), c_fp,
                                  c_fp]),
    "mcgra_bisect_init": (C.c_int, [c_fp, c_fp, C.c_double, c_fp, c_fp, c_fp]),
    "mcgra_bisect_pass": (C.c_int, [c_fp, i64, C.c_int, C.c_int, C.c_float, c_fp, c_fp, c_fp]),
    "mcgra_bisect_update": (C.c_int, [C.c_double, C.c_float, c_fp, c_fp, c_fp, c_fp]),
    "mcgra_bisect_finish": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, c_fp, c_fp, c_fp, C.c_int, c_fp]),
    "mcgra_decode_to_tiles": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, c_fp]),
    "mcgra_decode_band": (C.c_int, [c_fp, i64, i64, i64, c_fp, i64, c_fp]),
    "mcgra_gram_accumulate": (C.c_int, [c_fp, C.c_int, i64, C.c_int, c_fp, c_fp, i64, i64, i64, c_fp]),
    "mcgra_label_accumulate": (C.c_int, [c_fp, i64, c_fp, i64, i64, i64, c_fp]),
    "mcgra_dense_add": (C.c_int, [c_fp, c_fp, i64, c_fp]),
    "mcgra_history_push": (C.c_int, [c_fp, c_fp, i64, c_fp, c_fp]),
    "mcgra_ensemble": (C.c_int, [c_fp, i64, C.POINTER(EnsembleArgs), c_fp, i64, i64, i64, c_fp]),
    "mcgra_row_normalize": (C.c_int, [c_fp, i64, C.c_int, C.c_float, c_fp, c_fp]),
    "mcgra_gauss_stats": (C.c_int, [c_fp, C.c_int, c_fp, C.c_int, i64, C.c_float, C.c_float, c_fp, c_fp, c_fp, c_fp]),
    "mcgra_pair_dense": (C.c_int, [c_fp, C.c_int, i64, c_fp, i64, C.c_int, C.c_float, c_fp, c_fp]),
    "mcgra_cross_moments": (C.c_int, [c_fp, C.c_int, c_fp, C.c_int, c_fp, i64, c_fp, c_fp]),
    "mcgra_gemm_nt": (C.c_int, [C.POINTER(Image), C.POINTER(Image), C.POINTER(GemmEpilogue), c_fp]),
    "mcgra_image_from_dense": (C.c_int, [c_fp, i64, i64, i64, C.c_int, C.POINTER(Image), c_fp, c_fp]),
    "mcgra_image_ahat": (C.c_int, [c_fp, i64, c_fp, C.c_int, c_fp, C.POINTER(Image), c_fp, c_fp]),
    "mcgra_image_m1": (C.c_int, [c_fp, i64, C.POINTER(Image), c_fp, c_fp]),
    "mcgra_center_dense": (C.c_int, [c_fp, i64, i64, c_fp, c_fp]),
    "mcgra_dense_gemv": (C.c_int, [c_fp, i64, i64, i64, c_fp, C.c_double, C.c_int, c_fp, c_fp]),
    "mcgra_dense_sumsq": (C.c_int, [c_fp, i64, i64, i64, c_fp, c_fp]),
    "mcgra_sym_to_tiles": (C.c_int, [c_fp, i64, i64, C.c_int, C.c_int, C.c_float, c_fp, c_fp, c_fp, c_fp]),
    "mcgra_dense_scalars": (C.c_int, [C.c_int, c_fp, C.c_double, C.c_double, C.c_double, c_fp, c_fp, c_fp]),
    "mcgra_d2f": (C.c_int, [c_fp, i64, C.c_double, c_fp, c_fp]),
    "mcgra_kl2_pass": (C.c_int, [C.c_int, C.POINTER(Kl2Args), c_fp]),
    "mcgra_kl2_node": (C.c_int, [C.c_int, C.POINTER(Kl2Args), c_fp, c_fp, c_fp]),
    "mcgra_nd_scratch_doubles": (i64, [C.c_int]),
    "mcgra_nd_scratch_floats": (i64, [C.c_int]),
    "mcgra_nd_measure": (C.c_int, [C.POINTER(NdArgs), c_fp]),
    "mcgra_noise_clamp": (C.c_int, [c_fp, c_fp, C.c_float, i64, c_fp]),
    "mcgra_row_kl": (C.c_int, [c_fp, c_fp, i64, i64, i64, i64, c_fp, c_fp]),
    "mcgra_smooth": (C.c_int, [c_fp, c_fp, c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, C.c_float, c_fp, c_fp, c_fp,
                               c_fp]),
    "mcgra_smooth_node": (C.c_int, [i64, c_fp, c_fp, c_fp, c_fp, C.c_float, c_fp, c_fp, c_fp]),
    "mcgra_cross_moments_bwd": (C.c_int, [c_fp, C.c_int, c_fp, C.c_int, c_fp, i64, c_fp, c_fp, c_fp, c_fp]),
    "mcgra_kde_kv": (C.c_int, [c_fp, i64, C.c_int, i64, C.c_float, c_fp, c_fp]),
    "mcgra_kde_chain": (C.c_int, [c_fp, i64, c_fp, c_fp, C.c_int, i64, C.c_float, c_fp, C.c_int, c_fp]),
    "mcgra_kde_scalars": (C.c_int, [c_fp, C.c_int, C.c_double, C.c_double, c_fp, c_fp, c_fp]),
    "mcgra_slab_ahat": (C.c_int, [c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, C.c_int, c_fp, c_fp]),
    "mcgra_slab_ahat_noisy": (C.c_int, [c_fp, c_fp, c_fp, i64, C.c_int, C.c_int, c_fp, C.c_int, c_fp, c_fp]),
    "mcgra_kde_moments64": (C.c_int, [c_fp, c_fp, C.c_int, i64, C.c_double, C.c_double, c_fp, c_fp]),
    "mcgra_kde_chain64": (C.c_int, [c_fp, c_fp, C.c_int, i64, C.c_double, C.c_double, c_fp, c_fp, c_fp, c_fp]),
    "mcgra_slab_m1": (C.c_int, [c_fp, i64, C.c_int, c_fp, c_fp]),
    "mcgra_slab_to_tiles": (C.c_int, [c_fp, i64, C.c_int, C.c_int, C.c_int, c_fp, c_fp, c_fp]),
    "mcgra_softmax_rows": (C.c_int, [c_fp, c_fp, c_fp, i64, C.c_int, c_fp, c_fp]),
    "mcgra_softmax_chain": (C.c_int, [c_fp, c_fp, c_fp, i64, C.c_int, c_fp, c_fp]),
    "mcgra_auc_workspace_bytes": (i64, [i64, i64]),
    "mcgra_auc_ap": (C.c_int, [c_fp, c_fp, i64, i64, c_fp, c_fp, c_fp]),
    "mcgra_auc_hist_offset": (i64, [i64]),
    "mcgra_auc_stage": (C.c_int, [C.c_int, c_fp, c_fp, i64, i64, c_fp, c_fp, c_fp]),
    "mcgra_sort_workspace_bytes": (i64, [i64]),
    "mcgra_argsort_desc": (C.c_int, [c_fp, i64, c_fp, c_fp, c_fp]),
    "mcgra_topk_workspace_bytes": (i64, [i64, i64, i64]),
    "mcgra_topk_stage": (C.c_int, [C.c_int, c_fp, i64, i64, i64, i64, c_fp, i64, i64, c_fp, c_fp, c_fp]),
}
TOPK_HIST_OFFSET = 256       # MCGRA_TOPK_HIST_OFFSET
TOPK_BINS = 2048

_lib = None


class NativeError(RuntimeError):
    pass


def lib():
    """Load (once) and return the shared library; raises if it is missing -- there is no CPU fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  mcgra_b200 has no CPU / PyTorch fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
        # developer override for same-box A/B runs and profiling: MCGRA_ENGINES="0:5,1:2" (stage:engine, see mcgra.h)
        for item in filter(None, os.environ.get("MCGRA_ENGINES", "").split(",")):
            which, value = item.split(":")
            check(L.mcgra_set_engine(int(which), int(value)), f"MCGRA_ENGINES entry {item!r}")
    return _lib


def exported_symbols():
    return list(_SIGS)


def check(code, what):
    if code != 0:
        raise NativeError(f"{what} failed with code {code}" + (" (cudaError_t)" if code > 0 else " (bad argument)"))


def ptr(t):
    """Device address of a torch tensor (must be contiguous) or None -> NULL."""
    if t is None:
        return None
    assert t.is_contiguous(), "native kernels need contiguous tensors"
    return t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


LAUNCHES = {"count": 0, "kernels": 0}
# hand-written kernels launched per C entry with the default engines (everything else launches exactly one):
# propagate = k_colmax + k_prep_b16 + k_propagate_h; fold_adam = k_prep_w + k_fold_tc; auc_ap = compact + 4 x (hist, scan,
# scatter) + rank + finish; argsort_desc = make_keys + 4 x 3
KERNELS_PER_CALL = {"mcgra_propagate": 3, "mcgra_propagate_sel": 3, "mcgra_noise_stage": 2, "mcgra_fold_adam": 2, "mcgra_auc_ap": 15, "mcgra_argsort_desc": 13,
                    "mcgra_version": 0, "mcgra_set_engine": 0, "mcgra_tiles_in_rows": 0, "mcgra_propagate_ws_bytes": 0,
                    "mcgra_fold_ws_bytes": 0, "mcgra_auc_workspace_bytes": 0, "mcgra_sort_workspace_bytes": 0,
                    "mcgra_pairs_ws_bytes": 0, "mcgra_auc_hist_offset": 0, "mcgra_topk_workspace_bytes": 0, "mcgra_auc_stage": 5, "mcgra_nd_scratch_doubles": 0, "mcgra_nd_scratch_floats": 0, "mcgra_nd_measure": 5,
                    "mcgra_image_from_dense": 2, "mcgra_smooth": 2, "mcgra_center_dense": 2, "mcgra_sym_to_tiles": 2}


TIMERS = {"on": None}     # when a dict: name -> list of (start, end) CUDA events around each call


def call(name, *args, tag=None):
    """Call a C-ABI entry point, check its return code, count the launch (bench.py's gpu_launches)."""
    LAUNCHES["count"] += 1
    LAUNCHES["kernels"] += KERNELS_PER_CALL.get(name, 1)
    tm = TIMERS["on"]
    if tm is not None:
        import torch
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        check(getattr(lib(), name)(*args), name)
        e.record()
        tm.setdefault(tag or name, []).append((s, e))
        return
    check(getattr(lib(), name)(*args), name)
