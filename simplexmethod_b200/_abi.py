"""ctypes mirror of include/enumgpu.h (struct layouts and constants).

Shared by the product loader (_lib.py) and — because the oracle deliberately
uses the same structs — by oracle/enumcpu.py.  Keep in lock-step with the
header; tests/test_abi.py checks sizes and exported symbols.
"""
import ctypes as C

MAX_M = 16
MAX_N = 64
MAX_DEVICES = 16

OK = 0
NO_FEASIBLE = 1
ERR_ARG = -1
ERR_RANGE = -2
ERR_NONFINITE = -3
ERR_CUDA = -4

ALGO_AUTO = 0
ALGO_INDEPENDENT = 1
ALGO_SHARED = 2

PIVOT_ABSOLUTE = 0
PIVOT_RELATIVE = 1

UINT64_MAX = (1 << 64) - 1


class Problem(C.Structure):
    _fields_ = [
        ("m", C.c_int32), ("n", C.c_int32), ("lda", C.c_int32), ("maximize", C.c_int32),
        ("A_colmajor", C.c_void_p), ("b", C.c_void_p), ("c", C.c_void_p),
    ]


class Options(C.Structure):
    _fields_ = [
        ("eps_feas", C.c_double), ("eps_piv", C.c_double),
        ("rank_begin", C.c_uint64), ("rank_end", C.c_uint64),
        ("n_devices", C.c_int32), ("algo", C.c_int32),
        ("devices", C.POINTER(C.c_int32)),
        ("stream", C.c_void_p),
        ("shard_index", C.c_int32), ("shard_count", C.c_int32),
        ("pivot_rule", C.c_int32), ("reserved_", C.c_int32),
    ]


class Result(C.Structure):
    _fields_ = [
        ("status", C.c_int32), ("m", C.c_int32),
        ("basis", C.c_int32 * MAX_M),
        ("x_B", C.c_double * MAX_M),
        ("objective", C.c_double), ("key", C.c_double),
        ("best_rank", C.c_uint64), ("n_bases", C.c_uint64),
        ("n_singular", C.c_uint64), ("n_infeasible", C.c_uint64), ("n_feasible", C.c_uint64),
        ("kernel_ms", C.c_double),
        ("algo_used", C.c_int32), ("n_launches", C.c_int32),
    ]


class Partial(C.Structure):
    _fields_ = [
        ("key", C.c_double), ("best_rank", C.c_uint64),
        ("n_bases", C.c_uint64), ("n_singular", C.c_uint64),
        ("n_infeasible", C.c_uint64), ("n_feasible", C.c_uint64),
        ("objective", C.c_double),
        ("x_B", C.c_double * MAX_M),
        ("basis", C.c_int32 * MAX_M),
        ("m", C.c_int32), ("algo_used", C.c_int32),
    ]


assert C.sizeof(Partial) == 256, C.sizeof(Partial)

BASIS_FEASIBLE = 0
BASIS_INFEASIBLE = 1
BASIS_SINGULAR = 2

CERT_OPTIMAL = 0
CERT_BOUNDED = 1
CERT_UNBOUNDED = 2
CERT_UNDECIDED = 3


class Certificate(C.Structure):
    _fields_ = [
        ("status", C.c_int32), ("basis_class", C.c_int32), ("entering", C.c_int32),
        ("m", C.c_int32), ("n", C.c_int32), ("n_launches", C.c_int32),
        ("objective", C.c_double),
        ("y", C.c_double * MAX_M),
        ("reduced_cost", C.c_double * MAX_N),
        ("x_B", C.c_double * MAX_M),
        ("ray", C.c_double * MAX_N),
        ("n_aux_bases", C.c_uint64), ("n_rays", C.c_uint64),
    ]

OPT_WINNER = 0
OPT_WINDOW = 1
OPT_FALLBACK = 2


class Optimum(C.Structure):
    _fields_ = [
        ("cert", Certificate),
        ("basis", C.c_int32 * MAX_M),
        ("source", C.c_int32), ("n_launches", C.c_int32),
        ("rank", C.c_uint64), ("key_bound", C.c_double),
        ("n_window", C.c_uint64), ("window_index", C.c_uint64),
    ]


class CostRange(C.Structure):
    _fields_ = [
        ("decrease", C.c_double), ("increase", C.c_double),
        ("decrease_rank", C.c_uint64), ("increase_rank", C.c_uint64),
        ("decrease_ray", C.c_int32), ("increase_ray", C.c_int32),
    ]


class Ranging(C.Structure):
    _fields_ = [
        ("status", C.c_int32), ("n", C.c_int32), ("n_launches", C.c_int32), ("reserved_", C.c_int32),
        ("n_vertex_bases", C.c_uint64), ("n_ray_bases", C.c_uint64),
        ("kernel_ms", C.c_double),
        ("range", CostRange * MAX_N),
    ]


class RhsRange(C.Structure):
    _fields_ = [
        ("shadow_price", C.c_double), ("decrease", C.c_double), ("increase", C.c_double),
        ("decrease_rank", C.c_uint64), ("increase_rank", C.c_uint64),
    ]


class RhsRanging(C.Structure):
    _fields_ = [
        ("status", C.c_int32), ("m", C.c_int32), ("n_tight", C.c_int32), ("n_launches", C.c_int32),
        ("n_bases", C.c_uint64), ("n_singular", C.c_uint64),
        ("kernel_ms", C.c_double),
        ("tight", C.c_int32 * MAX_N),
        ("range", RhsRange * MAX_M),
    ]


# every symbol include/enumgpu.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "enumgpu_version": (C.c_int, []),
    "enumgpu_last_error": (C.c_char_p, []),
    "enumgpu_device_count": (C.c_int, []),
    "enumgpu_binomial": (C.c_uint64, [C.c_int32, C.c_int32]),
    "enumgpu_rank": (C.c_uint64, [C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    "enumgpu_unrank": (C.c_int, [C.c_int32, C.c_int32, C.c_uint64, C.POINTER(C.c_int32)]),
    "enumgpu_solve": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.POINTER(Result)]),
    "enumgpu_solve_device": (C.c_int, [C.POINTER(Problem), C.c_double, C.POINTER(Options), C.POINTER(Result)]),
    "enumgpu_eval_basis": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.POINTER(C.c_int32),
                                      C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "enumgpu_list_feasible": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.POINTER(C.c_uint64), C.c_uint64,
                                         C.POINTER(C.c_uint64), C.POINTER(Result)]),
    "enumgpu_eval_ranks": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.POINTER(C.c_uint64), C.c_uint64,
                                      C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "enumgpu_enqueue_device": (C.c_int, [C.POINTER(Problem), C.c_double, C.POINTER(Options), C.c_void_p,
                                          C.POINTER(C.c_int32)]),
    "enumgpu_partial_to_result": (None, [C.POINTER(Partial), C.POINTER(Result)]),
    "enumgpu_merge_partial": (None, [C.POINTER(Partial), C.POINTER(Partial)]),
    "enumgpu_shard_begin": (C.c_uint64, [C.c_int32, C.c_int32, C.c_uint64, C.c_uint64, C.c_int32, C.c_int32]),
    "enumgpu_fp64_peak_tflops": (C.c_double, [C.c_int32]),
    "enumgpu_fp64_peak_detail": (C.c_double, [C.c_int32, C.POINTER(C.c_double)]),
    "enumgpu_create": (C.c_int, [C.c_int32, C.POINTER(C.c_void_p)]),
    "enumgpu_destroy": (None, [C.c_void_p]),
    "enumgpu_solve_h": (C.c_int, [C.c_void_p, C.POINTER(Problem), C.POINTER(Options), C.POINTER(Result)]),
    "enumgpu_solve_hv": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.POINTER(Problem), C.POINTER(Options),
                                    C.POINTER(Result)]),
    "enumgpu_enqueue_h": (C.c_int, [C.c_void_p, C.POINTER(Problem), C.c_double, C.POINTER(Options), C.c_void_p,
                                     C.POINTER(C.c_int32)]),
    "enumgpu_handle_stream": (C.c_void_p, [C.c_void_p]),
    "enumgpu_enqueue_host_h": (C.c_int, [C.c_void_p, C.POINTER(Problem), C.POINTER(Options), C.c_void_p, C.POINTER(C.c_int32)]),
    "enumgpu_merge_records": (None, [C.c_void_p, C.c_int32, C.POINTER(Result)]),
    "enumgpu_selftest_rcp": (C.c_int, [C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_double)]),
    "enumgpu_find_ray": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.POINTER(Result)]),
    "enumgpu_certify": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.POINTER(C.c_int32), C.c_double,
                                   C.POINTER(Certificate)]),
    "enumgpu_list_window": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.c_double, C.POINTER(C.c_uint64),
                                       C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(Result)]),
    "enumgpu_certify_bases": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.POINTER(C.c_int32), C.c_uint64,
                                         C.c_double, C.POINTER(Certificate)]),
    "enumgpu_certify_optimum": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.POINTER(Result), C.c_double,
                                           C.c_uint64, C.POINTER(Optimum)]),
    "enumgpu_solve_objectives": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.c_int32, C.POINTER(C.c_double),
                                            C.c_int32, C.c_uint64, C.POINTER(Result)]),
    "enumgpu_cost_ranges": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.POINTER(Result), C.c_double, C.c_uint64,
                                       C.POINTER(Ranging)]),
    "enumgpu_rhs_ranges": (C.c_int, [C.POINTER(Problem), C.POINTER(Options), C.POINTER(Optimum), C.c_double,
                                      C.POINTER(RhsRanging)]),
}

MAX_OBJECTIVES = 1 << 20


def bind(lib, symbols=SYMBOLS):
    for name, (res, args) in symbols.items():
        fn = getattr(lib, name)          # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    return lib
