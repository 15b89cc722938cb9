"""ctypes binding of libmfgp_b200.so (the C-ABI of include/mfgp_b200.h).

There is NO fallback: if the shared library is missing or a GPU is not present the product raises.  PyTorch is used
only for plumbing (device memory, streams, NCCL); every arithmetic step of the hot path runs in the CUDA library.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_int, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libmfgp_b200.so")

MFGP_OK, MFGP_ERR_INVALID, MFGP_ERR_NOT_SPD, MFGP_ERR_CUDA, MFGP_ERR_EMPTY_CELL = 0, -1, -2, -3, -4
TILE = 64


class NativeLibraryMissing(RuntimeError):
    pass


class MfgpParams(Structure):
    _fields_ = [("s_L", c_double), ("l_L", c_double), ("s_H", c_double), ("l_H", c_double), ("rho", c_double),
                ("noise_L", c_double), ("noise_H", c_double), ("mean_L", c_double), ("mean_H", c_double),
                ("jitter", c_double), ("multi", c_int32), ("reserved", c_int32)]


class MfgpBatch(Structure):      # struct mfgp_batch (include/mfgp_b200.h)
    _fields_ = [(n, c_int64) for n in ("runs", "G", "nx", "ny", "A", "NL", "cap", "algo", "iterations", "max_samples")] + \
               [(n, c_double) for n in ("xmin", "xmax", "ymin", "ymax", "eps", "tie_tol", "amax_rel")] + \
               [(n, c_void_p) for n in ("xy", "f", "ux", "uy", "Xt", "y", "W", "z", "TxL", "TyL", "TxH", "TyH", "mu", "var", "pos",
                                        "prev", "cen", "pos_idx", "prob", "explore", "Ncur", "knew", "status", "noise_used",
                                        "nsamples", "ties", "noise", "unif", "log_loss", "log_agent", "log_sample",
                                        "q", "picks", "nplan", "plan_state", "pmask", "ccount", "cties", "tour_off", "tour_cur",
                                        "tour")]


# name -> (restype, argtypes); this table is also what tests/test_abi.py checks against include/mfgp_b200.h
SIGNATURES = {
    "mfgp_version": (c_char_p, []),
    "mfgp_last_error": (c_char_p, []),
    "mfgp_launch_count": (c_int64, []),
    "mfgp_debug_chol_trace": (c_int64, [c_void_p, c_int64]),
    "mfgp_npad": (c_int64, [c_int64]),
    "mfgp_workspace_bytes": (c_int64, [c_int64]),
    "mfgp_build_train_cov": (c_int, [c_void_p, c_int64, c_int64, POINTER(MfgpParams), c_void_p, c_int64, c_int64,
                                     c_void_p, c_void_p]),
    "mfgp_cholesky": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "mfgp_tri_inverse": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p]),
    "mfgp_whiten": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, POINTER(MfgpParams), c_void_p,
                            c_void_p]),
    "mfgp_posterior": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p,
                               POINTER(MfgpParams), c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "mfgp_grid_tables": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64,
                                 POINTER(MfgpParams), c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "mfgp_posterior_grid": (c_int, [c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                    c_int64, c_void_p, c_int64, c_int64, c_void_p, POINTER(MfgpParams), c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "mfgp_cholesky_append": (c_int, [c_void_p, c_int64, c_int64, c_int64, POINTER(MfgpParams), c_void_p, c_int64,
                                     c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                     c_void_p]),
    "mfgp_append_workspace_bytes": (c_int64, [c_int64]),
    "mfgp_posterior_update": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64,
                                      c_void_p, POINTER(MfgpParams), c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_int64, c_void_p]),
    "mfgp_posterior_grid_update": (c_int, [c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                           c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p, POINTER(MfgpParams),
                                           c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "mfgp_posterior_grid_factored": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64,
                                             c_int64, c_void_p, c_int64, c_int64, c_void_p, POINTER(MfgpParams), c_int64,
                                             c_int64, c_int64, c_int64, c_double, c_double, c_double, c_double, c_int64,
                                             c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "mfgp_posterior_grid_factored_trunc": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64,
                                                   c_int64, c_void_p, c_int64, c_int64, c_void_p, POINTER(MfgpParams), c_int64,
                                                   c_int64, c_int64, c_int64, c_double, c_double, c_double, c_double, c_int64,
                                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                                   c_void_p]),
    "mfgp_posterior_grid_factored_update": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64,
                                                    c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p, POINTER(MfgpParams),
                                                    c_int64, c_int64, c_int64, c_int64, c_double, c_double, c_double, c_double,
                                                    c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                                    c_void_p]),
    "mfgp_factored_workspace_bytes": (c_int64, [c_int64, c_int64, c_int64, c_int64, c_int64, c_int64, c_int64, c_int64]),
    "mfgp_factored_rhs_cols": (c_int64, [c_int64, c_int64, c_int64, c_int64]),
    "mfgp_factored_prepare": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_int64,
                                      c_int64, c_int64, POINTER(MfgpParams), c_int64, c_int64, c_int64, c_int64, c_double,
                                      c_double, c_double, c_double, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p]),
    "mfgp_cholesky_solve_workspace_bytes": (c_int64, [c_int64, c_int64]),
    "mfgp_cholesky_solve": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64,
                                    c_void_p, c_int64, c_void_p]),
    "mfgp_posterior_grid_factored_solved": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64,
                                                    c_int64, c_int64, POINTER(MfgpParams), c_int64, c_int64, c_int64,
                                                    c_int64, c_double, c_double, c_double, c_double, c_int64, c_void_p,
                                                    c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                    c_void_p, c_int64, c_void_p]),
    "mfgp_factored_rhs_cols_trunc": (c_int64, [c_int64, c_void_p]),
    "mfgp_factored_prepare_trunc": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_int64,
                                            c_int64, c_int64, POINTER(MfgpParams), c_int64, c_int64, c_int64, c_int64, c_double,
                                            c_double, c_double, c_double, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int64,
                                            c_void_p]),
    "mfgp_factored_gram_target": (c_void_p, [c_int64, c_int64, c_int64, c_int64, c_int64, c_int64, c_int64, POINTER(MfgpParams),
                                             c_int64, c_int64, c_int64, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64]),
    "mfgp_cholesky_solve_gram_workspace_bytes": (c_int64, [c_int64, c_int64]),
    "mfgp_cholesky_solve_gram": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64,
                                         c_void_p, c_int64, c_void_p, c_int64, c_void_p]),
    "mfgp_posterior_grid_factored_solved_gram": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64,
                                                         c_int64, c_int64, POINTER(MfgpParams), c_int64, c_int64, c_int64,
                                                         c_int64, c_double, c_double, c_double, c_double, c_int64, c_void_p,
                                                         c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                         c_void_p, c_void_p, c_int64, c_void_p]),
    "cov_assign_reduce": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                  c_void_p, c_int64, c_void_p, c_void_p, c_int64,
                                  c_void_p, c_int64, c_void_p, c_void_p, c_int64,
                                  c_double, c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_int64, c_void_p]),
    "cov_workspace_bytes": (c_int64, [c_int64, c_int64, c_int64]),
    "cov_assign_reduce_grid": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                       c_void_p, c_int64, c_void_p, c_void_p, c_int64,
                                       c_void_p, c_int64, c_void_p, c_void_p, c_int64,
                                       c_double, c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_int64, c_void_p]),
    "cov_voronoi_clip_workspace_bytes": (c_int64, [c_int64]),
    "cov_voronoi_clip": (c_int, [c_void_p, c_int64, c_double, c_double, c_double, c_double, c_double, c_void_p, c_void_p,
                                 c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "cov_finish": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_double,
                           c_double, c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "cov_argmax": (c_int, [c_void_p, c_int64, c_int64, c_double, c_double, c_void_p, c_void_p, c_void_p, c_int64,
                           c_void_p]),
    "choi_greedy": (c_int64, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p,
                              POINTER(MfgpParams), c_double, c_double, c_int64, POINTER(c_int64), c_void_p, c_int64,
                              c_void_p]),
    "choi_shard_workspace_bytes": (c_int64, [c_int64, c_int64]),
    "choi_shard_begin": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p,
                                 POINTER(MfgpParams), c_double, c_void_p, c_void_p, c_int64, c_void_p]),
    "choi_shard_append": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_void_p,
                                  POINTER(MfgpParams), c_double, c_void_p, c_int64, c_void_p]),
    "choi_shard_propose": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, POINTER(MfgpParams), c_double,
                                   c_void_p, c_void_p, c_int64, c_void_p]),
    "choi_shard_select": (c_int, [c_void_p, c_int64, c_int64, c_int64, POINTER(MfgpParams), c_double, c_double, c_int64,
                                  c_void_p, c_int64, c_void_p]),
    "choi_shard_status": (c_int, [c_int64, c_int64, c_void_p, c_int64, POINTER(c_int64), POINTER(c_int64), c_void_p]),
    "mfgp_batch_step": (c_int, [POINTER(MfgpBatch), POINTER(MfgpParams), c_int64, c_void_p]),
    "mfgp_batch_choi_begin": (c_int, [POINTER(MfgpBatch), POINTER(MfgpParams), c_void_p]),
    "mfgp_batch_choi_plan": (c_int, [POINTER(MfgpBatch), POINTER(MfgpParams), c_double, c_int64, c_void_p]),
    "mfgp_batch_choi_cluster": (c_int, [POINTER(MfgpBatch), c_void_p]),
    "mfgp_batch_choi_tours": (c_int, [POINTER(MfgpBatch), c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                      c_void_p]),
    "mfgp_nlml_workspace_bytes": (c_int64, [c_int64]),
    "mfgp_nlml_grad": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64,
                               POINTER(MfgpParams), c_void_p, c_void_p, c_int64, c_void_p]),
    "choi_tsp_workspace_bytes": (c_int64, [c_int64]),
    "choi_tsp_tours": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int64,
                               c_void_p]),
}

_lib = None


def lib():
    """The loaded shared library; raises NativeLibraryMissing (never falls back to a CPU path)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise NativeLibraryMissing(
                f"{LIB_PATH} not found: build it with `make -C {os.path.dirname(LIB_PATH)}` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def last_error():
    return lib().mfgp_last_error().decode()


def check(rc, what):
    if rc == MFGP_OK:
        return
    if rc == MFGP_ERR_CUDA:
        raise RuntimeError(f"{what}: CUDA error: {last_error()}")
    if rc == MFGP_ERR_INVALID:
        raise ValueError(f"{what}: invalid argument")
    raise RuntimeError(f"{what}: error code {rc}")


def npad(n):
    return max(TILE, (int(n) + TILE - 1) // TILE * TILE)


def ptr(t):
    """Device pointer of a torch tensor (or None -> NULL)."""
    return None if t is None else c_void_p(t.data_ptr())


_side_streams = {}


def side_stream(device=None):
    """A second stream per device for small independent launches (cell clipping, table building) that overlap the main
    stream's work; joined back with events."""
    import torch
    dev = torch.cuda.current_device() if device is None else torch.device(device).index
    if dev is None:
        dev = torch.cuda.current_device()
    if dev not in _side_streams:
        _side_streams[dev] = torch.cuda.Stream(device=dev)
    return _side_streams[dev]


def stream_ptr(stream=None):
    """cudaStream_t of `stream` (default: torch's current stream on the current device)."""
    import torch
    if stream is not None:
        return c_void_p(stream.cuda_stream)
    try:        # raw C accessor: the Python-level torch.cuda.current_stream() costs ~15 us per call
        return c_void_p(torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice()))
    except AttributeError:
        return c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("mfgp_coverage_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    lib()
