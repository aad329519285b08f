"""ctypes binding of libdqlb200.so (include/dqlb200.h).  There is no CPU fallback: if the CUDA library is
missing or does not export every symbol the header declares, importing the product path raises."""
from __future__ import annotations

import ctypes as C
import os
import pathlib

from . import constants as K

PKG = pathlib.Path(__file__).resolve().parent
# DQLB200_LIB: another build of the same library (kernel A/B measurements, tools/perf_probe.py); never a different backend
LIB_PATH = pathlib.Path(os.environ.get("DQLB200_LIB") or PKG / "libdqlb200.so")

SYMBOLS = [
    "dqlb200_abi_version", "dqlb200_config_bytes", "dqlb200_population_state_bytes", "dqlb200_last_error",
    "dqlb200_termination_string", "dqlb200_create", "dqlb200_destroy", "dqlb200_bind", "dqlb200_reset",
    "dqlb200_train", "dqlb200_train_host", "dqlb200_train_host_ext", "dqlb200_eval_greedy", "dqlb200_transfer", "dqlb200_check_errors",
    "dqlb200_shared_pack", "dqlb200_shared_apply", "dqlb200_mdp_facade_step", "dqlb200_agent_facade", "dqlb200_selftest_division", "dqlb200_replica_merge", "dqlb200_bind_merge_snapshot", "dqlb200_eval_greedy_2d", "dqlb200_eval2d_params_bytes", "dqlb200_bench_table_rmw", "dqlb200_train_merged", "dqlb200_env_reset", "dqlb200_env_step", "dqlb200_agent_select", "dqlb200_agent_update", "dqlb200_uses_default_instance", "dqlb200_config_is_default", "dqlb200_bench_launch_floor", "dqlb200_bind_filter_state", "dqlb200_bind_dynamics_state", "dqlb200_selftest_discretise", "dqlb200_env_state_bytes", "dqlb200_shared_sync_nccl", "dqlb200_eval_agents", "dqlb200_eval_pairs",
]

OP_ACTION, OP_OBSERVE, OP_CHECK, OP_REWARD, OP_RESET, OP_SIMULATION = 1, 2, 4, 8, 16, 256
AGENT_PREDICT, AGENT_UPDATE, AGENT_TRANSFER = 1, 2, 4

_lib = None


class Dqlb200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the library (building it is the job of build.py / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise Dqlb200Error(f"{LIB_PATH} not found: run `python -m dql_multirotor_landing_b200.build` "
                           "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    missing = [s for s in SYMBOLS if not hasattr(lib, s)]
    if missing:
        raise Dqlb200Error(f"libdqlb200.so does not export {missing}")
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    lib.dqlb200_abi_version.restype = C.c_int
    lib.dqlb200_config_bytes.restype = C.c_size_t
    lib.dqlb200_population_state_bytes.restype = C.c_size_t
    lib.dqlb200_eval2d_params_bytes.restype = C.c_size_t
    lib.dqlb200_env_state_bytes.restype = C.c_size_t
    lib.dqlb200_env_state_bytes.argtypes = [C.c_int, C.c_int]
    lib.dqlb200_last_error.restype = C.c_char_p
    lib.dqlb200_termination_string.restype = C.c_char_p
    lib.dqlb200_termination_string.argtypes = [i32]
    lib.dqlb200_create.argtypes = [C.POINTER(K.Config), C.POINTER(C.c_float), C.POINTER(K.PopulationParams), i32, C.POINTER(vp)]
    lib.dqlb200_destroy.argtypes = [vp]
    lib.dqlb200_uses_default_instance.argtypes = [vp]
    lib.dqlb200_config_is_default.argtypes = [C.POINTER(K.Config)]
    lib.dqlb200_bind.argtypes = [vp, vp, vp, vp]
    lib.dqlb200_reset.argtypes = [vp, i32, vp]
    lib.dqlb200_train.argtypes = [vp, i32, C.POINTER(K.Trace), vp]
    lib.dqlb200_train_host.argtypes = [vp, i32, vp, vp, vp, i32, vp]
    lib.dqlb200_train_host_ext.argtypes = [vp, i32, vp, vp, vp, vp, vp, i32, vp]
    lib.dqlb200_eval_greedy.argtypes = [vp, i32, vp, i64, i64, i32, vp, C.POINTER(K.Trace), i32, vp]
    lib.dqlb200_eval_agents.argtypes = [vp, i32, i64, i64, vp, vp, vp]
    lib.dqlb200_eval_pairs.argtypes = [vp, C.POINTER(K.Eval2DParams), vp, i32, i64, i64, vp, vp]
    lib.dqlb200_eval_greedy_2d.argtypes = [vp, C.POINTER(K.Eval2DParams), vp, vp, i64, i64, vp, C.POINTER(K.Trace2D), i32, vp]
    lib.dqlb200_bench_table_rmw.argtypes = [vp, vp, i64, i32, i32, i32, vp, vp]
    lib.dqlb200_train_merged.argtypes = [vp, i32, i32, i32, vp]
    lib.dqlb200_env_reset.argtypes = [vp, i32, C.c_uint32, vp, i32, i32, vp, vp]
    lib.dqlb200_env_step.argtypes = [vp, i32, C.c_uint32, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.dqlb200_agent_select.argtypes = [vp, i32, C.c_uint32, vp, vp, vp]
    lib.dqlb200_agent_update.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.dqlb200_bind_filter_state.argtypes = [vp, vp]
    lib.dqlb200_bind_dynamics_state.argtypes = [vp, vp]
    lib.dqlb200_bench_launch_floor.argtypes = [vp, i32, i32, i32, vp]
    lib.dqlb200_shared_sync_nccl.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, vp]
    lib.dqlb200_transfer.argtypes = [vp, i32, C.c_float, vp]
    lib.dqlb200_check_errors.argtypes = [vp, vp]
    lib.dqlb200_shared_pack.argtypes = [vp, vp, vp]
    lib.dqlb200_shared_apply.argtypes = [vp, vp, vp, i32, i32, vp]
    lib.dqlb200_selftest_discretise.argtypes = [vp, i32, i32, i64, vp, vp, vp]
    lib.dqlb200_mdp_facade_step.argtypes = [vp, i32, i32, i64, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.dqlb200_agent_facade.argtypes = [vp, i32, i64, vp, vp, vp, vp, vp, vp, C.c_double, vp, vp]
    lib.dqlb200_replica_merge.argtypes = [vp, vp, i32, vp]
    lib.dqlb200_bind_merge_snapshot.argtypes = [vp, vp]
    lib.dqlb200_selftest_division.argtypes = [vp, C.POINTER(C.c_uint64), vp]
    if lib.dqlb200_abi_version() != K.ABI_VERSION:
        raise Dqlb200Error("libdqlb200.so ABI version mismatch; rebuild")
    if lib.dqlb200_config_bytes() != C.sizeof(K.Config) or lib.dqlb200_population_state_bytes() != C.sizeof(K.PopulationState):
        raise Dqlb200Error("struct layout mismatch between constants.py and include/dqlb200.h; rebuild")
    if lib.dqlb200_eval2d_params_bytes() != C.sizeof(K.Eval2DParams):
        raise Dqlb200Error("dqlb200_eval2d_params layout mismatch between constants.py and include/dqlb200.h; rebuild")
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        msg = load().dqlb200_last_error().decode("utf-8", "replace")
        if rc == -4:
            raise ValueError(msg)          # the reference raises ValueError for these (PKG/mdp.py:170,353,442-452)
        raise Dqlb200Error(f"libdqlb200 error {rc}: {msg}")
