"""CPU-side checks of dqlb200_eval_agents_platforms through the bare library, no GPU needed: the dqlb200_platform layout, the
null-handle refusal, and the host-side validation of a platform list."""
import ctypes as C

import numpy as np
import pytest

from dql_multirotor_landing_b200 import _ffi
from dql_multirotor_landing_b200 import constants as K


def test_platform_struct_layout():
    lib = _ffi.load()
    assert lib.dqlb200_platform_bytes() == C.sizeof(K.Platform) == 16
    assert [f for f, _ in K.Platform._fields_] == ["dphase", "r", "rw", "rw2"]
    # the same fields, in the same order, as the platform part of dqlb200_population_params
    assert K.PopulationParams.r.offset - K.PopulationParams.dphase.offset == K.Platform.r.offset - K.Platform.dphase.offset
    assert K.PopulationParams.rw2.offset - K.PopulationParams.dphase.offset == K.Platform.rw2.offset


def test_null_handle_refused_without_gpu():
    lib = _ffi.load()
    pl = (K.Platform * 1)(K.Platform(*K.platform_constants(2.0, 0.8, 22.92, 1)))
    assert lib.dqlb200_eval_agents_platforms(None, 4, 0, 16, pl, 1, None, None) == -1      # DQLB200_ERR_ARG
    assert b"null handle" in lib.dqlb200_last_error()


def test_platform_list_validation():
    pl = K.platform_motions([(2, 0.4), (2.0, 1.6), (3.0, 0.0)])
    assert pl.dtype == np.float64 and pl.shape == (3, 2)
    for bad in ([], [2.0, 0.8], [(2.0, 0.8, 1.0)], [(2.0, float("nan"))], [(float("inf"), 0.8)], [(0.0, 0.8)], [(-1.0, 0.8)],
                [(2.0, -0.1)], [("a", 0.8)], [[(2.0, 0.8)]]):
        with pytest.raises(ValueError):
            K.platform_motions(bad)
