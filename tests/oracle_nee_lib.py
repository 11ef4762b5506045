"""TEST INFRASTRUCTURE: ctypes binding of oracle/liboracle_nee.so, the CPU restatement of next-event estimation
(RTB_INTEGRATOR_PATH_NEE; oracle/oracle_nee.c), built by __graft_entry__.build() next to liboracle.so.

Only tests/ import this module.  The product package never does.
"""
import ctypes as C
import os

import numpy as np

import oracle_lib as ol

ORACLE_NEE_SO = os.path.join(ol.ROOT, "oracle", "liboracle_nee.so")

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(ORACLE_NEE_SO):
            raise RuntimeError(f"{ORACLE_NEE_SO} missing: run __graft_entry__.build()")
        _lib = C.CDLL(ORACLE_NEE_SO)
    return _lib


def render_sum(scene, cam, width, height, samples, dielectric="stochastic", max_depth=5, seed=ol.abi.SCENE_SEED,
               sample_offset=0, threads=None):
    """per-pixel SUM over samples with the NEE estimator (keyed Philox), float64 [H,W,3]; returns
    (sum, (rays, prim_tests, shadow_rays, shadow_hits))"""
    h = ol._holder(scene)
    out = np.zeros((height, width, 3), dtype=np.float64)
    ctr = (C.c_longlong * 4)()
    p = ol.params("philox", dielectric, max_depth, seed, sample_offset, threads)
    lib().oracle_render_sum_nee(ol._dptr(out), h.objects, C.c_size_t(h.n), C.byref(cam), width, height, samples,
                                C.byref(p), ctr)
    return out, (ctr[0], ctr[1], ctr[2], ctr[3])
