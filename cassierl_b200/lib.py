"""ctypes binding of libcassie2d.so (include/cassie2d.h).  Fails loudly when the library has
not been built (`python -m cassierl_b200.build`) -- there is no fallback path."""
import ctypes as ct
import os

from .structs import (ControllerForce, ControllerOsc, ControllerPd, ControllerTorque, StateGeneral,
                      StateOperationalSpace)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CASSIE2D_LIB") or os.path.join(_HERE, "lib", "libcassie2d.so")

MODE_TORQUE, MODE_PD, MODE_JACOBIAN, MODE_OSC = 0, 1, 2, 3
TASK_STAND, TASK_IMITATE = 0, 1
AUTO_RESET, FRESH_OBS_ON_RESET, LIVE_QSTATE, TERMINAL_OBS = 1, 2, 4, 8
STATUS_DIVERGED = 3
# include/cassie3d.h
MODE3D_TORQUE, MODE3D_PD = 0, 1
AUTO_RESET_3D, TERMINAL_OBS_3D = 1, 8
OBS_DIM_3D = 45
POLICY_PARAMS_3D = 2868
POLICY_MAX_LAYERS_3D, POLICY_MAX_WIDTH_3D = 4, 256
F32, F64 = 32, 64

# every symbol include/cassie2d.h declares
LEGACY_SYMBOLS = ["Cassie2dInit", "Reset", "StepOsc", "StepTorque", "StepJacobian", "StepPd",
                  "GetGeneralState", "GetOperationalSpaceState", "Display", "Render"]
BATCH_SYMBOLS = ["CassieGetLastError", "Cassie2dBatchInit", "Cassie2dBatchDestroy", "Cassie2dBatchNumEnvs",
                 "Cassie2dBatchPrecision", "Cassie2dBatchDevice", "Cassie2dBatchRealSize", "Cassie2dBatchReset",
                 "Cassie2dBatchSetState", "Cassie2dBatchGetGeneralState", "Cassie2dBatchGetOperationalSpaceState",
                 "Cassie2dBatchStep", "Cassie2dBatchEnvStep", "Cassie2dBatchEnvReset", "Cassie2dBatchSetTrajectory",
                 "Cassie2dBatchSetTrajectoryDetail", "Cassie2dBatchEnvResetSampled",
                 "Cassie2dBatchSquat", "Cassie2dBatchRollout", "Cassie2dBatchDiscountedReturns", "Cassie2dBatchBaselineMoments", "Cassie2dBatchAdvantages", "Cassie2dBatchStepHost", "Cassie2dBatchEnvStepHost", "Cassie2dBatchSquatHost",
                 "Cassie2dBatchGetStats", "Cassie2dBatchGetEpisodeLengths", "Cassie2dBatchSetWarmStart", "Cassie2dBatchGetWarmStart", "Cassie2dBatchSync", "CassieMeasureFp32Peak", "CassieKernelLaunchCount"]

# every symbol include/cassie3d.h declares
BATCH3D_SYMBOLS = ["Cassie3dGetLastError", "Cassie3dBatchCreate", "Cassie3dBatchDestroy", "Cassie3dBatchSizes",
                   "Cassie3dBatchSetLanes", "Cassie3dBatchSetResetState", "Cassie3dBatchGetResetState", "Cassie3dBatchResetAll",
                   "Cassie3dBatchSetState", "Cassie3dBatchGetState", "Cassie3dBatchGetWarmStart", "Cassie3dBatchSetWarmStart",
                   "Cassie3dBatchStep", "Cassie3dBatchStepHost", "Cassie3dBatchGetStats", "Cassie3dBatchGetResets",
                   "Cassie3dBatchSetPdGains", "Cassie3dBatchEnvStep", "Cassie3dBatchEnvStepHost", "Cassie3dBatchEnvReset",
                   "Cassie3dBatchObserve", "Cassie3dBatchGetEpisodeLengths", "Cassie3dBatchRollout", "Cassie3dBatchRolloutMlp",
                   "Cassie3dBatchActionBox",
                   "Cassie3dBatchDiscountedReturns", "Cassie3dBatchBaselineMoments", "Cassie3dBatchAdvantages"]

_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("cassierl_b200: %s is missing -- build it with `python -m cassierl_b200.build` "
                          "(there is no CPU fallback)" % LIB_PATH)
    L = ct.CDLL(LIB_PATH)
    vp, ci, cd = ct.c_void_p, ct.c_int, ct.c_double
    L.CassieGetLastError.restype = ct.c_char_p
    L.Cassie2dBatchInit.restype = vp
    L.Cassie2dBatchInit.argtypes = [ci, ci, ct.c_char_p, ci]
    L.Cassie2dBatchDestroy.restype = None
    L.Cassie2dBatchDestroy.argtypes = [vp]
    for n in ("Cassie2dBatchNumEnvs", "Cassie2dBatchPrecision", "Cassie2dBatchDevice", "Cassie2dBatchRealSize",
              "Cassie2dBatchSync"):
        getattr(L, n).argtypes = [vp]
    L.Cassie2dBatchReset.argtypes = [vp, vp, ct.POINTER(cd), vp]
    L.Cassie2dBatchSetState.argtypes = [vp, vp, vp]
    L.Cassie2dBatchGetGeneralState.argtypes = [vp, vp, vp]
    L.Cassie2dBatchGetOperationalSpaceState.argtypes = [vp, vp, vp]
    L.Cassie2dBatchStep.argtypes = [vp, ci, vp, ci, vp, vp]
    L.Cassie2dBatchEnvStep.argtypes = [vp, ci, ci, vp, ci, ci, vp, vp, vp, vp]
    L.Cassie2dBatchEnvReset.argtypes = [vp, ci, ci, vp, vp]
    L.Cassie2dBatchSetTrajectory.argtypes = [vp, ct.POINTER(cd), ci, cd]
    L.Cassie2dBatchSetTrajectoryDetail.argtypes = [vp, ct.POINTER(cd), ct.POINTER(cd), ci]
    L.Cassie2dBatchEnvResetSampled.argtypes = [vp, ci, ct.c_ulonglong, ct.c_uint, ct.c_uint, vp, vp, vp, vp]
    L.Cassie2dBatchSquat.argtypes = [vp, ci, ci, vp, vp, vp]
    L.Cassie2dBatchDiscountedReturns.argtypes = [vp, vp, vp, vp, cd, ci, vp, vp]
    L.Cassie2dBatchBaselineMoments.argtypes = [vp, ci, vp, vp, vp, vp, ci, vp, vp, vp]
    L.Cassie2dBatchAdvantages.argtypes = [vp, ci, vp, vp, vp, vp, vp, cd, cd, ci, vp, vp, vp]
    L.Cassie2dBatchRollout.argtypes = [vp, ci, ci, vp, ci, ci, ci, ci, ci, ci, ct.c_ulonglong, ct.c_uint, vp, vp, vp, vp, vp, vp]
    L.Cassie2dBatchStepHost.argtypes = [vp, ci, vp, ci, vp]
    L.Cassie2dBatchEnvStepHost.argtypes = [vp, ci, ci, vp, ci, ci, vp, vp, vp]
    L.Cassie2dBatchSquatHost.argtypes = [vp, ci, ci, vp, vp]
    L.Cassie2dBatchGetStats.argtypes = [vp, vp, vp]
    L.Cassie2dBatchSetWarmStart.argtypes = [vp, vp, vp]
    L.Cassie2dBatchGetEpisodeLengths.argtypes = [vp, vp, vp]
    L.Cassie2dBatchGetWarmStart.argtypes = [vp, vp, vp]
    L.CassieMeasureFp32Peak.restype = cd
    L.CassieMeasureFp32Peak.argtypes = [ci]
    L.CassieKernelLaunchCount.restype = ct.c_longlong
    # legacy ABI, declared exactly as rllab/envs/cassie2d.py:25-50 does
    L.Cassie2dInit.argtypes = None
    L.Cassie2dInit.restype = vp
    L.Reset.argtypes = [vp, ct.POINTER(StateGeneral)]
    L.Reset.restype = None
    L.StepOsc.argtypes = [vp, ct.POINTER(ControllerOsc)]
    L.StepOsc.restype = None
    L.StepJacobian.argtypes = [vp, ct.POINTER(ControllerForce)]
    L.StepJacobian.restype = None
    L.StepTorque.argtypes = [vp, ct.POINTER(ControllerTorque)]
    L.StepTorque.restype = None
    L.StepPd.argtypes = [vp, ct.POINTER(ControllerPd)]
    L.StepPd.restype = None
    L.GetGeneralState.argtypes = [vp, ct.POINTER(StateGeneral)]
    L.GetGeneralState.restype = None
    L.GetOperationalSpaceState.argtypes = [vp, ct.POINTER(StateOperationalSpace)]
    L.GetOperationalSpaceState.restype = None
    L.Display.argtypes = [vp, ct.c_bool]
    L.Display.restype = None
    # 3-D batch ABI (include/cassie3d.h)
    i32p, u8p = ct.POINTER(ct.c_int32), ct.POINTER(ct.c_uint8)
    L.Cassie3dGetLastError.restype = ct.c_char_p
    L.Cassie3dBatchCreate.restype = vp
    L.Cassie3dBatchCreate.argtypes = [ct.c_char_p, ci, ci, ci]
    L.Cassie3dBatchDestroy.restype = None
    L.Cassie3dBatchDestroy.argtypes = [vp]
    L.Cassie3dBatchSizes.argtypes = [vp, i32p]
    L.Cassie3dBatchSetLanes.argtypes = [vp, ci]
    L.Cassie3dBatchSetResetState.argtypes = [vp, ct.POINTER(cd), ct.POINTER(cd)]
    L.Cassie3dBatchGetResetState.argtypes = [vp, ct.POINTER(cd), ct.POINTER(cd)]
    L.Cassie3dBatchResetAll.argtypes = [vp, vp, vp]
    L.Cassie3dBatchSetState.argtypes = [vp, vp, vp, vp]
    L.Cassie3dBatchGetState.argtypes = [vp, vp, vp, vp]
    L.Cassie3dBatchGetWarmStart.argtypes = [vp, vp, vp]
    L.Cassie3dBatchSetWarmStart.argtypes = [vp, vp, vp]
    L.Cassie3dBatchStep.argtypes = [vp, vp, ci, cd, ci, vp, vp]
    L.Cassie3dBatchStepHost.argtypes = [vp, vp, ci, cd, ci, vp, vp, vp]
    L.Cassie3dBatchGetStats.argtypes = [vp, vp, vp]
    L.Cassie3dBatchGetResets.argtypes = [vp, vp, vp]
    L.Cassie3dBatchSetPdGains.argtypes = [vp, ct.POINTER(cd), ct.POINTER(cd)]
    L.Cassie3dBatchEnvStep.argtypes = [vp, ci, vp, ci, ci, ci, vp, vp, vp, vp]
    L.Cassie3dBatchEnvStepHost.argtypes = [vp, ci, vp, ci, ci, ci, vp, vp, vp]
    L.Cassie3dBatchEnvReset.argtypes = [vp, vp, vp, vp]
    L.Cassie3dBatchObserve.argtypes = [vp, vp, vp]
    L.Cassie3dBatchGetEpisodeLengths.argtypes = [vp, vp, vp]
    L.Cassie3dBatchRollout.argtypes = [vp, ci, vp, ci, ci, ci, ci, ci, ct.c_ulonglong, ct.c_uint, vp, vp, vp, vp, vp, vp]
    L.Cassie3dBatchRolloutMlp.argtypes = [vp, ci, ci, i32p, vp, ci, ci, ci, ci, ci, ct.c_ulonglong, ct.c_uint, vp, vp, vp, vp,
                                          vp, vp]
    L.Cassie3dBatchActionBox.argtypes = [vp, ci, ct.POINTER(cd), ct.POINTER(cd)]
    L.Cassie3dBatchDiscountedReturns.argtypes = [vp, vp, vp, vp, cd, ci, vp, vp]
    L.Cassie3dBatchBaselineMoments.argtypes = [vp, vp, vp, vp, vp, ci, vp, vp, vp]
    L.Cassie3dBatchAdvantages.argtypes = [vp, vp, vp, vp, vp, vp, cd, cd, ci, vp, vp, vp]
    _lib = L
    return L


def last_error():
    return load().CassieGetLastError().decode()


def check(rc, what):
    if rc != 0:
        raise RuntimeError("libcassie2d %s failed: %s" % (what, last_error()))
