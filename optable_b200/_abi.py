"""ctypes mirror of include/optb.h (constants, structs). Keep in lock-step with the header;
tests/test_abi.py checks sizes and constants against the compiled library."""
import ctypes as C

ABI_VERSION = 8

# geometry kinds
G_GROUP, G_CIRCLE, G_RECT, G_SPHERE, G_ASPHERE, G_CYL, G_POLY2D, G_POLY3D, G_CSG, G_GRID = range(10)
CSG_SUBTRACT, CSG_UNION, CSG_MAX_DEPTH = -1, -2, 30
(GRID_NOUTER, GRID_NINNER, GRID_NEXT, GRID_R, GRID_C00, GRID_NHAT, GRID_UD, GRID_VD, GRID_RHOA, GRID_RHOB, GRID_CELLS) = (
    0, 1, 2, 3, 4, 7, 10, 13, 16, 17, 18)
# interaction kinds
I_NONE, I_MIRROR, I_REFRACT, I_THINLENS, I_ABSORB, I_PASS = range(6)
ROC_INF, ROC_CONST, ROC_ASPHERE_FD = range(3)
ASPH_PARAMETRIC, ASPH_EXACT_SPH = 1, 2

NI_GEOM, NI_INTER, NI_SKIP, NI_AABB, NI_MAT1, NI_MAT2, NI_CAPSLOT, NI_AUX, NI_ROCKIND, NI_LEAF, NI_ORTHO = range(11)
NI_STRIDE = 12
NF_AABB, NF_ORIGIN, NF_TINV, NF_T, NF_P = 0, 6, 9, 18, 27
NF_REFL, NF_TRANS, NF_FOCAL, NF_ROC, NF_CAPMAX, NF_STRIDE = 35, 36, 37, 38, 39, 40
POLY_HEADER = 19
MAT_CONST, MAT_SELLMEIER, MAT_LUT, MF_STRIDE = 0, 1, 2, 8
MON_ORIGIN, MON_TINV, MON_HW, MON_HH, MON_TY, MON_TZ, MON_ORTHO, MON_STRIDE = 0, 3, 12, 13, 14, 17, 20, 24
HIST_BINS = 30

RF_ALIVE, RF_HASQ = 1, 2

(C_SEGMENTS, C_INTERACTIONS, C_HITS, C_TESTS, C_DROPPED, C_STATUS, C_GENERATIONS, C_LAUNCHES, C_TESTS_CURVED,
 C_BOX_TESTS, C_FLAGGED, C_RESERVED) = range(12)
C_COUNT = 12
ST_SEG_OVERFLOW, ST_HIT_OVERFLOW, ST_WORK_OVERFLOW, ST_CAP_ORDER, ST_LUT_MISS = 1, 2, 4, 8, 16
# optb_trace_plan: variant bits of out[0]
PLAN_SMEM, PLAN_SERIAL, PLAN_BOX_SHIFT, PLAN_BOX_MASK = 1, 2, 2, 12
PLAN_ASPH, PLAN_SPLIT, PLAN_FLAG, PLAN_BRENT, PLAN_PASSK, PLAN_SWEEP, PLAN_HIST_SMEM = 16, 32, 64, 128, 256, 512, 1024
AMB_TIE, AMB_APERTURE, AMB_GRAZING, AMB_TIR, AMB_EPS, AMB_SCAN, AMB_SLAB = 1, 2, 4, 8, 16, 32, 64

_vp = C.c_void_p


class SceneDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("n_nodes", C.c_int32), ("n_leaves", C.c_int32),
        ("n_materials", C.c_int32), ("n_monitors", C.c_int32), ("n_capslots", C.c_int32),
        ("n_aux", C.c_int64),
        ("node_i", _vp), ("node_f", _vp), ("mat_kind", _vp), ("mat_f", _vp), ("mon_f", _vp), ("aux", _vp),
    ]


RAY_F64 = ("ox", "oy", "oz", "dx", "dy", "dz", "intensity", "wavelength", "q_re", "q_im",
           "pathlength", "n_medium", "length")


class Rays(C.Structure):
    _fields_ = ([("n", C.c_int64)] + [(k, _vp) for k in RAY_F64] + [("flags", _vp), ("family", _vp)]
                + [("broadcast", C.c_uint32), ("reserved", C.c_uint32)])


class Params(C.Structure):
    _fields_ = [
        ("max_trace_num", C.c_int64), ("unit", C.c_double),
        ("record_segments", C.c_int32), ("record_hits", C.c_int32), ("record_hist", C.c_int32),
        ("chain_len", C.c_int32), ("n_families", C.c_int32), ("caps_slack", C.c_int32),
        ("flag_ambiguity", C.c_int32), ("sorted_rows", C.c_int32),
        ("reference_roots", C.c_int32), ("reserved", C.c_int32),
    ]


SEG_F64 = ("seg_ox", "seg_oy", "seg_oz", "seg_dx", "seg_dy", "seg_dz", "seg_length", "seg_intensity",
           "seg_wavelength", "seg_q_re", "seg_q_im", "seg_pathlength", "seg_n")
SEG_U32 = ("seg_flags", "seg_root", "seg_pop")
SEG_I32 = ("seg_leaf",)
HIT_I32 = ("hit_monitor",)
HIT_U32 = ("hit_root", "hit_pop")
HIT_F64 = ("hit_px", "hit_py", "hit_pz", "hit_intensity", "hit_t", "hit_dx", "hit_dy", "hit_dz",
           "hit_q_re", "hit_q_im")


class Result(C.Structure):
    _fields_ = (
        [("seg_capacity", C.c_int64), ("hit_capacity", C.c_int64)]
        + [(k, _vp) for k in SEG_F64 + SEG_U32 + SEG_I32 + HIT_I32 + HIT_U32 + HIT_F64]
        + [("hit_key", _vp), ("root_flags", _vp)]
        + [("hist_y", _vp), ("hist_yz", _vp), ("cap_counts", _vp), ("counters", _vp)]
    )


EXPORTED_SYMBOLS = (
    "optb_abi_version", "optb_ctx_create", "optb_ctx_destroy", "optb_last_error",
    "optb_scene_upload", "optb_scene_upload_sweep", "optb_scene_upload_sweep_rows", "optb_scene_destroy",
    "optb_scene_update_nodes", "optb_workspace_bytes", "optb_trace",
    "optb_trace_host", "optb_trace_plan", "optb_measure_fp64_peak",
    "optb_sort_workspace_bytes", "optb_sort_rows",
    "optb_monitor_stats_grouped_workspace_bytes", "optb_monitor_stats_grouped",
    "optb_sweep_abcd_workspace_bytes", "optb_sweep_abcd_pivots", "optb_sweep_abcd",
    "optb_comm_unique_id", "optb_comm_init", "optb_monitor_merge", "optb_comm_destroy",
)


class MonitorFrame(C.Structure):
    _fields_ = [("tangent_y", C.c_double * 3), ("tangent_z", C.c_double * 3), ("normal", C.c_double * 3),
                ("half_width", C.c_double), ("half_height", C.c_double)]


(MS_COUNT, MS_SUM_I, MS_SUM_Y, MS_SUM_YY, MS_SUM_Z, MS_SUM_ZZ, MS_SUM_WD, MS_MIN_Y, MS_MAX_Y, MS_MIN_Z, MS_MAX_Z,
 MS_SUM_TY, MS_SUM_TYTY, MS_M2_Y, MS_M2_Z, MS_M2_TY) = range(16)
MS_HIST, MS_STRIDE = 16, 48
