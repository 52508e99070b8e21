"""ctypes mirror of include/lgdsp_b200.h (structs, constants, column names).

Kept in lock-step with the header by tests/test_abi.py, which compiles a tiny C program printing
sizeof/offsetof of every struct and compares them with these definitions.
"""
import ctypes as C

LGDSP_PARAMS_VERSION = 4
LGDSP_MAX_SAMPLES = 8192
LGDSP_MAX_DNI = 64
LGDSP_MAX_DNI_DEG = 3
LGDSP_MAX_SG = 33
LGDSP_MAX_FIR = 4096

LGDSP_OK = 0
LGDSP_ERR_INVALID_ARG = -1
LGDSP_ERR_CUDA = -2
LGDSP_ERR_UNSUPPORTED = -3
LGDSP_ERR_NO_DEVICE = -4
LGDSP_ERR_OOM = -5

GROUP_BASE = 0x01
GROUP_TIMING = 0x02
GROUP_TRAPS = 0x04
GROUP_QDRIFT = 0x08
GROUP_CUSPZAC = 0x10
GROUP_CURRENT = 0x20
GROUP_INTRACE = 0x40
GROUP_ALL = 0x7F
GROUP_PZTRAP = GROUP_BASE | GROUP_TIMING | GROUP_TRAPS
GROUP_LEAN = 0x80
GROUP_PZTRAP_LEAN = GROUP_PZTRAP | GROUP_LEAN

# computed columns of dsp_icpc in the order of /root/reference/src/dsp_icpc.jl:210-229
COLUMNS = (
    "blmean", "blsigma", "blslope", "bloffset",
    "tailmean", "tailsigma", "tailslope", "tailoffset",
    "qc_label",
    "t0", "t10", "t50", "t80", "t90", "t99",
    "t50_current",
    "drift_time",
    "tail_tau", "tail_mean", "tail_sigma",
    "e_max", "e_min",
    "e_10410", "e_535", "e_313",
    "e_10410_inv", "e_313_inv",
    "t0_inv",
    "e_trap", "e_cusp", "e_zac",
    "e_trap_max", "e_cusp_max", "e_zac_max",
    "t_trap_max", "t_cusp_max", "t_zac_max",
    "qdrift", "lq",
    "a_sg", "a_60", "a_100", "a_raw",
    "inTrace_intersect", "inTrace_n",
    "n_sat_low", "n_sat_high", "n_sat_low_cons", "n_sat_high_cons",
)
NCOL = len(COLUMNS)
assert NCOL == 49
COL = {name: i for i, name in enumerate(COLUMNS)}
INT_COLUMNS = ("qc_label", "inTrace_n", "n_sat_low", "n_sat_high", "n_sat_low_cons", "n_sat_high_cons")
# unit of every non-dimensionless column (documentation + Julia wrapper table)
UNITS = {
    "blslope": "1/ns", "tailslope": "1/ns",
    "t0": "us", "t10": "us", "t50": "us", "t80": "us", "t90": "us", "t99": "us", "t50_current": "us",
    "t0_inv": "us", "drift_time": "ns", "tail_tau": "ns",
    "t_trap_max": "ns", "t_cusp_max": "ns", "t_zac_max": "ns", "inTrace_intersect": "ns",
}


class Trap(C.Structure):
    _fields_ = [("navg", C.c_int32), ("ngap", C.c_int32), ("navg2", C.c_int32), ("reserved", C.c_int32)]

    def as_tuple(self):
        return (self.navg, self.ngap, self.navg2)

    @property
    def length(self):
        return self.navg + self.ngap + self.navg2


class Dni(C.Structure):
    _fields_ = [("n_w", C.c_int32), ("degree", C.c_int32),
                ("A", C.c_double * (LGDSP_MAX_DNI * (LGDSP_MAX_DNI_DEG + 1)))]


class Sg(C.Structure):
    _fields_ = [("n_taps", C.c_int32), ("offset", C.c_int32), ("h", C.c_double * LGDSP_MAX_SG)]


class CuspZac(C.Structure):
    _fields_ = [("n_taps", C.c_int32), ("flat", C.c_int32), ("sigma", C.c_double), ("tau", C.c_double),
                ("beta", C.c_double), ("coeffs", C.c_double * LGDSP_MAX_FIR)]


class IcpcParams(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("version", C.c_uint32),
        ("n_samples", C.c_int32), ("groups", C.c_uint32),
        ("t_first_ns", C.c_double), ("dt_ns", C.c_double),
        ("sat_low", C.c_int64), ("sat_high", C.c_int64),
        ("bl_from", C.c_int32), ("bl_until", C.c_int32),
        ("tail_from", C.c_int32), ("tail_until", C.c_int32),
        ("pz_km1", C.c_double),
        ("t0_trap", Trap), ("t0inv_trap", Trap),
        ("t0_threshold", C.c_double),
        ("t0_min_n", C.c_int32), ("tx_min_n", C.c_int32),
        ("tx_frac", C.c_double * 5),
        ("qdrift_first_ns", C.c_double), ("qdrift_last_ns", C.c_double),
        ("lq_first_ns", C.c_double), ("lq_last_ns", C.c_double),
        ("int_dni", Dni), ("sig_dni", Dni),
        ("trap_10410", Trap), ("trap_535", Trap), ("trap_313", Trap), ("trap_e", Trap),
        ("trap_pickoff_ns", C.c_double), ("cusp_pickoff_ns", C.c_double), ("zac_pickoff_ns", C.c_double),
        ("sg", Sg * 3),
        ("cur_from", C.c_int32 * 4), ("cur_until", C.c_int32 * 4),
        ("intrace_nsigma", C.c_double),
        ("intrace_min_n", C.c_int32),
        ("intrace_bl_from", C.c_int32), ("intrace_bl_until", C.c_int32),
        ("cuspzac_direct", C.c_int32), ("reserved0", C.c_int32),
        ("cusp", CuspZac), ("zac", CuspZac),
    ]


class TrapVariant(C.Structure):
    _fields_ = [("trap", Trap), ("pickoff_ns", C.c_double), ("pickoff_mode", C.c_int32), ("reserved", C.c_int32)]


class SweepParams(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("version", C.c_uint32),
        ("n_samples", C.c_int32), ("tx_min_n", C.c_int32),
        ("t_first_ns", C.c_double), ("dt_ns", C.c_double),
        ("bl_from", C.c_int32), ("bl_until", C.c_int32),
        ("pz_km1", C.c_double),
        ("sig_dni", Dni),
        ("out_f64", C.c_int32), ("reserved0", C.c_int32),
    ]


class SweepVariant(C.Structure):
    """lgdsp_sweep_variant: kind 0 trapezoid, 1 FIR (CUSP/ZAC coefficient array), 2 Savitzky-Golay + windowed maximum"""
    _fields_ = [
        ("kind", C.c_int32), ("pickoff_mode", C.c_int32), ("pickoff_ns", C.c_double),
        ("trap", Trap),
        ("n_taps", C.c_int32), ("sg_offset", C.c_int32), ("win_from", C.c_int32), ("win_until", C.c_int32),
        ("coeffs", C.POINTER(C.c_double)),
    ]


# ---- dsp_sipm (include/lgdsp_b200.h: enum lgdsp_sipm_col, lgdsp_sipm_params) ----
SIPM_COLUMNS = ("t_max", "t_min", "t_max_lar", "t_min_lar", "e_max", "e_min", "e_max_lar", "e_min_lar",
                "blmean", "blsigma", "blslope", "bloffset", "wfmean", "wfsigma", "wfslope", "wfoffset",
                "threshold", "threshold_DC", "threshold_trap", "threshold_DC_trap",
                "n_trig", "n_trig_DC", "n_trig_trap", "n_trig_DC_trap")
SIPM_COL = {name: i for i, name in enumerate(SIPM_COLUMNS)}
SIPM_NCOL = len(SIPM_COLUMNS)
SIPM_NLIST, SIPM_NFIELD = 4, 4
SIPM_MAX_TRIGGERS = 1024
SAMPLE_U16, SAMPLE_F32, SAMPLE_F64 = 2, 4, 8


class SipmParams(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("version", C.c_uint32),
        ("n_samples", C.c_int32), ("sample_kind", C.c_int32),
        ("t_first_ns", C.c_double), ("dt_ns", C.c_double),
        ("trunc_from", C.c_int32), ("trunc_until", C.c_int32),
        ("sg", Sg),
        ("sg_min_n", C.c_int32), ("sg_max_n", C.c_int32),
        ("sg_min_thr", C.c_double), ("sg_max_thr", C.c_double), ("sg_nsigma", C.c_double),
        ("sg_min_dc", C.c_double), ("sg_max_dc", C.c_double), ("sg_nsigma_dc", C.c_double),
        ("trap", Trap), ("pz_km1", C.c_double),
        ("trap_min_n", C.c_int32), ("trap_max_n", C.c_int32),
        ("trap_min_thr", C.c_double), ("trap_max_thr", C.c_double), ("trap_nsigma", C.c_double),
        ("trap_min_dc", C.c_double), ("trap_max_dc", C.c_double), ("trap_nsigma_dc", C.c_double),
        ("max_triggers", C.c_int32), ("reserved0", C.c_int32),
    ]


MI_MAX_THR, MI_MAX_HALF = 128, 8


class MultiIntersectParams(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("version", C.c_uint32),
        ("n_samples", C.c_int32), ("n_thresholds", C.c_int32),
        ("t_first_ns", C.c_double), ("dt_ns", C.c_double),
        ("min_n", C.c_int32), ("half_window", C.c_int32), ("degree", C.c_int32), ("rate", C.c_int32),
        ("ratios", C.c_double * MI_MAX_THR),
        ("A", C.c_double * (2 * MI_MAX_HALF * (LGDSP_MAX_DNI_DEG + 1))),
    ]


class SynthParams(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("n_samples", C.c_int32), ("mode", C.c_int32),
                ("noise_sigma", C.c_double), ("tau_samples", C.c_double)]


# ---- per-waveform primitives on waveform arrays (include/lgdsp_b200.h: LGDSP_WFSTAT_*, lgdsp_wfstats_params) ----
WFSTAT_SATURATION = 0x01
WFSTAT_EXTREMESTATS = 0x02
WFSTAT_TAILSTATS = 0x04
WFSTAT_WVF_MAXIMUM = 0x08
WFSTAT_THRESHOLDSTATS = 0x10
WFSTAT_THRESHOLDSTATS_MAD = 0x20
WFSTAT_INTERSECT_MAXIMUM = 0x40
WFSTAT_ALL = 0x7F
WFSTAT_COLUMNS = ("sat_low", "sat_high", "sat_max_cons_low", "sat_max_cons_high", "min", "max", "tmin", "tmax",
                  "tail_mean", "tail_sigma", "tail_tau", "wvf_max", "thr_sigma", "thr_mad", "multiplicity")
WFSTAT_COL = {name: i for i, name in enumerate(WFSTAT_COLUMNS)}
WFSTAT_NCOL = len(WFSTAT_COLUMNS)
WFSTAT_MAX_SAMPLES = 65536
WFSTAT_MAX_TRIGGERS = 65536


class WfstatsParams(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("version", C.c_uint32),
        ("n_samples", C.c_int32), ("sample_kind", C.c_int32),
        ("what", C.c_uint32), ("reserved0", C.c_int32),
        ("t_first_ns", C.c_double), ("dt_ns", C.c_double),
        ("sat_from", C.c_int32), ("sat_until", C.c_int32), ("ext_from", C.c_int32), ("ext_until", C.c_int32),
        ("tail_from", C.c_int32), ("tail_until", C.c_int32), ("max_from", C.c_int32), ("max_until", C.c_int32),
        ("sat_low", C.c_int64), ("sat_high", C.c_int64),
        ("thr_min", C.c_double), ("thr_max", C.c_double),
        ("im_min_n", C.c_int32), ("im_max_n", C.c_int32), ("max_triggers", C.c_int32), ("reserved1", C.c_int32),
    ]
