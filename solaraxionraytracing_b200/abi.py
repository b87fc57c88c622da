"""ctypes mirror of include/sart.h (the C-ABI boundary). Layout is checked against the library at load time
(sart_sizeof_*), so a drift between this file and the header fails loudly."""
from __future__ import annotations

import ctypes as C

ABI_VERSION = 2
SAMPLER_INVERSE_CDF, SAMPLER_ALIAS = 0, 1
MAX_SHELLS = 64
MAX_COATINGS = 8
IMAGE_BINS = 256
MAX_MASSES = 64
COMM_ID_BYTES = 128

# enums (raytracer.nim:16-46, 59-64, 164-167)
ES_CAST, ES_BABYIAXO = 0, 1
TK_LLNL, TK_XMM, TK_CUSTOM_BABYIAXO, TK_ABRIXAS, TK_OTHER = 0, 1, 2, 3, 4
SK_VACUUM, SK_GAS = 0, 1
DK_INGRID2017, DK_INGRID2018, DK_INGRIDIAXO = 0, 1, 2
WY_2017, WY_2018, WY_IAXO = 0, 1, 2
HT_NONE, HT_CROSS, HT_STAR, HT_CIRCLE, HT_SQUARE, HT_DIAMOND = 0, 1, 2, 3, 4, 5
RK_EFFECTIVE_AREA, RK_SINGLE_COATING, RK_MULTI_COATING = 0, 1, 2

EXPERIMENT_KINDS = {"CAST": ES_CAST, "BabyIAXO": ES_BABYIAXO}
TELESCOPE_KINDS = {"LLNL": TK_LLNL, "XMM": TK_XMM, "CustomBabyIAXO": TK_CUSTOM_BABYIAXO, "Abrixas": TK_ABRIXAS,
                   "Other": TK_OTHER}
STAGE_KINDS = {"vacuum": SK_VACUUM, "gas": SK_GAS}
DETECTOR_KINDS = {"InGrid2017": DK_INGRID2017, "InGrid2018": DK_INGRID2018, "InGridIAXO": DK_INGRIDIAXO}
WINDOW_YEAR_NAMES = {WY_2017: "2017", WY_2018: "2018", WY_IAXO: "BabyIAXO"}

# ConfigFlags (raytracer.nim:223-230)
CF_IGNORE_DET_WINDOW = 1 << 0
CF_IGNORE_GAS_ABS = 1 << 1
CF_IGNORE_REFLECTION = 1 << 2
CF_IGNORE_CONV_PROB = 1 << 3
CF_XRAY_TEST = 1 << 4
CF_READ_MAGNET_CONFIG = 1 << 5
CF_READ_DET_INSTALL_CONFIG = 1 << 6

# exit codes
(EXIT_PASSED, EXIT_MISSED_BORE, EXIT_CLIP_EXIT_CB, EXIT_CLIP_PIPE_VT3, EXIT_CLIP_PIPE_XRT, EXIT_OPAQUE,
 EXIT_OUTSIDE_SHELLS, EXIT_GLASS_FRONT, EXIT_NICKEL, EXIT_NO_MIRROR_HIT, EXIT_WINDOW_APERTURE, EXIT_ZERO_WEIGHT,
 EXIT_COLLIMATOR) = range(13)
N_EXIT_CODES = 13
EXIT_NAMES = ["passed", "missed_bore", "clip_exit_cb", "clip_pipe_vt3", "clip_pipe_xrt", "opaque", "outside_shells",
              "glass_front", "nickel", "no_mirror_hit", "window_aperture", "zero_weight", "collimator"]
CODE_MASK = 0xFF
FLAG_PASSED_TILL_WINDOW = 0x100
FLAG_INTERP_CLAMPED = 0x200

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)


class Magnet(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("lengthColdbore", "B", "lengthB", "radiusCB", "pGasRoom", "tGas")]


class Pipes(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("cb2vt3_length", "cb2vt3_radius", "vt3xrt_length", "vt3xrt_radius",
                                          "distanceCBAxisXRTAxis", "pipesTurned")]


class Telescope(C.Structure):
    _fields_ = [("kind", C.c_int32), ("nShells", C.c_int32), ("numberOfHoles", C.c_int32), ("holeType", C.c_int32),
                ("reflKind", C.c_int32), ("nCoatings", C.c_int32), ("layers", C.c_int32 * MAX_COATINGS),
                ("optics_entrance", C.c_double * 3), ("optics_exit", C.c_double * 3),
                ("telescope_turned_x", C.c_double), ("telescope_turned_y", C.c_double),
                ("lMirror", C.c_double), ("holeInOptics", C.c_double),
                ("allThickness", C.c_double * MAX_SHELLS), ("allR1", C.c_double * MAX_SHELLS),
                ("allXsep", C.c_double * MAX_SHELLS), ("allAngles", C.c_double * MAX_SHELLS)]


class TestSource(C.Structure):
    _fields_ = [("active", C.c_int32), ("parallel", C.c_int32)] + [
        (n, C.c_double) for n in ("energy", "distance", "radius", "offAxisUp", "offAxisLeft", "activity", "lengthCol")]


class DetectorInstall(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("distanceDetectorXRT", "distanceWindowFocalPlane", "lateralShift",
                                          "transversalShift")]


class Detector(C.Structure):
    _fields_ = [("windowYear", C.c_int32), ("numberOfStrips", C.c_int32)] + [
        (n, C.c_double) for n in ("stripDistWindow", "stripWidthWindow", "detectorWindowAperture", "theta",
                                  "radiusWindow", "openApertureRatio", "windowThickness", "alThickness", "depthDet")]


class Consts(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("radiusSun", "distanceSunEarth", "roomTemp", "mAxion", "g_agamma",
                                          "chipXMax", "chipYMax", "tesla_to_eV2", "m_to_inv_eV", "exposureFactor")]


class Setup(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("flags", C.c_uint32), ("experiment", C.c_int32), ("stage", C.c_int32),
                ("detectorKind", C.c_int32), ("reserved0", C.c_int32), ("magnet", Magnet), ("pipes", Pipes),
                ("telescope", Telescope), ("testSource", TestSource), ("detectorInstall", DetectorInstall),
                ("detector", Detector), ("consts", Consts)]


class Interp1D(C.Structure):
    _fields_ = [("n", C.c_int32), ("reserved", C.c_int32), ("x", c_double_p), ("y", c_double_p)]


class Tables(C.Structure):
    _fields_ = [("nRadii", C.c_int32), ("nEnergies", C.c_int32), ("energies", c_double_p),
                ("fluxRadiusCDF", c_double_p), ("diffFluxCDFs", c_double_p),
                ("nCoatings", C.c_int32), ("nAngles", C.c_int32), ("nReflEnergies", C.c_int32),
                ("reserved", C.c_int32), ("angleMin", C.c_double), ("angleMax", C.c_double),
                ("reflEnergyMin", C.c_double), ("reflEnergyMax", C.c_double), ("reflectivity", c_double_p),
                ("strongbackTransmission", Interp1D), ("windowTransmission", Interp1D), ("gasAbsorption", Interp1D),
                ("telescopeTransmission", Interp1D)]


RAY_OUT_REQUIRED = ("x", "y", "w", "code", "shell")
RAY_OUT_OPTIONAL = ("energy", "reflect", "transMagnet", "yaw", "alpha1", "alpha2", "pathCB", "r", "deviationDet",
                    "transProbArgon")


class RayOut(C.Structure):
    _fields_ = [("x", c_double_p), ("y", c_double_p), ("w", c_double_p), ("code", c_int32_p), ("shell", c_int32_p)] + [
        (n, c_double_p) for n in RAY_OUT_OPTIONAL]


PASSED_OUT_FIELDS = (("ray", C.c_uint32), ("x", C.c_float), ("y", C.c_float), ("w", C.c_float), ("shell", C.c_uint8),
                     ("energy", C.c_float), ("r", C.c_float), ("reflect", C.c_float), ("transMagnet", C.c_float),
                     ("yaw", C.c_float), ("alpha1", C.c_float), ("alpha2", C.c_float), ("pathCB", C.c_float),
                     ("deviationDet", C.c_float), ("transProbArgon", C.c_float))


class PassedOut(C.Structure):
    _fields_ = [(n, C.POINTER(t)) for n, t in PASSED_OUT_FIELDS]


class Counters(C.Structure):
    _fields_ = [("n_rays", C.c_uint64), ("n_exit", C.c_uint64 * 16), ("n_passed", C.c_uint64),
                ("n_passed_till_window", C.c_uint64), ("n_hit_nickel", C.c_uint64), ("n_interp_clamped", C.c_uint64),
                ("n_retraced", C.c_uint64), ("n_unresolved", C.c_uint64),
                ("sum_w", C.c_double), ("sum_w2", C.c_double), ("sum_x", C.c_double), ("sum_y", C.c_double),
                ("sum_r", C.c_double)]

    def as_dict(self) -> dict:
        d = {"n_rays": int(self.n_rays), "n_passed": int(self.n_passed),
             "n_passed_till_window": int(self.n_passed_till_window), "n_hit_nickel": int(self.n_hit_nickel),
             "n_interp_clamped": int(self.n_interp_clamped), "sum_w": float(self.sum_w), "sum_w2": float(self.sum_w2),
             "sum_x": float(self.sum_x), "sum_y": float(self.sum_y), "sum_r": float(self.sum_r),
             "n_retraced": int(self.n_retraced), "n_unresolved": int(self.n_unresolved)}
        d["n_exit"] = {EXIT_NAMES[i]: int(self.n_exit[i]) for i in range(N_EXIT_CODES)}
        return d


def struct_to_dict(s) -> dict:
    """Recursively converts a ctypes Structure to plain Python (for comparisons in tests)."""
    out = {}
    for name, _ in s._fields_:
        v = getattr(s, name)
        if isinstance(v, C.Structure):
            out[name] = struct_to_dict(v)
        elif isinstance(v, C.Array):
            out[name] = list(v)
        else:
            out[name] = v
    return out


EM_PRIMAKOFF, EM_COMPTON, EM_EE_BREMS, EM_FREE_FREE, EM_IRON57, EM_LONG_PLASMON = (1 << i for i in range(6))
EM_PROCESSES = {"primakoff": EM_PRIMAKOFF, "compton": EM_COMPTON, "ee_brems": EM_EE_BREMS, "free_free": EM_FREE_FREE,
                "iron57": EM_IRON57, "long_plasmon": EM_LONG_PLASMON}

# The exported symbols of libsart.so (every function include/sart.h declares) with their signatures.
H = C.c_void_p
SIGNATURES = {
    "sart_last_error": (C.c_char_p, []),
    "sart_abi_version": (C.c_int, []),
    "sart_sizeof_setup": (C.c_size_t, []),
    "sart_sizeof_tables": (C.c_size_t, []),
    "sart_sizeof_counters": (C.c_size_t, []),
    "sart_device_count": (C.c_int, []),
    "sart_init_setup": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.POINTER(Setup)]),
    "sart_calc_window_vals": (C.c_int, [C.c_double, C.c_int, C.c_double, c_double_p, c_double_p]),
    "sart_create": (C.c_int, [C.POINTER(Setup), C.POINTER(Tables), C.c_int, C.POINTER(H)]),
    "sart_destroy": (None, [H]),
    "sart_update_setup": (C.c_int, [H, C.POINTER(Setup)]),
    "sart_set_axion_masses": (C.c_int, [H, C.c_int, c_double_p]),
    "sart_set_precision": (C.c_int, [H, C.c_int]),
    "sart_has_precision": (C.c_int, [C.c_int]),
    "sart_set_compaction": (C.c_int, [H, C.c_int]),
    "sart_set_retrace": (C.c_int, [H, C.c_int, C.c_double]),
    "sart_stream": (C.c_void_p, [H]),
    "sart_build_cdfs": (C.c_int, [C.c_int, C.c_int, C.c_int, c_double_p, c_double_p, c_double_p, c_double_p,
                                  c_double_p]),
    "sart_emission_rates": (C.c_int, [C.c_int, C.c_int, c_double_p, c_double_p, c_double_p, C.c_int, c_double_p,
                                      C.c_uint32, C.c_double, C.c_double, C.c_double, c_double_p]),
    "sart_trace_presampled": (C.c_int, [H, C.c_size_t, c_double_p, c_double_p, c_double_p, C.POINTER(RayOut)]),
    "sart_trace_presampled_dev": (C.c_int, [H, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RayOut)]),
    "sart_trace_mc_rays": (C.c_int, [H, C.c_uint64, C.c_size_t, C.c_uint64, C.POINTER(RayOut)]),
    "sart_trace_mc_passed": (C.c_int, [H, C.c_uint64, C.c_uint64, C.c_uint64, C.c_size_t, C.POINTER(PassedOut),
                                       C.POINTER(C.c_uint64), C.POINTER(Counters)]),
    "sart_trace_words": (C.c_int, [H, C.c_size_t, C.POINTER(C.c_uint32), C.c_int, C.POINTER(RayOut), c_int32_p]),
    "sart_trace_mc": (C.c_int, [H, C.c_uint64, C.c_uint64, C.c_uint64]),
    "sart_reset_image": (C.c_int, [H]),
    "sart_enable_radial_hist": (C.c_int, [H, C.c_int, C.c_double]),
    "sart_read_radial_hist": (C.c_int, [H, c_double_p, C.POINTER(C.c_uint64)]),
    "sart_enable_spectra": (C.c_int, [H, C.c_int]),
    "sart_read_spectra": (C.c_int, [H, c_double_p, c_double_p, C.POINTER(C.c_uint64), c_double_p, C.POINTER(C.c_uint64)]),
    "sart_image_dev": (C.c_void_p, [H]),
    "sart_image_w2_dev": (C.c_void_p, [H]),
    "sart_counters_dev": (C.c_void_p, [H]),
    "sart_image_len": (C.c_size_t, [H]),
    "sart_read_image": (C.c_int, [H, c_double_p, c_double_p, C.POINTER(Counters)]),
    "sart_synchronize": (C.c_int, [H]),
    "sart_comm_unique_id": (C.c_int, [C.c_char_p]),
    "sart_comm_init_rank": (C.c_int, [H, C.c_int, C.c_int, C.c_char_p]),
    "sart_comm_init_all": (C.c_int, [C.POINTER(H), C.c_int]),
    "sart_comm_destroy": (None, [H]),
    "sart_allreduce": (C.c_int, [C.POINTER(H), C.c_int]),
    "sart_read_merged": (C.c_int, [H, c_double_p, c_double_p, C.POINTER(Counters)]),
    "sart_angular_scan": (C.c_int, [H, C.c_int, c_double_p, C.c_uint64, C.c_uint64, C.c_uint64, c_double_p, C.POINTER(Counters),
                                    c_double_p]),
    "sart_measure_fma_peak": (C.c_int, [C.c_int, C.c_int, c_double_p]),
    "sart_prepare_heatmap": (C.c_int, [H, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_size_t,
                                       c_double_p, c_double_p, c_double_p, C.c_double, c_double_p,
                                       C.POINTER(C.c_uint64)]),
    "sart_ray_uniforms": (None, [C.c_uint64, C.c_uint64, c_double_p]),
    "sart_cdf_thresholds": (None, [c_double_p, C.c_int, C.POINTER(C.c_uint32)]),
    "sart_set_sampler": (C.c_int, [H, C.c_int]),
    "sart_alias_table": (None, [C.POINTER(C.c_uint32), C.c_int, C.POINTER(C.c_uint32)]),
    "sart_error_budgets": (C.c_int, [C.POINTER(Setup), C.c_int, C.c_double, C.c_double, C.c_double, c_double_p, c_double_p,
                                     C.POINTER(C.c_int)]),
    "sart_shell_lookup": (C.c_int, [C.POINTER(Setup), C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "sart_throughput_supported": (C.c_int, [C.POINTER(Setup), C.c_char_p, C.c_int]),
}
