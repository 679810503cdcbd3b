"""ctypes mirror of include/sipnet_gpu.h (struct layouts, enums, constants).

Only data definitions live here -- no compute.  The C header is the source of
truth; tests/test_abi.py checks this mirror against it (sizes, enum values and
exported symbols).
"""
from __future__ import annotations

import ctypes as C

ABI_VERSION = 3
COMM_ID_BYTES = 128

# reference src/common/context.h:45-56
FLAG_NAMES = (
    "events", "gdd", "growthResp", "leafWater", "litterPool", "snow",
    "soilPhenol", "waterHResp", "nitrogenCycle", "anaerobic", "flooding",
    "carbonSaturation",
)
# reference src/common/context.c:35-46
DEFAULT_FLAGS = dict(events=1, gdd=1, growthResp=0, leafWater=0, litterPool=0,
                     snow=1, soilPhenol=0, waterHResp=1, nitrogenCycle=0,
                     anaerobic=0, flooding=0, carbonSaturation=0)

# reference src/sipnet/state.h:66-408 (struct Parameters, in order)
PARAM_NAMES = (
    "plantWoodInit", "laiInit", "soilInit", "soilWFracInit", "aMax",
    "aMaxFrac", "baseFolRespFrac", "psnTMin", "psnTOpt", "psnTMax",
    "dVpdSlope", "dVpdExp", "halfSatPar", "attenuation", "leafOnDay",
    "leafOffDay", "gddLeafOn", "baseVegResp", "vegRespQ10", "baseSoilResp",
    "soilRespQ10", "waterRemoveFrac", "wueConst", "soilWHC", "leafCSpWt",
    "cFracLeaf", "woodTurnoverRate", "waterDrainFrac", "litterInit",
    "snowInit", "frozenSoilEff", "immedEvapFrac", "fastFlowFrac", "snowMelt",
    "rdConst", "rSoilConst1", "rSoilConst2", "leafAllocation",
    "leafTurnoverRate", "frozenSoilFolREff", "frozenSoilThreshold",
    "litterBreakdownRate", "fracLitterRespired", "fineRootFrac",
    "coarseRootFrac", "woodAllocation", "fineRootAllocation",
    "coarseRootAllocation", "fineRootTurnoverRate", "coarseRootTurnoverRate",
    "baseFineRootResp", "baseCoarseRootResp", "fineRootQ10", "coarseRootQ10",
    "soilTempLeafOn", "leafGrowth", "fracLeafFall", "growthRespFrac",
    "soilRespMoistEffect", "leafPoolDepth", "minNInit", "soilOrgNInit",
    "litterOrgNInit", "plantStorageNInit", "nVolatilizationFrac",
    "nLeachingFrac", "leafCN", "woodCN", "fineRootCN", "kCN",
    "nFixationFracMax", "halfNFixationMax", "leafOnReallocFrac",
    "leafNResorptionFrac", "fAnoxia", "anaerobicDecompRate",
    "anaerobicTransExp", "soilMethaneRate", "litterMethaneRate",
    "soilCSaturation",
)
NPARAMS = len(PARAM_NAMES)
assert NPARAMS == 80
P = {n: i for i, n in enumerate(PARAM_NAMES)}

# outputState() columns, reference src/sipnet/sipnet.c:453-473
OUT_NAMES = (
    "plantWoodC", "plantLeafC", "woodCreation", "soilC", "coarseRootC",
    "fineRootC", "litterC", "soilWater", "soilWetnessFrac", "snow", "npp",
    "nee", "cumNEE", "gpp", "rAboveground", "rSoil", "rRoot", "ra", "rh",
    "rtot", "evapotranspiration", "fluxestranspiration", "minN", "soilOrgN",
    "litterN", "plantStorageN", "n2o", "nLeaching", "nFixation", "nUptake",
    "ch4", "nppStorage",
)
NOUT = len(OUT_NAMES)
assert NOUT == 32
O = {n: i for i, n in enumerate(OUT_NAMES)}

# --debug-log field order, reference src/sipnet/debug_log.c:51-170
ENVI_NAMES = (
    "plantWoodC", "plantLeafC", "soilC", "soilWater", "litterC", "snow",
    "coarseRootC", "fineRootC", "minN", "soilOrgN", "litterN",
    "plantStorageN", "plantCAccountingDelta",
)
FLUX_NAMES = (
    "photosynthesis", "leafLitter", "woodLitter", "rVeg", "rSoil", "rain",
    "transpiration", "drainage", "litterToSoil", "rLitter", "snowFall",
    "snowMelt", "sublimation", "immedEvap", "fastFlow", "evaporation",
    "fineRootLoss", "coarseRootLoss", "fineRootCreation",
    "coarseRootCreation", "rCoarseRoot", "rFineRoot", "leafCreation",
    "woodCreation", "leafOnCreation", "leafOnCreationFromWood",
    "nVolatilization", "nLeaching", "nOrgSoil", "nOrgLitter", "nMin",
    "nFixation", "nUptake", "leafOffNResorption", "reductionNResorption",
    "eventLeafC", "eventWoodC", "eventFineRootC", "eventCoarseRootC",
    "eventEvap", "eventSoilWater", "eventSoilC", "eventLitterC", "eventMinN",
    "eventSoilOrgN", "eventLitterN", "eventInputC", "eventOutputC",
    "eventInputN", "eventOutputN", "eventLeafOnCreation",
    "eventLeafOnCreationFromWood", "eventLeafOffLitter",
    "eventLeafOffNResorption", "soilMethane", "litterMethane",
)
TRACKER_NAMES = (
    "gpp", "rtot", "ra", "rh", "rRoot", "rSoil", "rAboveground", "npp", "nee",
    "woodCreation", "gdd", "evapotranspiration", "soilWetnessFrac",
    "yearlyGpp", "yearlyRtot", "yearlyRa", "yearlyRh", "yearlyNpp",
    "yearlyNee", "yearlyLitter", "totGpp", "totRtot", "totRa", "totRh",
    "totNpp", "totNee", "lastYear", "methane", "n2o", "nLeaching",
    "nFixation", "nUptake", "meanNPP",
)
DEBUG_NAMES = (
    tuple("envi." + n for n in ENVI_NAMES)
    + tuple("fluxes." + n for n in FLUX_NAMES)
    + tuple("t." + n for n in TRACKER_NAMES)
    + ("pt.didLeafGrowth", "pt.didLeafFall", "pt.lastYear", "s.isAlive")
)
NDEBUG = len(DEBUG_NAMES)
assert NDEBUG == 106
D = {n: i for i, n in enumerate(DEBUG_NAMES)}

STATE_NAMES = (
    "plantWoodC", "plantLeafC", "soilC", "soilWater", "litterC", "snow",
    "coarseRootC", "fineRootC", "minN", "soilOrgN", "litterN",
    "plantStorageN", "plantCAccountingDelta",
    "gdd", "soilWetnessFrac", "yearlyGpp", "yearlyRtot", "yearlyRa",
    "yearlyRh", "yearlyNpp", "yearlyNee", "yearlyLitter", "totGpp", "totRtot",
    "totRa", "totRh", "totNpp", "totNee", "trackersLastYear", "didLeafGrowth",
    "didLeafFall", "phenLastYear", "dTillMod", "meanSum", "meanStart",
    "meanLast", "harvestFracRemoved", "harvestFracTransferred",
)
S = {n: i for i, n in enumerate(STATE_NAMES)}
RING_SLOTS_REFERENCE = 250   # MEAN_NPP_MAX_ENTRIES, sipnet.c:40
NSTATE = len(STATE_NAMES)

# events.h:13-23
EV_FERTILIZATION, EV_HARVEST, EV_IRRIGATION, EV_PLANTING, EV_TILLAGE, \
    EV_LEAFON, EV_LEAFOFF, EV_PLANTDEATH = range(8)
EVENT_TYPE_BY_NAME = {"fert": EV_FERTILIZATION, "harv": EV_HARVEST,
                      "irrig": EV_IRRIGATION, "plant": EV_PLANTING,
                      "till": EV_TILLAGE, "leafon": EV_LEAFON,
                      "leafoff": EV_LEAFOFF, "plantdeath": EV_PLANTDEATH}
EVENT_NAME_BY_TYPE = {v: k for k, v in EVENT_TYPE_BY_NAME.items()}

OUT_FULL, OUT_DEBUG, OUT_LOGLIK, OUT_MOMENTS, OUT_QUANTILES, OUT_EVENTS = (
    0x01, 0x02, 0x04, 0x08, 0x10, 0x20)
MATH_VALIDATION, MATH_FAST, MATH_THROUGHPUT = 0, 1, 2

(GATHER_FULL, GATHER_DEBUG, GATHER_LOGLIK, GATHER_STATUS, GATHER_STATE,
 GATHER_MEAN, GATHER_VARIANCE, GATHER_QUANTILES, GATHER_EVENT_COUNTS,
 GATHER_EVENT_RECORDS, GATHER_LOGLIK_N, GATHER_RING_VALUES, GATHER_RING_WEIGHTS, GATHER_BALANCE, GATHER_COUNTERS,
 GATHER_PARAMS) = range(1, 17)
TF_IDENTITY, TF_LOG, TF_LOGIT = 0, 1, 2      # sipnet_gpu_jitter_spec transforms

ST_BAD_ALLOCATION, ST_RING_OVERFLOW, ST_CLAMPED, ST_DIED, ST_EVREC_OVERFLOW, \
    ST_NONFINITE, ST_REPLAY = 0x1, 0x2, 0x4, 0x8, 0x10, 0x20, 0x40
ST_BALANCE = 0x80
ST_LEAFON_LIMITED, ST_N_LIMITED, ST_MINN_LIMITED = 0x100, 0x200, 0x400
ST_ANALYSIS_FLOORED = 0x800
NBALANCE = 2
(CNT_LEAFON_LIMITED, CNT_N_LIMITED, CNT_MINN_LIMITED, CNT_CLAMPED, NCOUNTERS) = range(5)   # sipnet_gpu_counter

ERR_NO_DEVICE, ERR_BAD_ARGUMENT = 100, 101
EVREC_NVAL = 10

CLIM_COLS = ("time", "length", "tair", "tsoil", "par", "precip", "vpd",
             "vpdSoil", "vPress", "wspd", "gdd")


class Flags(C.Structure):
    _fields_ = [(n, C.c_int32) for n in FLAG_NAMES]


class Event(C.Structure):
    _fields_ = [("year", C.c_int32), ("day", C.c_int32), ("type", C.c_int32),
                ("method", C.c_int32), ("p", C.c_double * 4)]


class Site(C.Structure):
    _fields_ = (
        [("nsteps", C.c_int64),
         ("year", C.POINTER(C.c_int32)), ("day", C.POINTER(C.c_int32))]
        + [(n, C.POINTER(C.c_double)) for n in CLIM_COLS]
        + [("nevents", C.c_int64), ("events", C.POINTER(Event)),
           ("nee_obs", C.POINTER(C.c_double))]
    )


class EventRecord(C.Structure):
    _fields_ = [("step", C.c_int32), ("type", C.c_int32), ("nval", C.c_int32),
                ("variant", C.c_int32), ("val", C.c_double * EVREC_NVAL)]


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("device", C.c_int32), ("flags", Flags),
        ("nsites", C.c_int64), ("sites", C.POINTER(Site)),
        ("nmembers", C.c_int64), ("member_site", C.POINTER(C.c_int32)),
        ("params", C.POINTER(C.c_double)), ("params_ld", C.c_int64),
        ("outputs", C.c_uint32), ("math", C.c_int32),
        ("out_steps_capacity", C.c_int64),
        ("n_summary_cols", C.c_int32), ("summary_cols", C.POINTER(C.c_int32)),
        ("n_quantiles", C.c_int32), ("quantiles", C.POINTER(C.c_double)),
        ("nee_sigma", C.c_double),
        ("max_event_records", C.c_int32), ("block_threads", C.c_int32),
        ("stream", C.c_void_p),
        ("ring_slots", C.c_int32),
    ]


class ObsSpec(C.Structure):
    """sipnet_gpu_obs_spec: what sipnet_gpu_assimilate() fits the pools to."""
    _fields_ = [
        ("n_rows", C.c_int32), ("rows", C.POINTER(C.c_int32)),
        ("n_obs", C.c_int32), ("op", C.POINTER(C.c_double)),
        ("value", C.POINTER(C.c_double)), ("variance", C.POINTER(C.c_double)),
    ]


class InflationSpec(C.Structure):
    """sipnet_gpu_inflation_spec: the per-site prior inflation of sipnet_gpu_assimilate_inflated() (in/out arrays)."""
    _fields_ = [
        ("lambda_", C.POINTER(C.c_double)), ("lambda_sd", C.POINTER(C.c_double)),
        ("lambda_min", C.c_double), ("lambda_max", C.c_double), ("sd_min", C.c_double),
    ]


class JitterSpec(C.Structure):
    """sipnet_gpu_jitter_spec: which parameter rows sipnet_gpu_rejuvenate() moves, how, and with which normals."""
    _fields_ = [
        ("n_rows", C.c_int32), ("rows", C.POINTER(C.c_int32)), ("transform", C.POINTER(C.c_int32)),
        ("lower", C.POINTER(C.c_double)), ("upper", C.POINTER(C.c_double)),
        ("shrink", C.POINTER(C.c_double)), ("z", C.POINTER(C.c_double)),
    ]
