/*
 * sipnet_gpu.h -- C ABI of the B200 (sm_100a) batched SIPNET integrator.
 *
 * This is the drop-in boundary for ONE path of the reference: the body of the
 * run loop in runModelOutput() (reference src/sipnet/sipnet.c:1963-1982), i.e.
 *
 *     setupModel(); setupEvents();
 *     while (climate != NULL) { updateState(); outputState(...); ... }
 *
 * batched over many (site x parameter-ensemble member) runs.  Everything else
 * of the reference (CLI, sipnet.in, readers, text writers) stays host C and
 * talks to the device only through the entry points below.
 *
 * Conventions
 *  - plain C, plain pointers and sizes; no CUDA or torch types in signatures
 *  - every entry point returns 0 on success or one of the reference's own exit
 *    codes (reference src/common/exitCodes.h:16-27); the library never calls
 *    exit()
 *  - the caller owns every host array passed in; init copies what it needs
 *  - the handle owns all device memory
 *  - there is NO CPU fallback: if no CUDA device is usable init fails with
 *    SIPNET_GPU_ERR_NO_DEVICE
 */
#ifndef SIPNET_GPU_H
#define SIPNET_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SIPNET_GPU_ABI_VERSION 3

/* ---- return codes: reference src/common/exitCodes.h:16-27 ---------------- */
#define SIPNET_GPU_OK 0
#define SIPNET_GPU_ERR_FAILURE 1
#define SIPNET_GPU_ERR_BAD_PARAMETER_VALUE 3 /* e.g. non-positive step length, events.c:460 */
#define SIPNET_GPU_ERR_UNKNOWN_EVENT 4 /* unknown type / irrigation method, events.c:498,736 */
#define SIPNET_GPU_ERR_INPUT_FILE 5 /* event without climate record, events.c:476-481 */
#define SIPNET_GPU_ERR_FILE_OPEN 6
#define SIPNET_GPU_ERR_INTERNAL 7 /* mean-NPP ring overflow, sipnet.c:1562-1569 */
#define SIPNET_GPU_ERR_BAD_CLI 8
#define SIPNET_GPU_ERR_BAD_RESTART 9
/* library specific (outside the reference's range) */
#define SIPNET_GPU_ERR_NO_DEVICE 100 /* no usable CUDA device / CUDA runtime error */
#define SIPNET_GPU_ERR_BAD_ARGUMENT 101 /* NULL pointer, size mismatch, bad step range */

/* ---- model flags: struct Context, reference src/common/context.h:45-56 --- */
#define SIPNET_GPU_NFLAGS 12
typedef struct sipnet_gpu_flags {
  int32_t events;
  int32_t gdd;
  int32_t growthResp;
  int32_t leafWater;
  int32_t litterPool;
  int32_t snow; /* no arithmetic effect in the reference either (SURVEY 8a trap 6) */
  int32_t soilPhenol;
  int32_t waterHResp;
  int32_t nitrogenCycle;
  int32_t anaerobic;
  int32_t flooding;
  int32_t carbonSaturation;
} sipnet_gpu_flags;

/* ---- parameters: struct Parameters, reference src/sipnet/state.h:66-408 ---
 * Same order as the struct, so a maintainer can pass `(double *)&params`.
 * Values are the ones left in `params` by readParamData() (sipnet.c:290-427,
 * i.e. after the TINY floors) and BEFORE setupModel(); the library applies
 * setupModel()'s unit changes / derived values itself (sipnet.c:1858-1951).
 * psnTMax and coarseRootAllocation are derived (input value ignored).
 */
#define SIPNET_GPU_PARAM_LIST(X)                                               \
  X(plantWoodInit) X(laiInit) X(soilInit) X(soilWFracInit) X(aMax)             \
  X(aMaxFrac) X(baseFolRespFrac) X(psnTMin) X(psnTOpt) X(psnTMax)              \
  X(dVpdSlope) X(dVpdExp) X(halfSatPar) X(attenuation) X(leafOnDay)            \
  X(leafOffDay) X(gddLeafOn) X(baseVegResp) X(vegRespQ10) X(baseSoilResp)      \
  X(soilRespQ10) X(waterRemoveFrac) X(wueConst) X(soilWHC) X(leafCSpWt)        \
  X(cFracLeaf) X(woodTurnoverRate) X(waterDrainFrac) X(litterInit)             \
  X(snowInit) X(frozenSoilEff) X(immedEvapFrac) X(fastFlowFrac) X(snowMelt)    \
  X(rdConst) X(rSoilConst1) X(rSoilConst2) X(leafAllocation)                   \
  X(leafTurnoverRate) X(frozenSoilFolREff) X(frozenSoilThreshold)              \
  X(litterBreakdownRate) X(fracLitterRespired) X(fineRootFrac)                 \
  X(coarseRootFrac) X(woodAllocation) X(fineRootAllocation)                    \
  X(coarseRootAllocation) X(fineRootTurnoverRate) X(coarseRootTurnoverRate)    \
  X(baseFineRootResp) X(baseCoarseRootResp) X(fineRootQ10) X(coarseRootQ10)    \
  X(soilTempLeafOn) X(leafGrowth) X(fracLeafFall) X(growthRespFrac)            \
  X(soilRespMoistEffect) X(leafPoolDepth) X(minNInit) X(soilOrgNInit)          \
  X(litterOrgNInit) X(plantStorageNInit) X(nVolatilizationFrac)                \
  X(nLeachingFrac) X(leafCN) X(woodCN) X(fineRootCN) X(kCN)                    \
  X(nFixationFracMax) X(halfNFixationMax) X(leafOnReallocFrac)                 \
  X(leafNResorptionFrac) X(fAnoxia) X(anaerobicDecompRate)                     \
  X(anaerobicTransExp) X(soilMethaneRate) X(litterMethaneRate)                 \
  X(soilCSaturation)

enum sipnet_gpu_param {
#define SIPNET_GPU_X(name) SIPNET_P_##name,
  SIPNET_GPU_PARAM_LIST(SIPNET_GPU_X)
#undef SIPNET_GPU_X
      SIPNET_GPU_NPARAMS /* = 80 = sizeof(Params)/sizeof(double), state.h:410 */
};

/* ---- events: reference src/sipnet/events.h:13-83 -------------------------- */
enum sipnet_gpu_event_type { /* same numeric values as event_type_t, events.h:13-23 */
  SIPNET_EV_FERTILIZATION = 0, /* p = orgN, orgC, minN */
  SIPNET_EV_HARVEST = 1,       /* p = fracRemovedAbove, fracRemovedBelow, fracTransferredAbove, fracTransferredBelow */
  SIPNET_EV_IRRIGATION = 2,    /* p = amountAdded; method 0 canopy, 1 soil */
  SIPNET_EV_PLANTING = 3,      /* p = leafC, woodC, fineRootC, coarseRootC */
  SIPNET_EV_TILLAGE = 4,       /* p = tillageEffect */
  SIPNET_EV_LEAFON = 5,
  SIPNET_EV_LEAFOFF = 6,
  SIPNET_EV_PLANTDEATH = 7     /* computed only; never an input */
};

typedef struct sipnet_gpu_event {
  int32_t year;
  int32_t day;
  int32_t type;   /* enum sipnet_gpu_event_type */
  int32_t method; /* irrigation only */
  double p[4];
} sipnet_gpu_event;

/* ---- one site's forcing + event schedule ----------------------------------
 * Climate arrays hold what readClimData() leaves in the ClimateNode list
 * (reference sipnet.c:205-238, state.h:12-49): par already per day, precip in
 * cm, vpd/vpdSoil/vPress in kPa with the TINY floors, gdd per step.
 * Events are in events.in file order (ascending year, day), as returned by
 * readEventData() (events.h:109).
 */
typedef struct sipnet_gpu_site {
  int64_t nsteps;
  const int32_t *year;
  const int32_t *day;
  const double *time;
  const double *length;
  const double *tair;
  const double *tsoil;
  const double *par;
  const double *precip;
  const double *vpd;
  const double *vpdSoil;
  const double *vPress;
  const double *wspd;
  const double *gdd;
  int64_t nevents;
  const sipnet_gpu_event *events;
  /* optional NEE observations for the log-likelihood output (per step, NaN =
   * no observation); may be NULL */
  const double *nee_obs;
} sipnet_gpu_site;

/* ---- per-step output vector: the columns of outputState(), sipnet.c:453-473 */
enum sipnet_gpu_out_col {
  SIPNET_O_plantWoodC = 0, /* getTotalWoodC() = plantWoodC + plantCAccountingDelta */
  SIPNET_O_plantLeafC,
  SIPNET_O_woodCreation,
  SIPNET_O_soilC,
  SIPNET_O_coarseRootC,
  SIPNET_O_fineRootC,
  SIPNET_O_litterC,
  SIPNET_O_soilWater,
  SIPNET_O_soilWetnessFrac,
  SIPNET_O_snow,
  SIPNET_O_npp,
  SIPNET_O_nee,
  SIPNET_O_cumNEE,
  SIPNET_O_gpp,
  SIPNET_O_rAboveground,
  SIPNET_O_rSoil,
  SIPNET_O_rRoot,
  SIPNET_O_ra,
  SIPNET_O_rh,
  SIPNET_O_rtot,
  SIPNET_O_evapotranspiration,
  SIPNET_O_fluxestranspiration,
  SIPNET_O_minN,
  SIPNET_O_soilOrgN,
  SIPNET_O_litterN,
  SIPNET_O_plantStorageN,
  SIPNET_O_n2o,
  SIPNET_O_nLeaching,
  SIPNET_O_nFixation,
  SIPNET_O_nUptake,
  SIPNET_O_ch4,
  SIPNET_O_nppStorage, /* envi.plantCAccountingDelta */
  SIPNET_GPU_NOUT      /* = 32 */
};

/* Debug dump: every field the reference's --debug-log writes, in file order
 * (debug_log.c:51-170): 13 envi, 56 fluxes, 33 trackers (lastYear as double),
 * 3 phenology trackers, isAlive. */
#define SIPNET_GPU_NDEBUG_ENVI 13
#define SIPNET_GPU_NDEBUG_FLUX 56
#define SIPNET_GPU_NDEBUG_TRACK 33
#define SIPNET_GPU_NDEBUG (13 + 56 + 33 + 3 + 1)
/* With the debug dump the kernel also evaluates the reference's mass-balance tracker (updateBalanceTracker*() and
 * checkBalance(), balance.c:35-148, called from updatePoolsAndBalance(), sipnet.c:1769-1806): two check values per
 * step, balanceTracker.deltaC and deltaN (zeroed below EPS = 1e-8 like the reference's). */
#define SIPNET_GPU_NBALANCE 2

/* ---- computed/applied event records (for the host-side events.out writer) --
 * One record per events.out row (events.c:379-402): the (up to 10) deltas the
 * reference prints, in print order. */
#define SIPNET_GPU_EVREC_NVAL 10
typedef struct sipnet_gpu_event_record {
  int32_t step;   /* index into the site's climate arrays */
  int32_t type;   /* enum sipnet_gpu_event_type */
  int32_t nval;   /* number of valid entries in val[] */
  int32_t variant; /* leafon: 0 = computed (leafOnCreation), 1 = from events.in (eventLeafOnCreation) */
  double val[SIPNET_GPU_EVREC_NVAL];
} sipnet_gpu_event_record;

/* ---- output selection (bit mask) ------------------------------------------ */
#define SIPNET_GPU_OUT_FULL 0x01u    /* [NOUT][steps][M] doubles per run range */
#define SIPNET_GPU_OUT_DEBUG 0x02u   /* [NDEBUG][steps][M] doubles (validation) */
#define SIPNET_GPU_OUT_LOGLIK 0x04u  /* per-member Gaussian NEE log-likelihood */
#define SIPNET_GPU_OUT_MOMENTS 0x08u /* per site, per step ensemble mean+variance of summary_cols */
#define SIPNET_GPU_OUT_QUANTILES 0x10u /* per site, per step ensemble quantiles of summary_cols */
#define SIPNET_GPU_OUT_EVENTS 0x20u  /* per-member event records */

/* ---- arithmetic build selection -------------------------------------------- */
#define SIPNET_GPU_RING_SLOTS_REFERENCE 250
#define SIPNET_GPU_MATH_VALIDATION 0 /* the general kernel: IEEE division, full libm restatement; bit-identical to the
                                        reference's gcc -O0 x86-64 binary */
#define SIPNET_GPU_MATH_FAST 1       /* the optimistic kernel: branch-free main paths of the same arithmetic, members
                                        outside its guards replayed by the general kernel; ALSO bit-identical */
#define SIPNET_GPU_MATH_THROUGHPUT 2 /* tolerance-budgeted: reciprocal-multiply division, -fmad=true model arithmetic;
                                        within 1e-10 relative of the reference (north_star's bound), branch / clamp /
                                        event decisions unchanged on every test ensemble; NOT bit-identical */

typedef struct sipnet_gpu_config {
  int32_t abi_version; /* SIPNET_GPU_ABI_VERSION */
  int32_t device;      /* CUDA device ordinal */
  sipnet_gpu_flags flags;

  int64_t nsites;
  const sipnet_gpu_site *sites;

  int64_t nmembers;
  const int32_t *member_site; /* [nmembers], non-decreasing; NULL => all members on site 0 */
  const double *params;       /* SoA [SIPNET_GPU_NPARAMS][params_ld] */
  int64_t params_ld;          /* leading dimension (>= nmembers) */

  uint32_t outputs;           /* SIPNET_GPU_OUT_* mask */
  int32_t math;               /* SIPNET_GPU_MATH_* */
  int64_t out_steps_capacity; /* max steps per run() kept for FULL/DEBUG/summary gathers; 0 => max site nsteps */

  /* summaries */
  int32_t n_summary_cols;
  const int32_t *summary_cols; /* enum sipnet_gpu_out_col values */
  int32_t n_quantiles;
  const double *quantiles;     /* probabilities in [0,1], any order, repeats allowed; results in this order */
  double nee_sigma;            /* log-likelihood observation sigma (> 0) */

  int32_t max_event_records;   /* per member, for SIPNET_GPU_OUT_EVENTS */
  int32_t block_threads;       /* 0 => library default */
  void *stream;                /* cudaStream_t to launch on; NULL => library-owned stream */
  int32_t ring_slots;          /* slots of the 5-day mean-NPP ring per member.  0 => the smallest ring that cannot
                                  overflow sooner than the reference's (a few slots);
                                  SIPNET_GPU_RING_SLOTS_REFERENCE => the reference's own layout, slot for slot
                                  (MEAN_NPP_MAX_ENTRIES, sipnet.c:40) -- needed when the ring is exchanged with the
                                  reference through a restart checkpoint (restart.c:799-806) */
} sipnet_gpu_config;

typedef struct sipnet_gpu_handle sipnet_gpu_handle;

/* What gather() can return. */
enum sipnet_gpu_gather_what {
  SIPNET_GPU_GATHER_FULL = 1,     /* double [NOUT][n][M], n = steps of the last run() */
  SIPNET_GPU_GATHER_DEBUG = 2,    /* double [NDEBUG][n][M] */
  SIPNET_GPU_GATHER_LOGLIK = 3,   /* double [M] */
  SIPNET_GPU_GATHER_STATUS = 4,   /* uint32 [M] status bits (SIPNET_GPU_ST_*) */
  SIPNET_GPU_GATHER_STATE = 5,    /* double [SIPNET_GPU_NSTATE][M] carried state (restart-shaped) */
  SIPNET_GPU_GATHER_MEAN = 6,     /* double [nsites][n_summary_cols][n] */
  SIPNET_GPU_GATHER_VARIANCE = 7, /* double [nsites][n_summary_cols][n] (population variance) */
  SIPNET_GPU_GATHER_QUANTILES = 8, /* double [nsites][n_summary_cols][n_quantiles][n] */
  SIPNET_GPU_GATHER_EVENT_COUNTS = 9, /* int32 [M] */
  SIPNET_GPU_GATHER_EVENT_RECORDS = 10, /* sipnet_gpu_event_record [M][max_event_records] */
  SIPNET_GPU_GATHER_LOGLIK_N = 11, /* double [M]: number of observations that entered the likelihood */
  SIPNET_GPU_GATHER_RING_VALUES = 12,  /* double [ring_slots][M]: MeanTracker.values, slot-major (runmean.h) */
  SIPNET_GPU_GATHER_RING_WEIGHTS = 13, /* double [ring_slots][M]: MeanTracker.weights */
  SIPNET_GPU_GATHER_BALANCE = 14,      /* double [SIPNET_GPU_NBALANCE][n][M]: deltaC, deltaN of the mass-balance check
                                          (needs SIPNET_GPU_OUT_DEBUG) */
  SIPNET_GPU_GATHER_COUNTERS = 15,     /* uint32 [SIPNET_GPU_NCOUNTERS][M]: how often, since init / reset, the reference
                                          would have printed each of its informational messages for the member
                                          (SIPNET_GPU_CNT_* order; needs SIPNET_GPU_OUT_DEBUG) */
  SIPNET_GPU_GATHER_PARAMS = 16        /* double [SIPNET_GPU_NPARAMS][M]: the device's parameter rows, in device units:
                                          the values after setupModel() -- the nine rates it divides by 365 are per
                                          day, psnTMax and coarseRootAllocation are derived, fAnoxia and
                                          anaerobicDecompRate clamped.  They include resample() copies and
                                          rejuvenate() moves */
};

/* rows of SIPNET_GPU_GATHER_COUNTERS: the status bits say WHETHER, these say HOW OFTEN (validation dump only) */
enum sipnet_gpu_counter {
  SIPNET_GPU_CNT_LEAFON_LIMITED = 0, /* logInfo of checkLeafOnLimitation, limitations.c:48-61 (once per limited step) */
  SIPNET_GPU_CNT_N_LIMITED,          /* logInfo of checkNitrogenLimitation, limitations.c:98-102 */
  SIPNET_GPU_CNT_MINN_LIMITED,       /* mineral-N loss cap applied, limitations.c:119-130 (silent in the reference) */
  SIPNET_GPU_CNT_CLAMPED,            /* logWarning of ensureNonNegative, sipnet.c:1346-1356 (once per clamped stock) */
  SIPNET_GPU_NCOUNTERS
};

/* per-member status bits (instead of the reference's exit()) */
#define SIPNET_GPU_ST_BAD_ALLOCATION 0x1u /* ensureAllocation() failed, sipnet.c:1117-1122 (exit 3) */
#define SIPNET_GPU_ST_RING_OVERFLOW 0x2u  /* mean-NPP tracker out of space, sipnet.c:1562 (exit 7) */
#define SIPNET_GPU_ST_CLAMPED 0x4u        /* a stock went below -EPS and was clamped (warning, sipnet.c:1349) */
#define SIPNET_GPU_ST_DIED 0x8u           /* plant mortality happened at least once (sipnet.c:1702) */
#define SIPNET_GPU_ST_EVREC_OVERFLOW 0x10u /* more event records than max_event_records */
#define SIPNET_GPU_ST_NONFINITE 0x20u     /* a pool became NaN/Inf */
#define SIPNET_GPU_ST_BALANCE 0x80u       /* the mass-balance check found a non-zero deltaC or deltaN on some step (the
                                             reference's warning, balance.c:150-169; debug dump only) */
/* the reference's informational messages / flux caps of limitations.c, once per run and member: */
#define SIPNET_GPU_ST_LEAFON_LIMITED 0x100u /* leaf-on growth reduced by available C / N (limitations.c:46-62) */
#define SIPNET_GPU_ST_N_LIMITED 0x200u      /* plant growth reduced by N limitation (limitations.c:85-114) */
#define SIPNET_GPU_ST_MINN_LIMITED 0x400u   /* leaching + volatilisation capped by the mineral N pool (:119-130) */
#define SIPNET_GPU_ST_REPLAY 0x40u        /* the optimistic kernel met an input outside its guards and the member
                                             was re-run by the general kernel (informational; results are exact) */
#define SIPNET_GPU_ST_ANALYSIS_FLOORED 0x800u /* an assimilation left a pool below 0 and set it to +0.0 */

/* carried state rows for SIPNET_GPU_GATHER_STATE (restart.c:148-308 field list) */
enum sipnet_gpu_state_row {
  SIPNET_S_plantWoodC = 0, SIPNET_S_plantLeafC, SIPNET_S_soilC, SIPNET_S_soilWater,
  SIPNET_S_litterC, SIPNET_S_snow, SIPNET_S_coarseRootC, SIPNET_S_fineRootC,
  SIPNET_S_minN, SIPNET_S_soilOrgN, SIPNET_S_litterN, SIPNET_S_plantStorageN,
  SIPNET_S_plantCAccountingDelta,
  SIPNET_S_gdd, SIPNET_S_soilWetnessFrac, SIPNET_S_yearlyGpp, SIPNET_S_yearlyRtot, SIPNET_S_yearlyRa,
  SIPNET_S_yearlyRh, SIPNET_S_yearlyNpp, SIPNET_S_yearlyNee, SIPNET_S_yearlyLitter,
  SIPNET_S_totGpp, SIPNET_S_totRtot, SIPNET_S_totRa, SIPNET_S_totRh, SIPNET_S_totNpp, SIPNET_S_totNee,
  SIPNET_S_trackersLastYear, SIPNET_S_didLeafGrowth, SIPNET_S_didLeafFall, SIPNET_S_phenLastYear,
  SIPNET_S_dTillMod, SIPNET_S_meanSum, SIPNET_S_meanStart, SIPNET_S_meanLast,
  SIPNET_S_harvestFracRemoved, SIPNET_S_harvestFracTransferred, /* eventTrackers of the last step (restart.c:295-296) */
  SIPNET_GPU_NSTATE
};

/*
 * sipnet_gpu_init -- replaces initModel()+initEvents() hand-off and
 * setupModel()/setupEvents() (reference sipnet.h:26,35; events.h:173,178;
 * sipnet.c:1858-1951; events.c:435).  Validates the configuration (event
 * ordering / climate correspondence as processEvents() would, events.c:471-481,
 * step lengths events.c:460), binds every event to its step, uploads forcing,
 * parameters and schedules, and runs setupModel() for every member on the
 * device.
 */
int sipnet_gpu_init(const sipnet_gpu_config *cfg, sipnet_gpu_handle **out);

/*
 * sipnet_gpu_run -- replaces the `while (climate != NULL) { updateState(); ...}`
 * loop (reference sipnet.c:1969-1982) for steps [step_begin, step_end) of
 * every member.  step_begin must equal the number of steps already run
 * (contiguous segments, like the reference's restart segments,
 * restart.c / testRestartMVP.c:253-297).  Asynchronous: returns after the
 * launch; gather() (or sync()) waits.
 */
int sipnet_gpu_run(sipnet_gpu_handle *h, int64_t step_begin, int64_t step_end);

/*
 * sipnet_gpu_gather -- replaces the per-step side outputs of the loop
 * (outputState sipnet.c:453, writeEventOut events.c:404, outputDebugState
 * debug_log.c:277) by copying device results into a caller buffer.
 * `bytes` must be exactly the size documented at enum sipnet_gpu_gather_what.
 */
int sipnet_gpu_gather(sipnet_gpu_handle *h, int what, void *dst, size_t bytes);

/*
 * sipnet_gpu_run_to_host -- run steps [step_begin, step_end) and deliver the FULL per-step output
 * straight into a host buffer laid out double [NOUT][step_end - step_begin][M], pipelined: the range is
 * integrated in segments of `chunk_steps` (0 => library default) that alternate between the two halves
 * of the device output buffer while a copy stream drains the previous segment (use pinned memory,
 * sipnet_gpu_host_alloc, for the copies to overlap).  Equivalent to run() + gather(FULL) and bit-identical
 * to it; this is the reference loop's `updateState(); outputState();` pair with the device->host copy
 * hidden behind the next segment's arithmetic.  Returns when the data is in `dst`.
 */
int sipnet_gpu_run_to_host(sipnet_gpu_handle *h, int64_t step_begin, int64_t step_end, double *dst, size_t bytes,
                           int64_t chunk_steps);

/* Size in bytes gather(what) will write for the last run range. */
size_t sipnet_gpu_gather_bytes(const sipnet_gpu_handle *h, int what);

/* Block until all queued device work of this handle has finished. */
int sipnet_gpu_sync(sipnet_gpu_handle *h);

/* Reset every member to its post-setupModel() state (step counter back to 0). */
int sipnet_gpu_reset(sipnet_gpu_handle *h);

/*
 * sipnet_gpu_set_state -- overwrite the carried state of every member, the way
 * restartLoadCheckpoint() overwrites the globals after setupModel()+setupEvents()
 * (sipnet.c:1963-1967, restart.c:963-983).  state is [SIPNET_GPU_NSTATE][state_ld]
 * (rows of enum sipnet_gpu_state_row; the layout SIPNET_GPU_GATHER_STATE returns
 * with state_ld = nmembers), ring_values / ring_weights are [ring_slots][ring_ld]
 * (SIPNET_GPU_GATHER_RING_*; both NULL keeps the handle's rings).  The next run()
 * must start at next_step.  The yearly*, tot* (except totNee) and harvestFrac* rows
 * are carried only by handles created with SIPNET_GPU_OUT_DEBUG; they feed
 * nothing back into the model (sipnet.c:1420-1496).
 */
int sipnet_gpu_set_state(sipnet_gpu_handle *h, const double *state, int64_t state_ld, const double *ring_values,
                         const double *ring_weights, int64_t ring_ld, int64_t next_step);

/*
 * Sequential data assimilation: the serial ensemble adjustment Kalman filter (EAKF; Anderson 2001, 2003) on the
 * carried pools, per site, between two run() segments.
 *
 * rows[n_rows] are distinct pool rows SIPNET_S_plantWoodC .. SIPNET_S_plantStorageN (0..11); op[n_obs][n_rows] is the
 * linear observation operator: observation k of member i is y_i = sum_j op[k][j] * x_ji.  value / variance are
 * [nsites][n_obs]; a NaN value means the site has no observation k.
 *
 * A member takes part at its site iff its status has neither SIPNET_GPU_ST_BAD_ALLOCATION nor
 * SIPNET_GPU_ST_NONFINITE and all of its rows are finite; other members are neither read nor written.  For each
 * observation k in order and each site with a finite value y_obs (variance r), over the N members that take part:
 *   ybar, xbar_j = means;  S_yy = sum (y_i - ybar)^2;  S_jy = sum (x_ji - xbar_j)(y_i - ybar)   (two passes)
 *   skipped if N < 2 or S_yy == 0 or S_yy is not finite; otherwise
 *   s2 = S_yy / (N - 1);  ybar_a = ybar + s2 / (s2 + r) * (y_obs - ybar);  alpha = sqrt(r / (s2 + r))
 *   dy_i = (ybar_a - ybar) + (alpha - 1)(y_i - ybar);  x_ji += (S_jy / S_yy) * dy_i
 * Observation k + 1 sees the state observation k left.  After the last one, every value of a member that some
 * observation of the call updated and that is below 0 becomes +0.0, and the member gets
 * SIPNET_GPU_ST_ANALYSIS_FLOORED (sticky; reset() clears it).  Nothing else changes: other state rows, the ring,
 * parameters, log-likelihoods, event records, the last run range's outputs and summaries, the next step.  isAlive is
 * derived from the pools when the next run() starts, so an analysis can revive or end a plant there, exactly as
 * set_state() can.
 *
 * diag (may be NULL) receives double [nsites][n_obs][4] = {N, ybar, s2, ybar_a} per site and observation, taken before
 * that observation's update; N is always filled, the other three are NaN where the pair was skipped or unobserved.
 *
 * Rejected with SIPNET_GPU_ERR_BAD_ARGUMENT, state untouched: NULL pointers; n_rows or n_obs < 1; repeated or other
 * rows; a non-finite op entry or an all-zero op row; an infinite value; a missing, non-finite or non-positive variance
 * where the value is finite.  Every call returns when the update is complete.
 */
typedef struct sipnet_gpu_obs_spec {
  int32_t n_rows;
  const int32_t *rows;     /* pool rows the analysis adjusts */
  int32_t n_obs;
  const double *op;        /* [n_obs][n_rows] */
  const double *value;     /* [nsites][n_obs], NaN = not observed */
  const double *variance;  /* [nsites][n_obs], finite and > 0 where value is finite */
} sipnet_gpu_obs_spec;
int sipnet_gpu_assimilate(sipnet_gpu_handle *h, const sipnet_gpu_obs_spec *obs, double *diag);

/*
 * sipnet_gpu_assimilate() with prior covariance inflation, fixed or adaptive per site (Anderson 2007, 2009).  A
 * forecast without model error loses spread at every analysis; inflating the prior deviations keeps the filter from
 * trusting its ensemble more than the observations.  The caller owns lambda (and lambda_sd) and carries them from
 * call to call; the library keeps no per-site state.
 *
 * Participants and N are the EAKF's (above); lambda0_s is lambda[s] at the start of the call.
 * Prior inflation, once, before observation 0, at every site with lambda0_s finite, != 1 and N >= 2 (observed or not):
 *   xbar_j = (1/N) sum x_ji  (the EAKF's fixed-order sum);  x_ji <- xbar_j + sqrt(lambda0_s) * (x_ji - xbar_j)
 * for every listed row j and participant i.  The EAKF then runs on the inflated state, and an inflated site counts as
 * updated for the final floor (+0.0 and SIPNET_GPU_ST_ANALYSIS_FLOORED).  Other sites are not rewritten.
 * Adaptive update (gamma = 1: a site's state is all local to it), at sites with lambda_sd != NULL, lambda_sd[s] > 0
 * and lambda0_s finite, for every observation k the EAKF applies there (the pair is not skipped), in order, with
 * ybar and s2 of that observation: d = y_obs - ybar, r its variance, sp2 = s2 / lambda0_s (the variance without this
 * call's inflation), lp = lambda[s] and v = lambda_sd[s]^2 (current values), and
 *   g(l) = -(l - lp)^2 / (2v) - log(l sp2 + r) / 2 - d^2 / (2 (l sp2 + r)),
 * the log posterior of lambda under the prior N(lp, v) and the likelihood N(d; 0, l sp2 + r).  g'(l) = 0 is the cubic
 *   2 (l - lp)(sp2 l + r)^2 + v sp2 (sp2 l + r) - v d^2 sp2 = 0.
 *   lambda[s]    <- the argmax of g over [lambda_min, lambda_max] among the cubic's real roots inside it and the two
 *                   bounds (a tie: the smaller l);
 *   lambda_sd[s] <- max(sd_min, min(sd, sqrt(v / (2 D)))) with sd = lambda_sd[s], D = g(l_new) - g(l_new + sd), or
 *                   sd where D <= 0 or D is not finite: the uncertainty never grows.
 * Sites without the update (lambda_sd NULL or 0, lambda NaN, nothing applied) keep the bits of lambda and lambda_sd.
 *
 * diag is sipnet_gpu_assimilate()'s, taken after the inflation.  Rejected with SIPNET_GPU_ERR_BAD_ARGUMENT, nothing
 * changed (state, status, lambda, lambda_sd): whatever sipnet_gpu_assimilate() rejects; a NULL infl or lambda; a
 * lambda[s] neither NaN nor finite and > 0; bounds not finite or not 0 < lambda_min <= lambda_max; sd_min negative or
 * not finite; a lambda_sd[s] NaN, infinite, negative, or > 0 and below sd_min; lambda_sd[s] > 0 with a finite
 * lambda[s] outside [lambda_min, lambda_max].  A call without an inflated site takes sipnet_gpu_assimilate()'s
 * launches; one with some lambda[s] finite and != 1 takes two more.
 */
typedef struct sipnet_gpu_inflation_spec {
  double *lambda;                /* [nsites] in/out; NaN or 1 = no inflation at that site */
  double *lambda_sd;             /* [nsites] in/out, or NULL (all fixed); 0 = fixed at that site */
  double lambda_min, lambda_max; /* bounds of the adaptive estimate */
  double sd_min;                 /* floor of lambda_sd where it is updated */
} sipnet_gpu_inflation_spec;
int sipnet_gpu_assimilate_inflated(sipnet_gpu_handle *h, const sipnet_gpu_obs_spec *obs,
                                   sipnet_gpu_inflation_spec *infl, double *diag);

/*
 * Sequential Monte Carlo: the bootstrap particle filter (Gordon, Salmond & Smith 1993), per site, between two run()
 * segments.  Members of a site are weighted by a log-weight and replaced by copies of well-weighted members, chosen by
 * systematic resampling.  A copy carries its parameters with its pools, so forecast -> resample cycles also filter the
 * parameters.
 *
 * Log-weights: l_i = log_weights[i] (host, [nmembers]) when given, else the handle's log-likelihood (needs
 * SIPNET_GPU_OUT_LOGLIK).  Member i takes part iff its status has neither SIPNET_GPU_ST_BAD_ALLOCATION nor
 * SIPNET_GPU_ST_NONFINITE and l_i is finite (NaN and -inf: not taking part).  For a site of n members, N >= 1 of them
 * taking part, lmax = the largest l_i of the participants:
 *   w_i = exp(l_i - lmax) (glibc-exact exp);  ESS = (sum w)^2 / sum w^2, where both sums are sums of
 *   floor(x * 2^100) in integers, each converted to double (round to nearest) and scaled by 2^-100;
 *   the site is resampled iff u[s] is not NaN and ESS < ess_fraction * n (ess_fraction = INFINITY: always).
 * Ancestors, in integers: W_i = (uint64)(w_i * 2^40) (0 for non-participants); C_i = the exclusive prefix of W in
 * site-local member order; T = sum W; U = floor(u[s] * 2^32); slot k in [0, n) takes
 *   t_k = floor(((k * 2^32 + U) * T) / (n * 2^32))
 * and its ancestor is the i with C_i <= t_k < C_i + W_i.  Ancestors do not decrease with k.  Nothing depends on the
 * order of a sum, so a site gives the same bits in any partition.
 *
 * Every member (slot) of a resampled site, non-participants included, becomes a copy of its ancestor: every device
 * parameter row (nothing is re-derived), the carried state, both mean-NPP ring rows, the status (without internal
 * bits), the event count and records (SIPNET_GPU_OUT_EVENTS) and the message counters (SIPNET_GPU_OUT_DEBUG).  Its
 * log-likelihood and observation count become 0.  Members of other sites, the last run range's outputs and summaries,
 * and the next step do not change.
 *
 * ancestors (may be NULL) receives int64 [nmembers]: the ancestor's member index, -1 where the site was not resampled.
 * diag (may be NULL) receives double [nsites][4] = {N, ESS, lmax + log(sum w / N) (the incremental log-evidence
 * estimate), distinct ancestors (0 where not resampled)}; ESS and the log-evidence are NaN where N = 0.
 *
 * Rejected with SIPNET_GPU_ERR_BAD_ARGUMENT, nothing changed: NULL handle or u; u[s] neither NaN nor in [0, 1);
 * ess_fraction NaN or negative; a +inf log-weight; no log_weights on a handle without a log-likelihood; a site of more
 * than 2^23 members.  Every call returns when the copies are complete.
 */
int sipnet_gpu_resample(sipnet_gpu_handle *h, const double *u, double ess_fraction, const double *log_weights,
                        int64_t *ancestors, double *diag);

/*
 * Parameter rejuvenation after a resample: the kernel-shrinkage move of Liu & West (2001), per site, on listed
 * parameter rows.  Resampling only copies parameter vectors, so after a few cycles a site holds a few distinct ones;
 * this move spreads them again while keeping the site's ensemble mean and covariance (in the transformed space).
 *
 * Units: every value is in device units, i.e. after setupModel() (see SIPNET_GPU_GATHER_PARAMS).  A LOG or LOGIT move
 * is invariant to the 1/365 rescaling up to rounding, and so is an IDENTITY move, because the move is affine.
 *
 * rows[n_rows] (1..16) are distinct SIPNET_P_* rows other than psnTMax and coarseRootAllocation (derived); row j is
 * moved in phi = g_j(theta), transform[j] = SIPNET_GPU_TF_IDENTITY (phi = theta), SIPNET_GPU_TF_LOG (phi = log theta,
 * domain theta > 0) or SIPNET_GPU_TF_LOGIT (phi = log((theta - lo) / (hi - theta)), domain lo < theta < hi with
 * lo = lower[j], hi = upper[j]; lower / upper are read for LOGIT rows only and may be NULL without one).
 * shrink[nsites] is a in (0, 1) per site, NaN = leave the site alone.  z[n_rows][nmembers] (host) are standard normals
 * for the handle's members, supplied by the caller as resample() takes u.
 *
 * Member i takes part at its site iff its status has neither SIPNET_GPU_ST_BAD_ALLOCATION nor SIPNET_GPU_ST_NONFINITE
 * and every listed row is finite and inside its transform's domain.  A site with shrink[s] not NaN and N >= 2
 * participants is moved; with a = shrink[s], h = sqrt(1 - a^2), over the participants:
 *   phi_ij = g_j(theta_ij);  mean_j = (1/N) sum_i phi_ij;
 *   V_jl = (1/N) sum_i (phi_ij - mean_j)(phi_il - mean_l)   (population covariance, two passes)
 *   L: semidefinite Cholesky factor of V in column order: for each j, d = V_jj - sum_{m<j} L_jm^2; if
 *      d > 2^-40 V_jj and V_jj > 2^-80 mean_j^2 then L_jj = sqrt(d) and L_ij = (V_ij - sum_{m<j} L_im L_jm) / L_jj
 *      (i > j), else column j is zero; rank = the number of nonzero columns
 *   phi'_ij = a phi_ij + (1 - a) mean_j + h sum_{m<=j} L_jm z_mi;  theta'_ij = g_j^-1(phi'_ij)
 * The population covariance is what makes the mixture keep the ensemble's mean and covariance exactly.  A member's
 * proposal is rejected -- the member stays bit-identical and counts as kept -- when some theta' is not finite or not
 * inside its domain (the inverse can round onto a bound or underflow to 0), or when the proposed allocation fractions
 * fail ensureAllocation (sipnet.c:1111-1123).  Otherwise the listed rows become theta' and every row setupModel()
 * derives from other rows is derived again exactly as setupModel() does: coarseRootAllocation, psnTMax, the fAnoxia
 * and anaerobicDecompRate clamps, and the library's internal per-member constants.
 *
 * Nothing else changes: status bits, carried state, rings, log-likelihoods, event records, the last run range's
 * outputs and summaries, the next step.  Non-participants and sites left alone are untouched.  A later reset() starts
 * from the moved parameters; set_params() replaces them.
 *
 * diag (may be NULL) receives double [nsites][4] = {N, rank (-1 where the site was left alone), moved, kept}.
 *
 * Rejected with SIPNET_GPU_ERR_BAD_ARGUMENT, nothing changed: NULL handle, spec or arrays; n_rows outside 1..16;
 * a repeated, derived or out-of-range row; an unknown transform; LOGIT bounds that are not finite or with lo >= hi;
 * a shrink neither NaN nor in (0, 1); a non-finite z.  Every call returns when the move is complete.
 */
#define SIPNET_GPU_TF_IDENTITY 0 /* phi = theta */
#define SIPNET_GPU_TF_LOG 1      /* phi = log(theta), domain theta > 0 */
#define SIPNET_GPU_TF_LOGIT 2    /* phi = log((theta - lo) / (hi - theta)), domain lo < theta < hi */
typedef struct sipnet_gpu_jitter_spec {
  int32_t n_rows;              /* 1 .. 16 */
  const int32_t *rows;         /* distinct SIPNET_P_* rows; not psnTMax, not coarseRootAllocation (derived) */
  const int32_t *transform;    /* [n_rows] SIPNET_GPU_TF_* */
  const double *lower, *upper; /* [n_rows] bounds of LOGIT rows (read only for those; may be NULL without one) */
  const double *shrink;        /* [nsites] a in (0, 1); NaN = leave the site alone */
  const double *z;             /* [n_rows][nmembers] standard normals for this handle's members (host) */
} sipnet_gpu_jitter_spec;
int sipnet_gpu_rejuvenate(sipnet_gpu_handle *h, const sipnet_gpu_jitter_spec *spec, double *diag);

/*
 * Parameter calibration: a tempered random-walk Metropolis-Hastings move of listed parameter rows, per site, that
 * re-runs every member over the window [0, s) (s = the next step, s >= 1) and keeps or restores each member's
 * proposal.  It leaves the tempered posterior  p(theta) L(theta)^tau  of each site invariant, so a caller's
 * resample-move loop (temper, resample(), mh_move()) reaches the parameter posterior of a fixed calibration window.
 * L is the step kernel's Gaussian NEE likelihood (SIPNET_GPU_OUT_LOGLIK, nee_sigma).  Units as in rejuvenate().
 *
 * rows, transform, lower, upper: exactly as in sipnet_gpu_jitter_spec (same checks).  prior[j] of row j:
 *   SIPNET_GPU_PRIOR_FLAT    uniform in theta on [prior_a, prior_b] (prior_a < prior_b, either may be infinite: an
 *                            improper flat prior; on a LOGIT row lower <= prior_a and prior_b <= upper)
 *   SIPNET_GPU_PRIOR_NORMAL  normal in phi with mean prior_a (finite) and sd prior_b (finite, > 0): a lognormal
 *                            prior on theta for a LOG row, a logit-normal one for a LOGIT row
 * Its log density in phi (constants dropped): FLAT log|dtheta/dphi| = 0 (IDENTITY), phi (LOG),
 * log((theta - lo)(hi - theta) / (hi - lo)) (LOGIT), and -inf outside [prior_a, prior_b];
 * NORMAL -(phi - prior_a)^2 / (2 prior_b^2).  lp(phi) = sum over the rows.
 * scale[nsites] is the random-walk scale h per site (finite, > 0; NaN = leave the site alone); tempering[nsites] is
 * tau in [0, 1].  current_loglik[nmembers] is the members' log-likelihood over [0, s) (the handle's own is zeroed by
 * resample(), so the caller carries it); z[n_rows][nmembers] standard normals; log_u[nmembers] <= 0 (-inf allowed).
 *
 * Member i takes part at its site iff it would take part in rejuvenate(), current_loglik[i] is finite and lp(phi_i)
 * is finite.  A site with scale[s] not NaN and N >= 2 participants is moved: mean, population covariance V and its
 * semidefinite Cholesky factor L exactly as in rejuvenate(), and
 *   phi'_ij = phi_ij + h sum_{m<=j} L_jm z_mi   (rejuvenate() with a = 1, a symmetric proposal)
 * A proposal is invalid when some theta' is not finite or not inside its domain, fails ensureAllocation, or has
 * lp(phi') = -inf.  Every member with a valid proposal gets theta' and its derived rows (as rejuvenate()); then every
 * member is reset and run over [0, s) (reset(), run(0, s) in pieces of out_steps_capacity when outputs are kept),
 * giving its log-likelihood L'_i.  With
 *   delta_i = tau_s (L'_i - current_loglik[i]) + sum_j [lp_j(phi'_i) - lp_j(phi_i)]   (the tau term is 0 at tau = 0)
 * member i is accepted iff its proposal was valid, L'_i is finite (0 without SIPNET_GPU_OUT_LOGLIK), its status after
 * the run has neither SIPNET_GPU_ST_BAD_ALLOCATION nor SIPNET_GPU_ST_NONFINITE, and log_u[i] < delta_i.  An accepted
 * member keeps what the run produced.  Every other member -- non-participants, sites left alone, invalid and rejected
 * proposals -- gets back, bit for bit, everything it had before the call: parameter rows, state, rings, status, event
 * count and records, message counters, log-likelihood and observation count.
 *
 * Afterwards every member is at step s and there is no last run range: the per-step outputs and summaries of
 * [0, s) are gone, as after reset() (run again to get them).  Only windows that start at step 0 are supported.
 *
 * diag (may be NULL) receives double [nsites][4] = {N, rank (-1 where the site was left alone), invalid, accepted}.
 * A call whose scale is NaN at every site launches nothing and changes nothing; its diag rows are {NaN, -1, 0, 0}.
 *
 * Rejected with SIPNET_GPU_ERR_BAD_ARGUMENT, nothing changed: everything rejuvenate() rejects for rows, transforms
 * and z; NULL spec arrays; an unknown prior or out-of-range prior bounds or sd; a scale neither NaN nor finite > 0;
 * a tempering outside [0, 1]; a log_u entry NaN or > 0; s = 0; tau > 0 at a site with a scale on a handle without
 * SIPNET_GPU_OUT_LOGLIK.  Every call returns when the move is complete.
 */
#define SIPNET_GPU_PRIOR_FLAT 0   /* uniform in theta on [prior_a, prior_b] */
#define SIPNET_GPU_PRIOR_NORMAL 1 /* normal in phi, mean prior_a, sd prior_b */
typedef struct sipnet_gpu_mh_spec {
  int32_t n_rows;               /* 1 .. 16 */
  const int32_t *rows;          /* as sipnet_gpu_jitter_spec */
  const int32_t *transform;     /* [n_rows] SIPNET_GPU_TF_* */
  const double *lower, *upper;  /* [n_rows] bounds of LOGIT rows (read only for those; may be NULL without one) */
  const int32_t *prior;         /* [n_rows] SIPNET_GPU_PRIOR_* */
  const double *prior_a;        /* [n_rows] FLAT: lower bound on theta; NORMAL: mean of phi */
  const double *prior_b;        /* [n_rows] FLAT: upper bound on theta; NORMAL: sd of phi */
  const double *scale;          /* [nsites] random-walk scale h > 0; NaN = leave the site alone */
  const double *tempering;      /* [nsites] tau in [0, 1] */
  const double *current_loglik; /* [nmembers] the members' log-likelihood over [0, s) (host) */
  const double *z;              /* [n_rows][nmembers] standard normals (host) */
  const double *log_u;          /* [nmembers] log of uniforms, <= 0, -inf allowed (host) */
} sipnet_gpu_mh_spec;
int sipnet_gpu_mh_move(sipnet_gpu_handle *h, const sipnet_gpu_mh_spec *spec, double *diag);

/* Slots of the mean-NPP ring this handle uses (config ring_slots, or the automatic choice). */
int32_t sipnet_gpu_ring_slots(const sipnet_gpu_handle *h);

/*
 * sipnet_gpu_set_params -- load a new parameter ensemble into an existing
 * handle (same sites, same member->site map): host->device copy of
 * params[80][ld], setupModel() derivation, state reset.  This is the per-batch
 * entry point of an ensemble / MCMC driver that would otherwise re-run
 * readParamData()+setupModel() per member (sipnet.c:290, 1858).
 */
int sipnet_gpu_set_params(sipnet_gpu_handle *h, const double *params, int64_t params_ld);

/* Replaces cleanupModel() (sipnet.c:2012-2023) for device-side resources. */
void sipnet_gpu_destroy(sipnet_gpu_handle *h);

/* ---- introspection / measurement helpers ----------------------------------- */
/* Device time (ms, CUDA events on the launching stream) of the step kernel(s)
 * of the most recent run(); waits for completion. */
int sipnet_gpu_last_run_ms(sipnet_gpu_handle *h, float *ms);
/* CUDA-event stopwatch on the handle's stream: start() records an event, stop_ms()
 * records a second one, waits for it and returns the device time between them
 * (covers every copy and kernel this handle queued in between). */
int sipnet_gpu_timer_start(sipnet_gpu_handle *h);
int sipnet_gpu_timer_stop_ms(sipnet_gpu_handle *h, float *ms);
/* Number of kernels this library launched since init (all kinds). */
int64_t sipnet_gpu_launch_count(const sipnet_gpu_handle *h);
/* Device pointer of a gatherable buffer (for zero-copy collectives); NULL if absent. */
void *sipnet_gpu_device_ptr(sipnet_gpu_handle *h, int what);
/* Pinned host allocation helpers so gathers run at full PCIe rate. */
void *sipnet_gpu_host_alloc(size_t bytes);
void sipnet_gpu_host_free(void *p);
const char *sipnet_gpu_last_error(void);
int sipnet_gpu_abi_version(void);
/* FP64 FMA issue-rate probe: runs a register-resident DFMA chain on every SM and
 * returns achieved TFLOP/s (the FP64 roofline denominator; SURVEY 7 hard part 7). */
int sipnet_gpu_measure_fp64_peak(int device, double *tflops);

/*
 * Row summaries on caller-owned DEVICE memory: rows[r * ld + j], r < nrows, j < ncols.  For every row:
 * mean / population variance over the finite entries and the requested quantiles (numpy "linear" rule).
 * Used for exact cross-GPU quantiles: after an all-to-all time-transpose each rank holds complete
 * ensembles for its share of the steps and summarises them locally.  d_mean/d_var are [nrows],
 * d_quant is [nq][nrows] (any of them may be NULL); `probs` is a host array of probabilities in [0,1], in any order
 * (row q of d_quant belongs to probs[q]); `stream` a cudaStream_t or NULL.
 * On a non-NULL stream the call only enqueues work (results are ordered on that stream); on the NULL stream it
 * returns when the results are complete.
 */
int sipnet_gpu_rows_summary(int device, const double *d_rows, int64_t nrows, int64_t ncols, int64_t ld,
                            const double *probs, int32_t nq, double *d_mean, double *d_var, double *d_quant,
                            void *stream);

/* Validation hook: evaluate the device exp (op 0: out = exp(x)) or pow (op 1: out = pow(x, y))
 * on host arrays of n doubles, so the device libm can be compared bit for bit with the
 * reference's host libm (glibc) -- see sipnet_b200/csrc/sip_libm.cuh.
 * ops 2..5 evaluate the optimistic policy of the production kernel (sip_num.cuh FastNum): 2 = exp(x),
 * 3 = pow(x, y), 4 = pow(x, y) through the cached log of x, 5 = x / y.  An input outside the policy's guards
 * (the member would be replayed by the general kernel) yields SIPNET_GPU_EVAL_FLAGGED instead of a value.
 * ops 6, 7 evaluate the throughput policy's divisions (ThroughNum): 6 = x / y as one multiplication by the refined
 * reciprocal of y, 7 = x / y of the soil-water balance (the reciprocal plus one residual step); they are flagged by
 * the divisor check only.  op 8 = the refined reciprocal of x itself (y unused, never flagged). */
#define SIPNET_GPU_EVAL_FLAGGED 0x7ff8bad0bad0bad0ull
int sipnet_gpu_eval_libm(int device, int op, const double *x, const double *y, double *out, int64_t n);

/* ---- multi-GPU (SURVEY 8e) ---------------------------------------------------------------------------------------
 * Members are independent (no cross-member term anywhere in updateState(), sipnet.c:1818-1855), so the loop
 * `while (climate) { updateState(); ... }` (sipnet.c:1969-1982) shards trivially: every GPU integrates its share
 * and `run` needs no communication.  NCCL appears only in the final gather of log-likelihoods and of the summaries
 * of a site whose members are spread over GPUs.  NCCL is loaded at run time (libnccl.so.2) by these entry points
 * only.
 *
 * (a) one process per GPU (torchrun, mpirun, ...): each rank creates its handle with ITS members of every site
 *     (all ranks list the same sites; rank order = member order) and joins a team: rank 0 makes the id, the
 *     caller's launcher broadcasts its SIPNET_GPU_COMM_ID_BYTES bytes, every rank calls init_rank (collective).
 */
#define SIPNET_GPU_COMM_ID_BYTES 128
typedef struct sipnet_gpu_comm sipnet_gpu_comm;
int sipnet_gpu_comm_unique_id(void *id);
int sipnet_gpu_comm_init_rank(sipnet_gpu_handle *h, int32_t nranks, int32_t rank, const void *id, sipnet_gpu_comm **out);
void sipnet_gpu_comm_destroy(sipnet_gpu_comm *c); /* before sipnet_gpu_destroy() of the handle */
int32_t sipnet_gpu_comm_nranks(const sipnet_gpu_comm *c);
/* Collective.  Ensemble mean / variance / exact quantiles of the last run range over the members of ALL ranks,
 * into the handle's summary buffers: gather(MEAN / VARIANCE / QUANTILES) and device_ptr() then return the team's
 * result on every rank.  No member value leaves its GPU: per key-bit level the ranks all-reduce 8 KB of histogram
 * per (site, column, step) row (sip_gsum.cuh).  With nranks == 1 the same kernels run without any exchange. */
int sipnet_gpu_comm_summaries(sipnet_gpu_comm *c);
/* Histogram levels the last sipnet_gpu_comm_summaries() needed (diagnostic). */
int32_t sipnet_gpu_comm_last_levels(const sipnet_gpu_comm *c);
/* Collective.  Log-likelihoods of the members of all ranks, rank-major: double [sum of member counts]. */
int sipnet_gpu_comm_gather_loglik(sipnet_gpu_comm *c, double *dst, size_t bytes);
int sipnet_gpu_comm_member_counts(const sipnet_gpu_comm *c, int64_t *counts /* [nranks] */);
/* Collective.  sipnet_gpu_assimilate() over the members of ALL ranks: every rank passes the same spec (a mismatch,
 * found through an all-gathered hash, fails on every rank) and gets the same diag.  Per observation the ranks
 * all-gather per-site partial sums (2 x 128 B per site) and sum them in rank order, so every rank applies identical
 * coefficients; no member value leaves its GPU. */
int sipnet_gpu_comm_assimilate(sipnet_gpu_comm *c, const sipnet_gpu_obs_spec *obs, double *diag);
/* Collective.  sipnet_gpu_assimilate_inflated() over the members of ALL ranks: the same spec and inflation arguments
 * on every rank (lambda, lambda_sd and the three scalars join the compared hash); the ranks also all-gather the
 * inflation's per-site partial sums, and every rank returns the same lambda / lambda_sd bits. */
int sipnet_gpu_comm_assimilate_inflated(sipnet_gpu_comm *c, const sipnet_gpu_obs_spec *obs,
                                        sipnet_gpu_inflation_spec *infl, double *diag);
/* Collective.  sipnet_gpu_resample() over the members of ALL ranks, in site-local order rank by rank: u and
 * ess_fraction are the same on every rank (a mismatch, found through an all-gathered hash, fails on every rank),
 * log_weights holds the rank's own members.  ancestors receives the team's int64 [sum of member counts], rank-major
 * (as sipnet_gpu_comm_gather_loglik); every rank gets the same diag.  The ranks exchange two per-site records, then
 * each source rank sends every destination rank the records of the slots it supplies (NCCL send / receive). */
int sipnet_gpu_comm_resample(sipnet_gpu_comm *c, const double *u, double ess_fraction, const double *log_weights,
                             int64_t *ancestors, double *diag);
/* Collective.  sipnet_gpu_rejuvenate() over the members of ALL ranks: every rank passes the same spec except z, which
 * holds the rank's own members (a mismatch, found through an all-gathered hash of everything but z, fails on every
 * rank); every rank gets the same diag.  The ranks all-gather two per-site partial sums (N and the sums of phi, then
 * the centred cross sums) and add them in rank order, so every rank applies identical coefficients. */
int sipnet_gpu_comm_rejuvenate(sipnet_gpu_comm *c, const sipnet_gpu_jitter_spec *spec, double *diag);
/* Collective.  sipnet_gpu_mh_move() over the members of ALL ranks: current_loglik, z and log_u hold the rank's own
 * members, everything else (and the next step) is the same on every rank (a mismatch, found through an all-gathered
 * hash, fails on every rank); every rank gets the same diag.  The ranks exchange the two moment passes' partial sums
 * as rejuvenate() does and then the integer counts; each rank resets and runs its own members, with no exchange. */
int sipnet_gpu_comm_mh_move(sipnet_gpu_comm *c, const sipnet_gpu_mh_spec *spec, double *diag);

/* (b) one process, one host thread, several GPUs: the single-GPU configuration, partitioned by the library --
 *     whole sites per device when there are at least as many sites as devices, otherwise an even contiguous share
 *     of every site's members per device.  ndevices <= 0: all visible devices; devices == NULL: 0..ndevices-1.
 *     cfg->device and cfg->stream are ignored (a caller stream cannot span devices: rejected if set).
 *     A device that would get no member (fewer members than devices in a site or in a device's site range) is left
 *     out: the team is then smaller than the list.
 *     A list that names ONE device several times (e.g. {0, 0, 0}) forms a loopback team: as many ranks as entries,
 *     all on that device, partitioned as above; the team's collectives are device-to-device copies and a histogram
 *     add instead of NCCL (NCCL does not put two ranks of a communicator on one GPU), and NCCL is not loaded.  It
 *     exists to test the cross-rank select on one GPU; it is no faster than one rank.  A list that repeats a device
 *     and also names others is rejected.
 *     gather() delivers exactly what one GPU would: per-member data in the configuration's member order, summaries
 *     per site (through the team select when a site is split).  This is what `sipnet_gpu --site-list` uses. */
typedef struct sipnet_gpu_multi sipnet_gpu_multi;
int sipnet_gpu_multi_init(const sipnet_gpu_config *cfg, int32_t ndevices, const int32_t *devices, sipnet_gpu_multi **out);
int sipnet_gpu_multi_run(sipnet_gpu_multi *m, int64_t step_begin, int64_t step_end); /* clamped per device to its longest site */
int sipnet_gpu_multi_gather(sipnet_gpu_multi *m, int what, void *dst, size_t bytes);
size_t sipnet_gpu_multi_gather_bytes(const sipnet_gpu_multi *m, int what);
int sipnet_gpu_multi_reset(sipnet_gpu_multi *m);
int sipnet_gpu_multi_sync(sipnet_gpu_multi *m);
int32_t sipnet_gpu_multi_ndevices(const sipnet_gpu_multi *m);
sipnet_gpu_handle *sipnet_gpu_multi_handle(sipnet_gpu_multi *m, int32_t i); /* device i's handle (owned by m) */
/* sipnet_gpu_assimilate() on the whole configuration (value / variance / diag in global site order): split sites go
 * through the team exchange, whole sites are updated by each device alone. */
int sipnet_gpu_multi_assimilate(sipnet_gpu_multi *m, const sipnet_gpu_obs_spec *obs, double *diag);
/* sipnet_gpu_assimilate_inflated() on the whole configuration (lambda / lambda_sd in global site order, as value). */
int sipnet_gpu_multi_assimilate_inflated(sipnet_gpu_multi *m, const sipnet_gpu_obs_spec *obs,
                                         sipnet_gpu_inflation_spec *infl, double *diag);
/* sipnet_gpu_resample() on the whole configuration (u, log_weights, ancestors, diag in configuration order): split
 * sites go through the team exchange, whole sites are resampled by each device alone. */
int sipnet_gpu_multi_resample(sipnet_gpu_multi *m, const double *u, double ess_fraction, const double *log_weights,
                              int64_t *ancestors, double *diag);
/* sipnet_gpu_rejuvenate() on the whole configuration (shrink, z [n_rows][nmembers] and diag in configuration order):
 * split sites go through the team exchange, whole sites are moved by each device alone. */
int sipnet_gpu_multi_rejuvenate(sipnet_gpu_multi *m, const sipnet_gpu_jitter_spec *spec, double *diag);
/* sipnet_gpu_mh_move() on the whole configuration (current_loglik, z [n_rows][nmembers], log_u in configuration
 * order; scale, tempering and diag in global site order), over [0, the multi handle's next step). */
int sipnet_gpu_multi_mh_move(sipnet_gpu_multi *m, const sipnet_gpu_mh_spec *spec, double *diag);
void sipnet_gpu_multi_destroy(sipnet_gpu_multi *m);

#ifdef __cplusplus
}
#endif
#endif /* SIPNET_GPU_H */
