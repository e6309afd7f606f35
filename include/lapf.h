/*
 * liblapf -- C ABI of the B200-native LAPF step-2 hot path.
 *
 * The reference (logan-pearce/olpefit) has no FFI of its own: it is a set of Python
 * scripts whose hot loop calls two in-process functions per Gibbs update,
 *     model = build_analytical_model(parameters_proposal)      apf_step2.py:314 (def :106-124)
 *     chi   = chi_squared(image_nanmask, model_proposal, err)   apf_step2.py:316 (def :134-137)
 * inside `while np.min(total_tries) < accept_min:` (apf_step2.py:300-351).  This header puts
 * the boundary at exactly those two seams: a stateless batched model+chi-square operator and
 * a whole-loop sampler object.  The Python binding a maintainer would add is in INTEGRATION.md.
 *
 * Conventions
 *   - every entry point returns 0 (LAPF_OK) or a negative lapf_status; nothing throws;
 *     lapf_last_error() returns a thread-local description of the last failure;
 *   - all pointers marked "device" are CUDA device pointers owned by the caller
 *     (e.g. torch tensors: tensor.data_ptr()); `stream` is a cudaStream_t passed as void*;
 *   - calls are asynchronous on `stream` unless stated otherwise;
 *   - there is NO CPU fallback: without an sm_100 device every compute call fails.
 *
 * Parameter vectors use the reference layouts, in FRAME pixel coordinates (0-based,
 * x = column, y = row):
 *   2-body, P = 16 (apf_step2.py:108):  xcs ycs xcc ycc dx dy amps ampc ampratio bkgd
 *                                       sigmax sigmay sigmax2 sigmay2 theta theta2
 *   3-body, P = 19 (3body/apf_step2_3body.py:108-109,266-288): xca yca xcb ycb xcc ycc dx dy
 *                                       ampa ampb ampc ampratio bkgd sigmax sigmay sigmax2
 *                                       sigmay2 theta theta2
 */
#ifndef LAPF_H
#define LAPF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LAPF_ABI_VERSION 2
#define LAPF_MAX_PARAMS 19
/* lapf_problem.flags: evaluate every component at every pixel, also where its value is provably
 * below 2^-24 of the floor (default: such far-field rows are skipped; results agree to FP32 rounding) */
#define LAPF_FLAG_NO_CULL 1
/* lapf_problem.flags: always take the plain pixel loop (one exponential per pixel and component)
 * instead of the factorised one (one exponential per 2x4-pixel block and component; DESIGN.md 4).
 * The factorised loop falls back to the plain one by itself for vectors outside its safe range;
 * this switch exists to compare the two. */
#define LAPF_FLAG_PLAIN_LOOP 2

typedef enum lapf_status {
    LAPF_OK = 0,
    LAPF_ERR_INVALID = -1,      /* bad argument / unsupported shape */
    LAPF_ERR_CUDA = -2,         /* a CUDA runtime call failed (see lapf_last_error) */
    LAPF_ERR_NO_DEVICE = -3,    /* no sm_100 device: there is no CPU path */
    LAPF_ERR_NOMEM = -4,
    LAPF_ERR_SELFTEST = -5      /* the batched sampler of this build disagrees with the stateless operator */
} lapf_status;

/* The pixel domain: F frames (epochs), each an ny x nx cut-out ("stamp") or a full frame.
 * Replaces the module-level image_nanmask / err arrays of apf_step2.py:188,210: `weight` is
 * 1/err^2 with 0 on masked pixels, so chi2 = sum weight * (data - model)^2. */
typedef struct lapf_problem {
    int32_t nbody;          /* 2 (apf_step2 / apf_step2a) or 3 (apf_step2_3body) */
    int32_t ny, nx;         /* rows, columns of every frame */
    int32_t n_frames;       /* F */
    int32_t floor_index;    /* parameter slot added as the constant floor: 12 reproduces the
                               reference for both layouts (apf_step2.py:120 -- sigmax2 --
                               and 3body/apf_step2_3body.py:121 -- bkgd) */
    int32_t flags;          /* 0, or LAPF_FLAG_NO_CULL | LAPF_FLAG_PLAIN_LOOP */
    const float* data;      /* device [F][ny][nx]; finite everywhere (0 on masked pixels) */
    const float* weight;    /* device [F][ny][nx] */
    const int32_t* origin;  /* device [F][2]: frame coordinates (x0, y0) of pixel [0][0] */
    const double* outside;  /* device [F][3] or NULL.  When the frames are cut-outs of larger images:
                               sum w, sum w*d, sum w*d^2 over the image pixels OUTSIDE the cut-out.
                               There the reference's model is the constant floor f (the Gaussians
                               are below double rounding), so those pixels add
                               S2 - 2 f S1 + f^2 S0 to chi-square: with this set, chi-square is the
                               reference's whole-frame value (apf_step2.py:94,134-137) at stamp cost */
} lapf_problem;

/* Configuration of a batch of independent walkers (replaces "one MPI rank per walker",
 * apf_step2.py:54-57).  Walker i of this batch has global id id_base + i * id_stride; the
 * random stream of a walker depends only on (seed, global id, update index), so results do
 * not depend on how walkers are sharded over GPUs. */
typedef struct lapf_config {
    lapf_problem problem;
    int64_t n_walkers;
    int64_t id_base, id_stride;
    uint64_t seed;
    const int32_t* frame_of;    /* device [n_walkers] frame index per walker, or NULL (frame 0) */
    const double* init_params;  /* device [n_walkers][P] starting point (apf_step2.py:247-273) */
    const double* widths;       /* HOST [P] jump widths, or NULL for the reference table
                                   (apf_step2.py:234 / 3body:220-238) */
    int64_t burn_in;            /* chain rows are produced once count >= burn_in (apf_step2.py:342) */
    int32_t thin;               /* keep every thin-th row after burn-in (1 = reference) */
    int32_t team_warps;         /* 0 or 1: batched kernel, a warp owns up to 32 walkers (throughput);
                                   4 or 16: that many warps cooperate on ONE walker (latency, for the
                                   reference's 24-64 walkers; 16 needs stamps of 64 or 128 pixels) */
} lapf_config;

typedef struct lapf_sampler lapf_sampler;

int lapf_abi_version(void);
const char* lapf_last_error(void);

/* Number of parameters (16 / 19) for nbody, or a negative status. */
int lapf_num_params(int nbody);
/* Copies the reference jump widths / log10-proposal flags for nbody into out[P]. */
int lapf_default_widths(int nbody, double* widths_out, int32_t* is_log_out);

/* K1 -- build_analytical_model + chi_squared (apf_step2.py:106-137) for B parameter vectors.
 *   params     device [B][P] double
 *   frame_of   device [B] or NULL (all vectors use frame 0)
 *   model_out  device [B][ny][nx] float or NULL
 *   chi2_out   device [B] double or NULL */
int lapf_model_chi2(const lapf_problem* prob, const double* params, int64_t B,
                    const int32_t* frame_of, float* model_out, double* chi2_out, void* stream);

/* K2 -- the sampler loop (apf_step2.py:276-351).  create() copies init_params, evaluates the
 * initial chi-square (apf_step2.py:283-289) and zeroes the try/accept counters (:276). */
int lapf_sampler_create(const lapf_config* cfg, lapf_sampler** out, void* stream);
int lapf_sampler_destroy(lapf_sampler* s);

/* Self-test of the batched sampler (team_warps 0/1), run by lapf_sampler_create unless the
 * environment variable LAPF_NO_SELFTEST is set: three updates of every walker, each one recorded,
 * whose TRIAL chi-squares (apf_step2.py:314-316) are compared bit for bit with lapf_model_chi2 of
 * the same trial vectors; then the sampler is put back exactly as it was (checkpoint round trip).
 * liblapf.so is rebuilt in-tree with whatever nvcc the box has; the sampler kernel keeps its pixels
 * in tensor memory behind `.sync.aligned` loads, and one experimental build of it evaluated the
 * update after every recorded update wrongly while passing every state-based check (DESIGN.md 10).
 * Returns LAPF_ERR_SELFTEST on any difference.  Synchronises the stream. */
int lapf_sampler_selftest(lapf_sampler* s, void* stream);

/* Start a new batch in an existing sampler: new starting points (device [n_walkers][P]) and seed,
 * counters, moments and update count back to zero, initial chi-square re-evaluated against the
 * CURRENT contents of the problem's data/weight buffers (which the caller may have overwritten
 * with new frames of the same shape).  frame_of, widths, burn_in and thin are kept.  Lets a
 * stream of epochs reuse one handle without reallocating device memory. */
int lapf_sampler_reset(lapf_sampler* s, const double* init_params, uint64_t seed, void* stream);

/* Checkpoint / resume.  A walker is (parameters, chi-square, counters, moments, update count; the
 * batch adds its seed and current jump widths) and
 * its random stream is a pure function of (seed, walker id, update count), so a saved blob restores
 * the batch exactly: run(a); save; ...; load; run(b) gives the bits of run(a+b).  The blob is a
 * device buffer of lapf_sampler_checkpoint_bytes() bytes owned by the caller; load() expects a
 * sampler created with the same shape (walkers, model, frame_of) and with the same optional state
 * below enabled the same way before either call (it travels in the blob).  The reference's only resume
 * point is the chain file / step2a.csv (apf_step2.py:248-256).
 *
 * Layout: a head, then one section per kind of state, in this order; a section that is off is absent.
 * A descriptor is 32 bytes, int64 {magic, a, b, c}.
 *   head                  int64 count, int64 seed, double jump widths [LAPF_MAX_PARAMS]
 *   core                  state, shift (lapf_sampler_start), moments, exps, tries, accepts
 *   sketches, if on       no descriptor; walker sums, histograms
 *   batch means, if on    {'LAPFBM01', batch_rows, levels, C}; walker state
 *   draws, if on          {'LAPFRS01', K, P+1, 0}; values, row indices
 *   frame widths, if on   {'LAPFFW01', F, P, 0}; widths, adaptation snapshot
 * load() refuses a blob (LAPF_ERR_INVALID, the sampler unchanged) that is smaller than this sampler's
 * layout, whose head is corrupt, that lacks a descriptor this sampler expects or differs in one, or
 * whose bytes just past this sampler's layout start with a known magic (a section this sampler does
 * not have).  So a blob loads only into a sampler with the same batch means, draws and frame widths.
 * The sketch section has no descriptor: a blob whose sketch setting differs from the sampler's is
 * refused only when that shifts a later descriptor or the blob is too small. */
int64_t lapf_sampler_checkpoint_bytes(const lapf_sampler* s);
int lapf_sampler_save(lapf_sampler* s, void* blob, int64_t blob_bytes, void* stream);
int lapf_sampler_load(lapf_sampler* s, const void* blob, int64_t blob_bytes, void* stream);

/* Replace the jump widths (HOST [P]) for the following runs.  The reference's widths are fixed
 * (apf_step2.py:234); this exists for burn-in-only tuning, which the CLI offers as --adapt.
 * LAPF_ERR_INVALID once per-frame widths are on (lapf_sampler_set_frame_widths). */
int lapf_sampler_set_widths(lapf_sampler* s, const double* widths);

/* Chain rows a run of n_updates starting at the sampler's current count will produce. */
int64_t lapf_sampler_rows_for(const lapf_sampler* s, int64_t n_updates);

/* Advance every walker by n_updates Gibbs updates (one proposed parameter each).
 *   chain_out  device [rows][n_walkers][P+1] double (P parameters then chi-square, the column
 *              order of <rank>_finalarray_mpi.csv, apf_step2.py:346-351), or NULL to record
 *              nothing; rows_cap = capacity in rows (must be >= lapf_sampler_rows_for).  In the
 *              event formats below chain_out must also hold lapf_sampler_chain_bytes bytes. */
int lapf_sampler_run(lapf_sampler* s, int64_t n_updates, void* chain_out, int64_t rows_cap,
                     void* stream);

/* Format of the rows lapf_sampler_run writes to chain_out (default LAPF_CHAIN_F64):
 *   LAPF_CHAIN_F64        double [rows][n_walkers][P+1], the values themselves
 *   LAPF_CHAIN_F32_DELTA  float  [rows][n_walkers][P+1], value minus the walker's starting point
 *                         (lapf_sampler_start): half the bytes that leave the device, and no
 *                         precision lost where it matters -- a chain stays within a few jump
 *                         widths of its start, so the float carries the difference to ~1e-7 of
 *                         itself (positions: 512.3 +- 0.003 would keep only 2e-5 as plain floats).
 * Replaces the text rows of apf_step2.py:346-360 for batches of 10^4 .. 10^6 walkers.
 *
 * Event formats (thin = 1 only: then a row differs from the one before it in at most one parameter
 * and chi-square).  The values are doubles (LAPF_CHAIN_EVENTS_F64) or float differences from the
 * starting point computed exactly as LAPF_CHAIN_F32_DELTA does (LAPF_CHAIN_EVENTS_F32_DELTA).  With
 * e = 8 or 4 bytes per value, a run that records R rows of W walkers writes one contiguous buffer:
 *   key     e * [W][P+1]   row 0 of this run, byte for byte what the dense format writes as row 0
 *   codes   uint8 [R][W], padded with zeros to a multiple of 16 bytes: bits 0-4 = k, the parameter
 *           drawn for the update of row r; bit 7 = that update was accepted
 *   values  e * [R][W]     column k of row r after accept / reject (the old value when rejected)
 *   chi     e * [R][W]     chi-square column of row r
 * Row r is row r-1 with row[k] = value and row[P] = chi (row -1 = key).  Event 0 repeats the key on
 * purpose: the codes are then a trace of every recorded update (with burn_in = 0 they count exactly
 * the tries and accepts of lapf_sampler_state).  Every byte is written: equal runs, equal buffers. */
#define LAPF_CHAIN_F64 0
#define LAPF_CHAIN_F32_DELTA 1
#define LAPF_CHAIN_EVENTS_F64 2
#define LAPF_CHAIN_EVENTS_F32_DELTA 3
/* LAPF_ERR_INVALID for an event format on a sampler with thin != 1 (lapf_sampler_run checks again). */
int lapf_sampler_set_chain_format(lapf_sampler* s, int32_t format);
/* Bytes the next lapf_sampler_run of n_updates writes to chain_out in the current format: dense
 * formats rows * W * (P+1) * e, event formats the layout above (0 when the run records no row). */
int64_t lapf_sampler_chain_bytes(const lapf_sampler* s, int64_t n_updates);
/* The starting point of every walker and its chi-square: start_out device double [n_walkers][P+1]
 * (the reference point of LAPF_CHAIN_F32_DELTA rows and of the running moments). */
int lapf_sampler_start(lapf_sampler* s, double* start_out, void* stream);

/* Current state: state_out device [n_walkers][P+1] double; counters device [n_walkers][P]
 * uint32 each (total_tries / total_accept of apf_step2.py:276,304,323).  Any may be NULL. */
int lapf_sampler_state(lapf_sampler* s, double* state_out, uint32_t* tries_out,
                       uint32_t* accepts_out, void* stream);

/* K4 -- batch statistics, written to device memory:
 *   totals_out  device int64[2P+2]: sum over walkers of tries[P], accepts[P], then the minimum
 *               over walkers and parameters of tries (stop rule of apf_step2.py:300, globalised),
 *               then the number of component evaluations (pixels x Gaussian components) the
 *               sampler really did so far (what is left of ny*nx*K per update after far-field
 *               culling; roofline accounting)
 *   moments_out device double[F][P+1][4] or NULL: per frame and column, over that frame's
 *               walkers and the rows recorded so far: a reference value r, sum of (chain mean - r),
 *               sum of (chain mean - r)^2, sum of chain variances -- the ingredients of the
 *               Gelman-Rubin statistic (apf_step3.py:265-276), centred so nothing cancels
 *   counts_out  device int64[F+1] or NULL: walkers per frame, then rows recorded per walker */
int lapf_sampler_stats(lapf_sampler* s, int64_t* totals_out, double* moments_out,
                       int64_t* counts_out, void* stream);

/* K4b -- separation / position angle of the recorded rows without the chain (apf_step3.py:255-256,
 * 283-291: sep = sqrt(dx^2 + dy^2), pa = degrees(atan2(-dx, dy)) of each companion relative to the
 * first object; 3-body: both pairs, 3body/apf_step3_3body.py:273-276,318-324; medians and standard
 * deviations are what :436-437 report).  Once enabled, every recorded row of every walker enters,
 * per frame and companion, two fixed-width histograms (separation in PIXELS, position angle in
 * degrees; n_bins bins centred on a per-frame centre value, plus an underflow and an overflow bin)
 * and the walker's running sums.  Histograms are integer counts: they add up exactly over walkers
 * and over GPUs (all-reduce them; give every rank the same centres).
 *   centers    device double [F][nbody-1][2] (separation, position angle) or NULL: the starting
 *              point of the first walker of each frame in THIS batch
 * Enable before the first lapf_sampler_run; lapf_sampler_reset zeroes the sketches. */
int lapf_sampler_sketch_enable(lapf_sampler* s, int32_t n_bins, double sep_bin_pixels, double pa_bin_degrees,
                               const double* centers, void* stream);
/*   hist_out     device uint32 [F][nbody-1][2][n_bins+2] or NULL (bin 0: below range, bin n_bins+1: above / nan)
 *   summary_out  device double [F][nbody-1][2][4] or NULL: centre, sum of (value - centre), sum of
 *                (value - centre)^2, number of values (position-angle differences wrapped to +-180) */
int lapf_sampler_sketch(lapf_sampler* s, uint32_t* hist_out, double* summary_out, void* stream);

/* K4c -- batch means of the recorded rows without the chain: the ingredients of a Monte Carlo standard
 * error and an effective sample size for every walker (DESIGN.md, "Batch means").  Quantity c < P+1 is
 * chain column c minus the walker's starting point (what the running moments add up); if sketches were
 * enabled before, quantities P+1 + 2(o-1) + q follow, the separation (q = 0) and position angle (q = 1)
 * of companion o minus the frame's sketch centre, exactly as the sketch sums add them: C quantities.
 * Every walker keeps, per quantity and level l < levels, two doubles: snap, its running sum M1 at the
 * last row count that is a multiple of b_l = batch_rows * 2^l (the sum of its complete level-l batches),
 * and s2, the sum of the squared sums of those batches.  A row that brings the walker's recorded-row
 * count to a multiple of b_l does S = M1 - snap; s2 = s2 + S*S; snap = M1 (rounded to nearest, never
 * fused); rows that close no batch cost nothing more.  The state depends neither on how runs are split
 * into launches nor on the chain format.
 * Batch means of every recorded value at batch lengths batch_rows * 2^l rows, l < levels
 * (1 <= batch_rows <= 2^30, 1 <= levels <= 24).  LAPF_ERR_INVALID once any row has been recorded.  Runs
 * lapf_sampler_selftest with the batch means active (unless LAPF_NO_SELFTEST) and leaves the sampler as
 * it was.  Once they are on, lapf_sampler_sketch_enable returns LAPF_ERR_INVALID (C would change);
 * lapf_sampler_reset zeroes them; checkpoints carry them (see lapf_sampler_save for the layout and the
 * load rule). */
int lapf_sampler_batchmeans_enable(lapf_sampler* s, int32_t batch_rows, int32_t levels, void* stream);
/*   walker_out device double [W][C][levels][2] (snap, s2) or NULL
 *   frame_out  device double [F][C][1 + levels] or NULL: [0] sum over the frame's walkers of the
 *              population variance of their recorded values (np.std()**2), [1+l] sum over the frame's
 *              walkers of the sample variance of their level-l batch means, each
 *              (s2 - snap^2 / J) / (b_l^2 (J - 1)) with J = rows / b_l complete batches (0 where J < 2).
 *              Sums over walkers: all-reduce them over GPUs like the moments. */
int lapf_sampler_batchmeans(lapf_sampler* s, double* walker_out, double* frame_out, void* stream);

/* K4d -- posterior draws: a uniformly random sample of K recorded rows per walker, kept on the device
 * (DESIGN.md, "Posterior draws").  Reservoir sampling (algorithm R) over the rows the moments see (after
 * burn-in and thinning, with or without chain_out): walker row n (0 for the first recorded row, counted
 * across launches) fills slot n if n < K; otherwise it replaces slot j = mulhi64(r, n + 1) if j < K, where
 * r = r0 | r1 << 32 of philox4x32_10(counter = (n low, n high, seed high, 'LAPR'), key = (seed low, walker
 * id)), the walker id of make_draw (id_base + w * id_stride).  The selection depends on (seed, walker id, n)
 * only; the update stream is untouched.  mulhi64 without rejection biases j by at most (n + 1) / 2^64.
 * A slot holds the row's P+1 values (state after accept / reject, chain column order, frame coordinates)
 * and n; an empty slot has n = -1 and all-ones (NaN) values.  Memory W * K * (P + 2) * 8 bytes.
 * 1 <= per_walker <= 65536.  LAPF_ERR_INVALID once any row has been recorded, or if draws are already on.
 * Independent of sketches and batch means, in either order.  Runs lapf_sampler_selftest with the reservoir
 * active and one slot (unless LAPF_NO_SELFTEST), so that self-test rows 1 and 2 replace slot 0, and leaves
 * the sampler as it was.  lapf_sampler_reset empties the reservoir; checkpoints carry it (see
 * lapf_sampler_save for the layout and the load rule). */
int lapf_sampler_draws_enable(lapf_sampler* s, int32_t per_walker, void* stream);
/*   values_out device double [W][K][P+1] or NULL; rows_out device int64 [W][K] or NULL */
int lapf_sampler_draws(lapf_sampler* s, double* values_out, int64_t* rows_out, void* stream);

/* K4e -- per-frame jump widths, tuned on the device (DESIGN.md, "Per-epoch jump widths").  Epochs differ in
 * flux, seeing and Strehl, so one width vector cannot suit them all.  Once on, the proposal of a walker of
 * frame f reads widths[f][k] instead of the batch's widths[k]; widths change only between runs.
 *   widths  HOST double [F][P], or NULL: the batch widths (lapf_sampler_set_widths / the config) in every row.
 * The first call allocates the table and an adaptation snapshot (int64 [F][P][2], zero) and runs
 * lapf_sampler_selftest with the table active (unless LAPF_NO_SELFTEST); later calls replace the widths and
 * keep the snapshot.  Widths that are negative or not finite give LAPF_ERR_INVALID.  While the table is on,
 * lapf_sampler_set_widths returns LAPF_ERR_INVALID (one source of truth).  lapf_sampler_reset keeps the
 * widths and zeroes the snapshot, because the counters start again.  Checkpoints carry the table and the
 * snapshot (see lapf_sampler_save for the layout and the load rule).  With every row equal to the batch
 * widths the chains are bit for bit those without the table. */
int lapf_sampler_set_frame_widths(lapf_sampler* s, const double* widths, void* stream);
/*   out device double [F][P]: the current table.  LAPF_ERR_INVALID without the table. */
int lapf_sampler_frame_widths(lapf_sampler* s, double* out, void* stream);
/* Per-frame acceptance, with or without the table: out device int64 [F][P][2], per frame and parameter the
 * sum over the frame's walkers of tries and of accepts since the last reset.  Integer sums: exact, in any
 * order; all-reduce them over ranks. */
int lapf_sampler_frame_counts(lapf_sampler* s, int64_t* out, void* stream);
/* One adaptation step from cumulative counts (lapf_sampler_frame_counts, already summed over ranks):
 * per (f, j), with (T, A) = counts[f][j] and (T', A') = the snapshot, dt = T - T', da = A - A'; if dt > 0,
 * widths[f][j] *= min(max(exp(da / dt - target), 0.5), 2.0) (the CLI's --adapt rule on the window since
 * the previous step, per frame; division, subtraction and product rounded to nearest, never fused); a
 * (f, j) with dt = 0 keeps its width.  Then snapshot = counts.  Stream-ordered, no host synchronisation:
 * ranks that apply it to the same counts keep the same widths.  LAPF_ERR_INVALID without the table or
 * unless 0 < target < 1. */
int lapf_sampler_adapt_widths(lapf_sampler* s, const int64_t* counts, double target, void* stream);

/* Total update count so far (same for every walker). */
int64_t lapf_sampler_count(const lapf_sampler* s);
/* Kernel launches issued by this sampler so far (for benchmark accounting). */
int64_t lapf_sampler_launches(const lapf_sampler* s);

/* K3 -- ordered device->pinned-host copy of a finished chain segment: copy_stream waits for
 * everything queued on compute_stream, then copies nbytes.  Replaces the whole-file rewrite
 * of apf_step2.py:355-360 as the way rows leave the sampler. */
int lapf_chain_drain(const void* device_src, void* pinned_dst, size_t nbytes,
                     void* compute_stream, void* copy_stream);

/* Host-side writer of one walker's <rank>_finalarray_mpi.csv (apf_step2.py:357-360):
 * optionally a leading all-nan row (the seed column of :278-279), then n_rows rows of n_cols
 * doubles taken from rows[r*row_stride + c], comma separated, CRLF terminated (csv.writer's
 * default dialect), shortest round-trip decimal.  Synchronous, CPU only.  With
 * LAPF_CSV_APPEND the rows are appended, so a chain can be written segment by segment instead
 * of the reference's whole-file rewrite every 10 updates (:355-360). */
#define LAPF_CSV_LEADING_NAN_ROW 1
#define LAPF_CSV_APPEND 2
int lapf_write_chain_csv(const char* path, const double* rows, int64_t n_rows, int32_t n_cols,
                         int64_t row_stride, int32_t flags);

/* Frame preparation on device (apf_step2.py:176-210): saturation mask + noise map folded into
 * the weight map, and cut-outs taken from full frames.
 *   frames     device [F][fy][fx] float      header scalars as in the reference
 *   origin     device [F][2] (x0, y0) of each cut-out
 *   data_out, weight_out device [F][ny][nx] float */
int lapf_frame_prep(const float* frames, int32_t n_frames, int32_t fy, int32_t fx,
                    const int32_t* origin, int32_t ny, int32_t nx, double satlevel,
                    double readnoise, float* data_out, float* weight_out, void* stream);

/* The part of the reference's whole-frame chi-square that lies OUTSIDE the cut-outs
 * (lapf_problem.outside): per frame sum w, sum w*d, sum w*d^2 over those pixels, with the weight
 * map of lapf_frame_prep, in FP64 and a fixed order.
 *   cut          device [F][2] (x, y) of each cut-out INSIDE its frame array
 *   outside_out  device double [F][3] */
int lapf_frame_outside(const float* frames, int32_t n_frames, int32_t fy, int32_t fx, const int32_t* cut,
                       int32_t ny, int32_t nx, double satlevel, double readnoise, double* outside_out,
                       void* stream);

/* The sampler's random stream for updates first_update .. first_update+n-1 of one walker, in the
 * reference's draw order (apf_step2.py:302 index, :64/:68 normal, :143 uniform): parameter index,
 * standard normal, natural log of the uniform.  Device outputs of length n.  Philox4x32-10 with
 * key = (seed low 32 bits, walker id) and counter = (update low, update high, seed high, 'LAPF');
 * the normal is Box-Muller of two 32-bit words, the uniform carries 53 bits like numpy's rand(). */
int lapf_philox_draws(uint64_t seed, uint64_t walker_id, uint64_t first_update, int32_t n, int32_t nparam,
                      int32_t* index_out, double* normal_out, double* log_uniform_out, void* stream);

/* Micro-benchmarks for the roofline denominators: issue rates of MUFU.EX2 and FFMA on the
 * current device.  Synchronous.  out[0] = ex2 results/s, out[1] = FFMA lane-ops/s,
 * out[2] = SM clock (MHz) reported by the driver, out[3] = SM count. */
int lapf_measure_peaks(double* out4);

#ifdef __cplusplus
}
#endif
#endif /* LAPF_H */
