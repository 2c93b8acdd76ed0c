/*
 * f2cnn_b200.h -- C ABI of libf2cnn_b200.so: the B200 (sm_100a) implementation of F2CNN's
 * feature-extraction hot path (gammatone filterbank -> ENV1 envelope -> windowing).
 *
 * The reference (tictacmenthe/F2CNN) is pure Python and has no FFI of its own; its boundary
 * is a set of module-level numpy functions (SURVEY.md section 8b).  Each entry point below
 * names the reference function (file:line under the reference tree) whose arithmetic it
 * replaces; f2cnn_b200/ mirrors those Python signatures on top of this ABI, and
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes only; every function returns an int status
 * (F2_OK == 0) and never throws; f2_last_error() gives the message of the calling thread's
 * last failure.  All data pointers are DEVICE pointers on the plan's device unless the
 * parameter is documented as host; `stream` is a cudaStream_t passed as void* (NULL = the
 * legacy default stream).  The caller owns every buffer, including the workspace.  A plan is
 * immutable after creation and may be shared by several streams; a batch may be run on one
 * stream at a time.  There is no CPU fallback: without a CUDA device every call fails with
 * F2_ERR_CUDA.
 */
#ifndef F2CNN_B200_H
#define F2CNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define F2_API __attribute__((visibility("default")))
#else
#define F2_API
#endif

#define F2_OK 0
#define F2_ERR_INVALID 1     /* bad argument */
#define F2_ERR_CUDA 2        /* CUDA runtime error (see f2_last_error) */
#define F2_ERR_WORKSPACE 3   /* workspace too small */
#define F2_ERR_UNSUPPORTED 4 /* size or filterbank outside the supported range */
#define F2_ERR_INDEX 5       /* a window index leaves its utterance (the reference raises IndexError) */

/* sample / matrix element types */
#define F2_I16 0
#define F2_F32 1
#define F2_F64 2

typedef struct f2_plan f2_plan;
typedef struct f2_batch f2_batch;

F2_API const char* f2_last_error(void);
/* ABI version of the library (bumped on any signature change). */
F2_API int f2_abi_version(void);

/* ---- plan: one gammatone filterbank ----------------------------------------------------
 * coefs: HOST pointer to the (n_channels, 10) float64 matrix returned by
 * gammatone.filters.make_erb_filters (gammatone/filters.py:186-190: columns
 * A0, A11, A12, A13, A14, A2, B0, B1, B2, gain).  Derives the float32 per-channel
 * parameter block in float64 and uploads it to `device`.  The kernels compute in float32: a bank whose
 * predicted float32 error (f2_bank_check) exceeds the 1e-4 x RMS tolerance is refused with
 * F2_ERR_UNSUPPORTED, unless the environment sets F2CNN_B200_ALLOW_IMPRECISE.  Same as
 * f2_plan_create_ex with flags 0. */
F2_API int f2_plan_create(const double* coefs, int n_channels, int device, f2_plan** out);
/* flags of f2_plan_create_ex */
#define F2_PLAN_FLOAT64_SECTIONS 1u /* in a bank f2_bank_check refuses (> 1), the groups of 32 channels
                                       predicted above the tolerance in float32 (f2_bank_check_groups > 1)
                                       run their four sections in float64; the bank is accepted and
                                       F2CNN_B200_ALLOW_IMPRECISE plays no part.  A bank f2_bank_check
                                       accepts runs in float32 exactly as without the flag. */
F2_API int f2_plan_create_ex(const double* coefs, int n_channels, int device, unsigned flags, f2_plan** out);
/* Which groups of 32 channels run in float64: mask[g] = 1 or 0 for g < n_groups (mask may be null when
 * n_groups == 0).  Returns how many groups do, or -1 for a null plan or bad arguments (f2_last_error). */
F2_API int f2_plan_float64_groups(const f2_plan* plan, unsigned char* mask, int n_groups);
/* Host-only check f2_plan_create applies (no device needed).  The kernels compute in float32 and are
 * held to 1e-4 x channel RMS against the reference's float64: the real cascade of the channels
 * nearest to z = 1 is run on the host in float32 with the kernel's exact operations and in float64,
 * on probe signals (loud tones, white noise); *predicted = worst error in units of that tolerance,
 * *worst_channel (nullable) where.  f2_plan_create fails with F2_ERR_UNSUPPORTED when it exceeds 1
 * (make_erb_filters(fs, cf, width) is public API, gammatone/filters.py:89: e.g. LOW_FREQ = 20 Hz with
 * width = 2), unless the environment sets F2CNN_B200_ALLOW_IMPRECISE. */
F2_API int f2_bank_check(const double* coefs, int n_channels, double* predicted, int* worst_channel);
/* The same prediction per group of 32 channels (one warp of the fused kernel), host only:
 * per_group[g] for g < ceil(n_channels / 32), from the group's own channels nearest to z = 1. */
F2_API int f2_bank_check_groups(const double* coefs, int n_channels, double* per_group);
F2_API int f2_plan_destroy(f2_plan* plan);
F2_API int f2_plan_channels(const f2_plan* plan);
/* Warm-up lengths in samples (rounded up to multiples of 256); <= 0 keeps the default that
 * plan creation derived from the slowest pole.  w_imag: periodic start of the Hilbert path;
 * w_edge: tail used for the edge residuals; w_casc: warm-up of a chunk that starts mid-signal. */
F2_API int f2_plan_set_warmup(f2_plan* plan, int w_imag, int w_edge, int w_casc);
F2_API int f2_plan_get_warmup(const f2_plan* plan, int* w_imag, int* w_edge, int* w_casc);

/* ---- batch: a set of utterances laid out for one launch sequence ------------------------
 * lengths: HOST array of n_utts sample counts; utterance u occupies samples
 * [sum(lengths[:u]), +lengths[u]) of the flat wave buffer.  step/phase define the decimated
 * grid t = phase + j*step (InputGenerator.py:65 STEP = int(FRAMERATE*SAMPLING_PERIOD/1e6);
 * LabelDataGenerator.py:48-50 puts every timepoint on that grid).  target_items <= 0 lets
 * the library choose how finely long utterances are split into time chunks; > 0 splits them
 * until there are about that many (utterance, 128 channels, chunk) units of work (1 = never
 * split).  f2_batch_num_items reports CTAs: (utterance, group of 32 channels, chunk). */
F2_API int f2_batch_create(f2_plan* plan, const int64_t* lengths, int n_utts, int step, int phase, int64_t target_items,
                    f2_batch** out);
F2_API int f2_batch_destroy(f2_batch* batch);
F2_API int64_t f2_batch_total_samples(const f2_batch* batch);
F2_API int64_t f2_batch_total_frames(const f2_batch* batch);
F2_API int64_t f2_batch_num_items(const f2_batch* batch);
/* frame_offsets: HOST array of n_utts+1: first decimated frame of each utterance. */
F2_API int f2_batch_frame_offsets(const f2_batch* batch, int64_t* frame_offsets);
/* Device workspace f2_batch_run needs for this batch, whatever outputs it is asked for: want_full_gfb and
 * want_full_env are ignored (the fused kernel stores every full-rate output itself). */
F2_API size_t f2_batch_workspace_bytes(const f2_batch* batch, int want_full_gfb, int want_full_env);

typedef struct f2_run_args {
    uint32_t struct_size; /* = sizeof(f2_run_args) of the caller's header: a struct that is shorter than
                           * the library's (an older binding) is rejected with F2_ERR_INVALID instead
                           * of being read past its end */
    const void* wave; /* flat samples of all utterances, wave_dtype                        */
    int wave_dtype;   /* F2_I16 (WAV), F2_F32, F2_F64 (noise-mixed, Evaluating.py:200)     */
    int lpf;          /* LPF flag of ExtractEnvelopeFromMatrix (EnvelopeExtraction.py:51)  */
    double cutoff_hz; /* CUTOFF; Nyquist fixed at 8000 Hz as in EnvelopeExtraction.py:47   */
    void* gfb;        /* out, nullable: erb_filterbank result, (C,n_u) blocks back to back */
    int gfb_dtype;    /* F2_F64 (reference dtype) or F2_F32                                */
    void* env;        /* out, nullable: ExtractEnvelopeFromMatrix result, same layout      */
    int env_dtype;
    float* env_t;     /* out, nullable: envelope time-major [sum n][C] float32             */
    float* dec;       /* out, nullable: decimated envelope frames [total_frames][C] float32.  The one output that may
                       * also be page-locked HOST memory the device can address under the same pointer (f2_host_pin):
                       * the kernel then stores the frames over PCIe as it produces them (the corpus pipeline) */
    void* ev_fused_start; /* nullable cudaEvent_t recorded on `stream` right before ...     */
    void* ev_fused_stop;  /* ... and right after the fused kernel (for roofline timing)     */
    /* Windows on the decimated grid written by the fused kernel itself (the rows GenerateInputData
     * builds for a label CSV whose timepoints are consecutive grid steps, InputGenerator.py:73-83 with
     * LabelDataGenerator.py:48-50): window k of utterance u = decimated frames k .. k+win_dots-1, for
     * k < win_offsets[u+1] - win_offsets[u]; it is row win_offsets[u] + k of `windows`
     * ([rows][win_dots][C] float32, rows >= win_offsets[n_utts]: the caller sizes it from its host copy
     * of the offsets).  win_offsets: DEVICE array of n_utts+1 row offsets.  Arbitrary timepoints take
     * `dec` + f2_gather_windows (or f2_place_windows on the host) instead. */
    float* windows;             /* out, nullable */
    const int64_t* win_offsets; /* device, required with windows */
    int win_dots;               /* 2*RADIUS+1 */
} f2_run_args;

/* Replaces, fused: filters.erb_filterbank (gammatone/filters.py:195-239),
 * ExtractEnvelopeFromMatrix (EnvelopeExtraction.py:51-67) and the decimated reads of
 * GenerateInputData (InputGenerator.py:73-80). */
F2_API int f2_batch_run(f2_batch* batch, const f2_run_args* args, void* workspace, size_t workspace_bytes, void* stream);

/* Decimated envelope frames of 1..4 envelope settings from ONE filterbank and Hilbert pass (the reference's
 * `prepare input --cutoff K` for several K: input_data_LPF<K>.npy, input_data_NOLPF.npy).  cutoffs_hz: HOST
 * array of n_settings entries, each a cutoff in (0, 8000) Hz or 0 for no low-pass.  Setting j's frames go to
 * dec + j * plane_stride, [total_frames][C] float32 on the batch's grid, exactly as f2_run_args.dec of an
 * f2_batch_run with that setting; plane_stride >= total_frames * C lets a sub-batch write its slice of a
 * larger [K][frames][C] array.  dec is device memory or memory pinned with f2_host_pin.  Workspace:
 * f2_batch_workspace_bytes.  Whole-utterance batches give every plane bit for bit what f2_batch_run gives;
 * in a time-chunked batch every chunk warms up for the slowest setting, the low-pass pole of largest |a1| (the
 * lowest cutoff, or the highest when it lies nearer 8000 Hz than the lowest lies to 0), so that setting's plane
 * is bit-identical and the others differ from their own runs only by the longer warm-up (below float32
 * resolution).  The warm-up bound |a1|^W < 1e-7 holds for either sign of the pole.
 * F2_ERR_INVALID: n_settings outside 1..4, a cutoff that is NaN or outside {0} u (0, 8000), a null dec or a
 * short plane_stride; F2_ERR_WORKSPACE: a short workspace. */
F2_API int f2_batch_run_cutoffs(f2_batch* batch, const void* wave, int wave_dtype, const double* cutoffs_hz,
                                int n_settings, float* dec, int64_t plane_stride, void* workspace,
                                size_t workspace_bytes, void* stream);

/* ---- stand-alone envelope of arbitrary matrix rows ---------------------------------------
 * ExtractEnvelopeFromMatrix(matrix, LPF, CUTOFF) for a matrix that did not come from this
 * library (e.g. loaded from .GFB.npy, EnvelopeExtraction.py:70-83): rows x n, row-major. */
F2_API size_t f2_envelope_rows_workspace_bytes(int64_t rows, int64_t n);
F2_API int f2_envelope_rows(f2_plan* plan, const void* matrix, int dtype, int64_t rows, int64_t n, int lpf,
                     double cutoff_hz, void* out, int out_dtype, void* workspace, size_t workspace_bytes,
                     void* stream);

/* The same machinery for the two other row-wise functions of EnvelopeExtraction.py:
 * F2_ROWS_HILBERT = imaginary part of paddedHilbert(row) (:20-36), F2_ROWS_LOWPASS =
 * lowPassFilter(row, cutoff) alone (:39-48, lpf must be 1).  F2_ROWS_ENVELOPE == f2_envelope_rows. */
#define F2_ROWS_ENVELOPE 0
#define F2_ROWS_HILBERT 1
#define F2_ROWS_LOWPASS 2
F2_API int f2_rows_op(f2_plan* plan, const void* matrix, int dtype, int64_t rows, int64_t n, int op, int lpf,
                      double cutoff_hz, void* out, int out_dtype, void* workspace, size_t workspace_bytes,
                      void* stream);

/* ---- windowing ---------------------------------------------------------------------------
 * out[w][j][c] = frames[base_rows[w] + j*stride_rows][c], j < dots: the window gather of
 * InputGenerator.py:73-80 on decimated frames (base = frame of center - RADIUS*STEP,
 * stride 1) or on a time-major full-rate envelope (base = center - RADIUS*STEP, stride STEP). */
F2_API int f2_gather_windows(const float* frames, int n_channels, const int64_t* base_rows, int64_t n_windows, int dots,
                      int64_t stride_rows, float* out, void* stream);
/* out[i][c] = src[idx[i]][c]: arbitrary rows (timepoints that wrap like a negative Python index). */
F2_API int f2_gather_index(const float* src, int n_channels, const int64_t* idx, int64_t n_idx, float* out, void* stream);
/* out[i][c] = (float) env[c*n + idx[i]]: the same gather from a (C,n) matrix in the reference's
 * own layout (a loaded .ENV1.npy, InputGenerator.py:72); F2_F64 -> float32 rounds like numpy. */
F2_API int f2_gather_windows_cn(const void* env, int dtype, int n_channels, int64_t n, const int64_t* idx,
                                int64_t n_idx, float* out, void* stream);
/* Dense framing of Evaluating.py:70-78: frame i = env_t rows i + k*step, k < dots, for
 * i0 <= i < i1; normalize != 0 applies Training.normalizeInput (Training.py:13-28) per frame
 * and sets *bad_flag (device int) when a frame has a value <= 0 (the reference raises).
 * n_rows: rows of env_t; frames that would read past it are rejected (F2_ERR_INVALID). */
F2_API int f2_dense_frames(const float* env_t, int64_t n_rows, int n_channels, int dots, int step, int64_t i0, int64_t i1,
                    int normalize, void* out, int out_dtype, int* bad_flag, void* stream);

/* ---- host side of the window stage ---------------------------------------------------------
 * All pointers in this section are HOST pointers and none of these functions needs a device.
 * When every timepoint of the label CSV lies on the decimated grid, row k of the reference's input
 * tensor (InputGenerator.py:73-80) is the block of `dots` CONSECUTIVE decimated frames that starts
 * at frame (center - RADIUS*STEP - phase)/STEP: the (N, dots, C) tensor repeats every frame `dots`
 * times.  Instead of copying that tensor over PCIe, the frames (`dec` of f2_batch_run) can travel
 * and the rows be placed on the host: one contiguous copy of dots*C floats per row, bit patterns
 * untouched. */
typedef struct f2_win_run {
    int64_t first_frame; /* row of the [frame][C] matrix where the first window of the run starts */
    int64_t row0;        /* output row of that window                                            */
    int64_t count;       /* windows in the run: window i = frames first_frame+i .. +dots-1 -> row0+i */
} f2_win_run;

/* Label timepoints -> runs.  centers: the window centres of all utterances back to back (counts[u] of
 * them for utterance u, in output order); lengths[u]: samples; frame_offsets: as returned by
 * f2_batch_frame_offsets for a batch with the same step and *phase; row_offsets: first output row of
 * each utterance, or NULL for rows in utterance order.  *phase < 0 on entry: taken from the first
 * window ((center - radius*step) mod step) and returned.  Index semantics of InputGenerator.py:76: an
 * index in [-n, 0) wraps like a Python index, any other index outside [0, n) fails with
 * F2_ERR_INDEX.  *n_runs = -1 when the timepoints are legal but are not all windows of consecutive
 * frames of ONE grid (a wrapping window, mixed phases): such requests take f2_gather_index instead.
 * runs == NULL only counts. */
F2_API int f2_window_runs(const int64_t* centers, const int64_t* counts, const int64_t* lengths,
                          const int64_t* frame_offsets, const int64_t* row_offsets, int n_utts, int radius, int step,
                          int* phase, f2_win_run* runs, int64_t max_runs, int64_t* n_runs, int64_t* n_rows);
/* out[(row0+i)][j][c] = frames[first_frame+i+j][c] for every run, on n_threads host threads (<= 0:
 * all the calling thread may run on), non-temporal stores.  Synchronous. */
F2_API int f2_place_windows(const float* frames, int n_channels, int dots, const f2_win_run* runs, int64_t n_runs,
                            float* out, int n_threads);
/* The same on a persistent worker pool fed in stream order: with after_stream != 0 the job becomes
 * runnable when everything queued on `stream` before this call has completed (cudaLaunchHostFunc) --
 * e.g. the device->host copy of `frames` -- so the host never blocks between sub-batches.  `runs` is
 * copied; frames and out must stay valid until f2_placer_wait returns. */
typedef struct f2_placer f2_placer;
F2_API int f2_placer_create(int n_threads, f2_placer** out);
F2_API int f2_placer_destroy(f2_placer* placer);
F2_API int f2_placer_threads(const f2_placer* placer);
F2_API int f2_placer_submit(f2_placer* placer, int after_stream, void* stream, const float* frames, int n_channels,
                            int dots, const f2_win_run* runs, int64_t n_runs, float* out);
F2_API int f2_placer_wait(f2_placer* placer);
/* Trace of the finished jobs, 4 doubles each: submit, runnable, done (CLOCK_MONOTONIC seconds) and the
 * rows placed.  Returns the number of jobs written (out == NULL: the number recorded); clear != 0
 * empties the trace. */
F2_API int64_t f2_placer_trace(f2_placer* placer, double* out, int64_t max_jobs, int clear);
/* Anonymous host memory advised to use transparent huge pages (a fresh 7.5 GB tensor of 4 KiB pages
 * costs two million page faults on its first write). */
F2_API int f2_host_alloc(size_t bytes, void** out);
F2_API int f2_host_free(void* ptr, size_t bytes);
/* Page-lock a block from f2_host_alloc for the current device and make it addressable from kernels under
 * its host pointer (cudaHostRegister, portable | mapped, after faulting the pages in); f2_host_unpin before
 * f2_host_free.  F2_ERR_UNSUPPORTED where device and host pointer of registered memory differ. */
F2_API int f2_host_pin(void* ptr, size_t bytes);
F2_API int f2_host_unpin(void* ptr);

/* ---- label generation (SURVEY.md section 8f rank 2) ---------------------------------------
 * Least-squares line through the `dots` = 2*RADIUS+1 formant frames around each timepoint and the
 * two-sided p-value of its Pearson correlation: the body of the step loop of
 * LabelDataGenerator.py:60-68 (numpy.linalg.lstsq + scipy.stats.pearsonr), one item per kept
 * timepoint.  formant: device float64 track(s); first[i]: index of item i's first frame in it
 * (FBFileReader.py:77-78: int(timepoint/wavToFormant - RADIUS)); center[i]: the timepoint in
 * samples; abscissae are center[i] + (k - RADIUS)*step.  out: device float64 [n_items][4] =
 * (slope a, intercept b, r, p); constant input gives r = p = NaN as scipy does.  float64
 * arithmetic throughout (the CSV keeps round(a, 5), round(p, 5)). */
F2_API int f2_label_fit(const double* formant, const int64_t* first, const int32_t* center, int64_t n_items, int dots,
                        int step, double* out, void* stream);
/* Label accuracy of `cnn eval*` (Evaluating.py:87-110) for many utterances in one launch.  scores: [F][2]
 * float32 (falling, rising), 8-byte aligned, utterance u's frames at rows score_offsets[u] .. score_offsets[u+1]
 * (n_utts + 1 non-decreasing entries), as f2_cnn_forward_segments lays them out.  Utterance u's labels are
 * entries label_offsets[u] .. label_offsets[u+1] of label_times (samples, non-decreasing within the utterance,
 * as ExtractLabel writes them) and label_classes.  Frame i of an utterance (its own frame number, compared with
 * the times as the reference does) decides 1 when scores[1] > scores[0] (equal or NaN: 0) and counts when
 * t_j < i < t_{j+1} for consecutive labels and i - t_j < step or t_{j+1} - i < step; its target is class j when
 * i - t_j <= t_{j+1} - i, else class j+1.  hits[u] / counted[u] (n_utts int64 each, overwritten) are then the
 * reference's accuracy.  Every array is device memory; decreasing times or offsets give counts of no meaning.
 * F2_ERR_INVALID: n_utts < 0, step <= 0, a null pointer or misaligned scores. */
F2_API int f2_label_accuracy(const float* scores, const int64_t* score_offsets, const int64_t* label_times,
                             const int32_t* label_classes, const int64_t* label_offsets, int n_utts, int step,
                             int64_t* hits, int64_t* counted, void* stream);

/* ---- CNN forward of `cnn eval*` on the tensor cores (SURVEY.md section 8f rank 1) ---------------------
 * The reference network (scripts/CNN/Training.py:93-114): Conv32 3x3 same, Conv32 3x3, MaxPool2, Conv64 3x3
 * same, Conv64 3x3, MaxPool2, Flatten(1920), Dense516, Dense2 softmax, ReLU after each convolution and the
 * first dense layer -- evaluated on every stride-1 frame of an utterance (Evaluating.py:70-87: frame i =
 * envelope samples i + k*STEP, k < 11, normalizeInput per frame, model.predict).  Here: three tcgen05
 * kernels, bf16 operands with float32 accumulation in tensor memory, frames taken straight from the
 * time-major envelope (`env_t` of f2_batch_run), so the (frames, 11, 128) tensor is never materialised.
 * arrays: 12 HOST float32 pointers in Keras' get_weights() order -- conv kernels HWIO and biases of the
 * four convolutions, then the two dense kernels (in, out) and biases.  Only the configured geometry
 * (dots = 11, channels = 128) is built; anything else fails with F2_ERR_UNSUPPORTED. */
typedef struct f2_cnn f2_cnn;
F2_API int f2_cnn_create(int device, const float* const* arrays, int dots, int channels, f2_cnn** out);
F2_API int f2_cnn_destroy(f2_cnn* cnn);
/* Device workspace of f2_cnn_forward / f2_cnn_forward_segments for n_frames frames: the intermediate tensors of
 * one chunk of min(n_frames, 32768) frames and room for that chunk's run table (16 bytes per frame, used when a
 * chunk crosses more segment boundaries than travel with the launch). */
F2_API size_t f2_cnn_workspace_bytes(const f2_cnn* cnn, int64_t n_frames);
/* Frames i0 <= i < i1 of env_t ([n_rows][128] float32, device); scores: [i1 - i0][2] float32 softmax
 * (falling, rising), device.  flags: two device ints the caller zeroes: flags[0] != 0 afterwards when a
 * frame held a value <= 0 (Training.normalizeInput raises ValueError there), flags[1] != 0 when the
 * tensor-core pipeline did not complete.  Frames are processed in chunks through `workspace`. */
F2_API int f2_cnn_forward(f2_cnn* cnn, const float* env_t, int64_t n_rows, int step, int64_t i0, int64_t i1, float* scores,
                          int* flags, void* workspace, size_t workspace_bytes, void* stream);
/* Many utterances in one pass: segment s is seg_frames[s] frames of env_t starting at row seg_rows[s] (frame i of
 * it = rows seg_rows[s] + i + k*step, k < 11), e.g. every frame of utterance s of a batch whose env_t holds
 * several.  seg_rows and seg_frames are HOST arrays of n_segs entries; zero-frame segments are legal.  The
 * segments' scores lie back to back in `scores` ([sum seg_frames][2] float32, device), and a chunk of frames
 * crosses segment boundaries, so a corpus of short utterances runs in full chunks.  flags: n_segs + 1 device
 * ints the caller zeroes: flags[s] != 0 afterwards when a frame of segment s held a value <= 0, flags[n_segs] != 0
 * when the tensor-core pipeline did not complete.  Workspace: f2_cnn_workspace_bytes(cnn, sum seg_frames).
 * F2_ERR_INVALID: a negative row or frame count, or a segment whose frames would read past n_rows;
 * F2_ERR_WORKSPACE: a short workspace.  f2_cnn_forward(i0, i1) is the one segment (i0, i1 - i0). */
F2_API int f2_cnn_forward_segments(f2_cnn* cnn, const float* env_t, int64_t n_rows, int step, const int64_t* seg_rows,
                                   const int64_t* seg_frames, int n_segs, float* scores, int* flags, void* workspace,
                                   size_t workspace_bytes, void* stream);
/* Where the intermediate tensors of the LAST chunk sit in the workspace (tests compare them layer by layer):
 * pooled conv2 output at the aligned start, [frame][4 planes][4*63 pixels][8 channels] bf16; the 1920
 * features per frame (Keras flatten order) as bf16 at *features_offset. */
F2_API int f2_cnn_workspace_layout(int64_t n_frames, int64_t* chunk_frames, size_t* features_offset);
/* Self-test of the tcgen05 operand conventions the CNN kernels rest on: D[r][j] = sum_k A[shift+r][k] *
 * B[j][k] for r < 128, A [a_rows][K] and B [N][K] row-major bf16 (device), D [128][N] float32 (device),
 * *status (device int) != 0 when the tensor-core pipeline did not complete.  variant 0 is the layout in
 * use; variant 1 swaps the descriptor's leading / stride offsets and must give a different result. */
F2_API int f2_umma_selftest(const void* a, int a_rows, const void* b, int n, int k, int shift, int variant, float* d,
                            int* status, void* stream);

/* Host -> device upload of n_spans byte ranges on `stream` (cudaMemcpyAsync each): the utterances of a
 * shard picked out of one host buffer that holds the whole corpus.  src_host should be page-locked
 * for the copies to be asynchronous.  Offsets and sizes in bytes, HOST arrays. */
F2_API int f2_upload_spans(void* dst_device, const void* src_host, const int64_t* src_off, const int64_t* dst_off,
                           const int64_t* nbytes, int64_t n_spans, void* stream);

/* ---- CUDA event helpers so that a host without a CUDA binding can time on the device ----- */
F2_API int f2_event_create(void** event);
F2_API int f2_event_destroy(void* event);
F2_API int f2_event_record(void* event, void* stream);
F2_API int f2_event_synchronize(void* event);
F2_API int f2_event_elapsed_ms(void* start, void* stop, float* ms);

/* butter(1, cutoff_hz/8000, 'low') as used by lowPassFilter (EnvelopeExtraction.py:47):
 * y[t] = b0*(x[t]+x[t-1]) - a1*y[t-1].  Host-only helper. */
F2_API int f2_lowpass_coefficients(double cutoff_hz, double* b0, double* a1);

#ifdef __cplusplus
}
#endif
#endif /* F2CNN_B200_H */
