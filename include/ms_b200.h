/*
 * ms_b200.h - C ABI of the B200-native Vicon Nexus loader / windowing / NMF-MU library
 * (libms_b200.so, built from muscle_synergies_b200/csrc/ for sm_100a).
 *
 * The reference (elvis-sik/muscle_synergies) is pure Python and has no FFI; the seam this
 * library replaces is the body of
 *     load_vicon_file(csv_filename)            src/muscle_synergies/vicon_data/load_csv.py:96-135
 * below the 2 x 5 header lines, i.e. for every data row
 *     csv.reader tokenisation                  load_csv.py:21-31
 *     GettingMeasurementsState._is_blank_line  reader.py:886-901
 *     DataState._parse_row / float()           reader.py:927-948
 *     DeviceAggregator.add_data column cut     aggregator.py:96-124, 229-241
 *     Builder._extract_dataframe               user_data.py:391-396   (float64, channel-major block)
 * and, for the windowing of project/segment.py,
 *     _transition_indices                      segment.py:667-755
 *     DeviceData.__getitem__(slice) row cuts   user_data.py:727-731
 * plus the declared extension behind find_synergies / vaf (analysis.py:597-667, 713-914).
 *
 * Conventions
 *   - plain C types only; every pointer named d_* is DEVICE memory owned by the caller,
 *     h_* is host memory; the library allocates nothing persistent.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - every entry point returns 0 on success or a negative MS_E_* code; kernels are
 *     enqueued asynchronously on `stream` unless stated otherwise.
 *   - re-entrant: one workspace per concurrent call.  The only process-wide state is bookkeeping that no result
 *     depends on: an atomic count of kernel launches (ms_launch_count) and, per calling thread, the text of the
 *     last CUDA failure (ms_last_cuda_error).
 */
#ifndef MS_B200_H
#define MS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MS_OK 0
#define MS_E_INVALID (-1)   /* bad argument (null pointer, misaligned buffer, bad size) */
#define MS_E_CUDA (-2)      /* a CUDA runtime call failed; see ms_last_cuda_error() */
#define MS_E_WORKSPACE (-3) /* workspace too small */
#define MS_E_NO_DEVICE (-4) /* no CUDA device / wrong architecture */

#ifndef MS_TILE_BYTES
#define MS_TILE_BYTES 49152     /* bytes of CSV owned by one thread block */
#endif
#define MS_MAX_ROW_BYTES 8192   /* longest CSV row of the tiled kernels (overhang staged past a tile); ms_parse_long beyond */
#define MS_MAX_BLANK_ROWS 8     /* blank rows reported by ms_scan (first ones, file order) */
#define MS_MAX_SECTIONS 4

/* flags in ms_scan_summary.flags */
#define MS_SCAN_HAS_HIGH_BYTES 1u    /* some byte >= 0x80 */
#define MS_SCAN_BLANK_OVERFLOW 2u    /* more blank rows than can be ordered exactly */
#define MS_SCAN_HAS_CR 4u

/* Result of ms_scan: written to DEVICE memory (copy it back after the stream is done). */
typedef struct ms_scan_summary {
    int64_t n_bytes;
    int64_t n_rows;        /* csv rows: terminators (\n, \r\n, lone \r) + unterminated last row */
    int64_t n_terminators;
    int64_t n_quotes;      /* '"' bytes in the whole buffer */
    int64_t n_blank_rows;  /* rows whose every field is empty after str.strip() (reader.py:886-901) */
    uint32_t flags;
    uint32_t n_reported;   /* entries valid in the arrays below (<= MS_MAX_BLANK_ROWS) */
    int64_t blank_row[MS_MAX_BLANK_ROWS];  /* 0-based csv row index of each blank row */
    int64_t blank_end[MS_MAX_BLANK_ROWS];  /* byte offset of the last byte of its terminator
                                              (== n_bytes for an unterminated last row) */
} ms_scan_summary;

/* One run of data rows that share a column layout (one per CSV section). */
typedef struct ms_section {
    int64_t row_begin;  /* first data row (0-based csv row index) */
    int64_t row_end;    /* one past the last data row */
    int32_t num_cols;   /* fields parsed per row: reader.py:241-243 (rest of the row is ignored) */
    int32_t n_keep;     /* channels stored: csv columns [2, 2 + n_keep) (aggregator.py:96-124) */
    double* d_out;      /* [n_keep][stride] float64, channel-major (user_data.py:396 block layout) */
    int64_t stride;     /* elements between channels, >= row_end - row_begin */
} ms_section;

/* status key written by ms_parse: ~0 when every field parsed, else
 * (byte offset of the first offending field << 3) | kind, minimum over the file. */
#define MS_ERR_NONE 0xFFFFFFFFFFFFFFFFull
#define MS_ERR_KIND_BAD_FLOAT 1u   /* float(field) raises ValueError */
#define MS_ERR_KIND_NON_ASCII 2u   /* byte >= 0x80 in a numeric field: unsupported on device */
#define MS_ERR_KIND_ROW_TOO_LONG 3u /* a row exceeds MS_MAX_ROW_BYTES: parse the buffer with ms_parse_long */

/* ---- loader ------------------------------------------------------------------------- */

/* Bytes of device workspace needed to scan + parse a buffer of n_bytes. */
int64_t ms_workspace_bytes(int64_t n_bytes);

/* Offset in the workspace of the per-16-byte delimiter masks ms_scan leaves behind (uint32 per
 * segment: row-terminator bits | comma bits << 16); lets a caller map a byte offset to its row. */
int64_t ms_workspace_masks_offset(int64_t n_bytes);

/* Pass 1: row terminators per tile, blank rows, quote count.  d_bytes must be 16-byte
 * aligned and readable up to n_bytes rounded up to 16 (pad the allocation). */
int ms_scan(const uint8_t* d_bytes, int64_t n_bytes, void* d_workspace, int64_t workspace_bytes,
            ms_scan_summary* d_summary, void* stream);

/* Copies up to max_bytes bytes that follow blank row `which` of a finished ms_scan (the header lines of
 * the next section, reader.py:250-835 parses them on the host) to d_out, and {offset, count} to d_info
 * ({-1, 0} when that blank row was not reported): the host then needs one transfer, not two. */
int ms_peek_after_blank(const uint8_t* d_bytes, int64_t n_bytes, const ms_scan_summary* d_summary, int32_t which,
                        uint8_t* d_out, int32_t max_bytes, int64_t* d_info, void* stream);

/* Rescan for buffers whose DATA rows contain '"' (ms_scan counted more quotes than the header
 * lines hold): same outputs, but commas and line ends inside quoted fields (csv excel dialect,
 * load_csv.py:30) are not delimiters.  Call after ms_scan, same buffer and workspace. */
int ms_scan_quoted(const uint8_t* d_bytes, int64_t n_bytes, void* d_workspace, int64_t workspace_bytes,
                   ms_scan_summary* d_summary, void* stream);

/* Pass 2: parse the data rows of up to MS_MAX_SECTIONS sections into channel-major
 * float64 arrays.  Needs the workspace filled by ms_scan for the same buffer.
 * d_status: one uint64 in device memory (see MS_ERR_*). */
int ms_parse(const uint8_t* d_bytes, int64_t n_bytes, const void* d_workspace, const ms_section* h_sections,
             int32_t n_sections, uint64_t* d_status, void* stream);

/* Rows of any length: ms_parse reports MS_ERR_KIND_ROW_TOO_LONG for a buffer with a row it cannot stage
 * (> MS_MAX_ROW_BYTES); this entry point parses such a buffer instead - one thread per row, straight from global
 * memory, same outputs and status word.  Needs the workspace of ms_scan (or ms_scan_quoted) for the same buffer,
 * its summary's n_terminators, and d_rows: ms_parse_long_workspace_bytes(n_terminators) bytes of device scratch. */
int64_t ms_parse_long_workspace_bytes(int64_t n_terminators);
int ms_parse_long(const uint8_t* d_bytes, int64_t n_bytes, const void* d_workspace, const ms_section* h_sections,
                  int32_t n_sections, int64_t n_terminators, void* d_rows, uint64_t* d_status, void* stream);

/* ---- loader, single pass ----------------------------------------------------------------- */

/* The whole of load_vicon_file below its header text (load_csv.py:96-135) in ONE launch: row terminators,
 * blank (section separator) rows, the section a row belongs to and its index there (a decoupled look-back
 * between thread blocks), the column count of each section from its coordinates line (reader.py:772-783),
 * float() of every field (reader.py:940-948) and the channel-major float64 blocks (aggregator.py:96-124,
 * user_data.py:391-396).  Every CSV byte is read from HBM once, every kept double written once.
 *
 * It answers for well-formed files only (two sections, at most one trailing blank row, no quote characters
 * in the data rows, rows of at most MS_MAX_ROW_BYTES, outputs that fit the arena): anything else sets a bit
 * in ms_load_result.flags, the arrays are then meaningless and the caller runs ms_scan / ms_parse, which
 * reproduce the reference's behaviour - its errors included - on every input. */
#define MS_LOAD_PEEK 8192 /* bytes of header text copied out per section */

/* ms_load_result.flags */
#define MS_LOAD_ROW_TOO_LONG 1u  /* a row does not end within MS_MAX_ROW_BYTES of the end of its tile */
#define MS_LOAD_DENSE_ROWS 2u    /* too many rows start in one tile */
#define MS_LOAD_MANY_BLANKS 4u   /* more than two blank rows in one tile */
#define MS_LOAD_TAIL_ROWS 8u     /* rows after the second blank row (the reference raises there) */
#define MS_LOAD_OVERFLOW 16u     /* a section does not fit the arena / its row capacity */
#define MS_LOAD_BAD_HEADER 32u   /* a coordinates line with fewer than 3 fields (or more than 65535) */
#define MS_LOAD_HIGH_BYTES 64u   /* some byte >= 0x80 next to a line end, quote or blank (the only ones looked at) */
/* ms_load_result.have */
#define MS_LOAD_HAVE_HEADER0 1u  /* << section: header_offset / peek_bytes are set */
#define MS_LOAD_HAVE_DESC0 4u    /* << section: num_cols / n_keep / stride / out_offset are set */
#define MS_LOAD_HAVE_ROWS0 16u   /* << section: data_rows is set */

typedef struct ms_load_plan {
    double* d_arena;      /* device memory for both sections' blocks, 16-byte aligned */
    int64_t arena_elems;  /* doubles in the arena */
    int64_t cap_rows[2];  /* row capacity (= channel stride) of each section's block; cap_rows[1] == 0: the
                             second block takes what the first one leaves of the arena */
    int32_t tile_bytes;   /* CSV bytes per thread block, a multiple of 16, at least 4096; 0 = the largest that fits
                             shared memory next to the overhang (MS_TILE_BYTES at most when overhang_bytes is 0) */
    int32_t overhang_bytes; /* bytes staged past a tile to finish its last row = the longest row this launch can
                             take (longer: MS_LOAD_ROW_TOO_LONG); a multiple of 16 in [512, MS_MAX_ROW_BYTES];
                             0 = MS_MAX_ROW_BYTES.  Tile + overhang share 56 KiB: short rows leave more to the tile. */
} ms_load_plan;

/* Written to DEVICE memory; copy it back after the stream is done. */
typedef struct ms_load_result {
    uint64_t status;           /* as ms_parse: MS_ERR_NONE, or (byte offset << 3) | kind of the first bad field */
    uint32_t flags;            /* MS_LOAD_*: non-zero = not a file for this entry point */
    uint32_t have;             /* MS_LOAD_HAVE_* */
    uint32_t n_blank_rows;     /* blank rows in the file, saturating at 3 */
    uint32_t reserved;
    int64_t tail_rows;         /* csv rows after the last blank row (all rows if there is none) */
    int64_t n_quotes;          /* '"' bytes next to a line end or blank, plus every one the parser met */
    int64_t header_offset[2];  /* byte offset of the section's first header line */
    int64_t peek_bytes[2];     /* bytes of header text copied to d_peek + section * MS_LOAD_PEEK */
    int64_t blank_end[2];      /* offset of the last byte of the blank row that closes the section */
    int64_t data_rows[2];      /* data rows of the section (negative: it ended inside its header) */
    int32_t num_cols[2];       /* fields parsed per row */
    int32_t n_keep[2];         /* channels stored: num_cols - 2 */
    int64_t stride[2];         /* elements between channels of the section's block */
    int64_t out_offset[2];     /* element offset of the block in the arena: block[c * stride + row] */
} ms_load_result;

int64_t ms_load_workspace_bytes(int64_t n_bytes, int32_t tile_bytes);
/* d_bytes as for ms_scan; d_workspace: ms_load_workspace_bytes(), 16-byte aligned; d_peek: 2 * MS_LOAD_PEEK bytes. */
int ms_load_fused(const uint8_t* d_bytes, int64_t n_bytes, const ms_load_plan* h_plan, void* d_workspace,
                  int64_t workspace_bytes, ms_load_result* d_result, uint8_t* d_peek, void* stream);

/* ---- windowing ------------------------------------------------------------------------ */

/* _transition_indices (segment.py:667-755): alternating search for the first run of
 * >= min_phase_size samples with exactly one / exactly two loaded plates (value != 0, NaN
 * counts as loaded; a run cut short by the end of the signal counts).  Writes up to
 * num_segments sample indices to d_transitions, for each of them which plates are loaded
 * there to d_loaded (bit 0 left, bit 1 right; may be NULL) and the number found to
 * d_n_found.  d_work: ms_transitions_workspace_bytes(n) bytes of device scratch. */
int64_t ms_transitions_workspace_bytes(int64_t n);
int ms_find_transitions(const double* d_left_fz, const double* d_right_fz, int64_t n, int32_t min_phase_size,
                        int32_t num_segments, void* d_work, int64_t* d_transitions, int32_t* d_loaded,
                        int32_t* d_n_found, void* stream);

/* ms_find_transitions and, in the same launch, ms_plan_phase_windows for up to MS_MAX_WINDOW_PLANS devices (the
 * block that finishes the bitmaps last runs the search and the plans): what Segmenter(data) needs from the GPU is
 * then one launch, and the gathers of ms_cut_windows can be queued right behind it. */
#define MS_MAX_WINDOW_PLANS 4
typedef struct ms_window_plan {
    int64_t divisor;     /* 1 for force plates / EMG, num_subframes for trajectory markers */
    int64_t n_rows;      /* rows of the device's block */
    int32_t n_channels;
    int32_t cycles;      /* 0: the 32 phase windows, else the 8 cycle windows */
    int64_t* d_starts;   /* outputs, as ms_plan_phase_windows */
    int64_t* d_stops;
    int64_t* d_offsets;
} ms_window_plan;
int ms_segment_trial(const double* d_left_fz, const double* d_right_fz, int64_t n, int32_t min_phase_size,
                     int32_t num_segments, void* d_work, int64_t* d_transitions, int32_t* d_loaded, int32_t* d_n_found,
                     const ms_window_plan* h_plans, int32_t n_plans, void* stream);

/* Row ranges of the 32 phase windows (cycles == 0; order: trecho, cycle, phase) or the 8 cycle windows
 * (cycles != 0) of one device, from transitions still in device memory (the output of
 * ms_find_transitions with num_segments >= 40), so that ms_cut_windows can be queued without a host
 * round trip: start = t_j / divisor, stop = (t_next - 1) / divisor, the values
 * DeviceData.to_index(Segmenter.get_times_of(...)) yields (segment.py:862-917, user_data.py:513-661);
 * divisor = 1 for force plates / EMG, num_subframes for trajectory markers.  Writes starts, stops
 * (n_windows each) and offsets (n_windows + 1 prefix sums of len * n_channels).  All windows are
 * empty when fewer than num_segments transitions were found. */
int ms_plan_phase_windows(const int64_t* d_transitions, const int32_t* d_n_found, int32_t num_segments,
                          int32_t cycles, int64_t divisor, int64_t n_rows, int32_t n_channels, int64_t* d_starts,
                          int64_t* d_stops, int64_t* d_offsets, void* stream);

/* DeviceData.__getitem__(slice) (user_data.py:727-731) for many windows at once: copies rows
 * [start_w, stop_w) of every channel of a channel-major array (d_src[c * src_stride + row])
 * to d_out[out_offset_w + c * (stop_w - start_w) + r].  max_window_len: the longest window
 * (sizes the grid). */
int ms_cut_windows(const double* d_src, int64_t src_stride, int32_t n_channels, const int64_t* d_starts,
                   const int64_t* d_stops, const int64_t* d_out_offsets, int32_t n_windows, double* d_out,
                   int64_t max_window_len, void* stream);

/* ---- EMG envelope chain (SURVEY.md section 8f rank 1; float64, tolerance parity) ---------------- */

/* zero_center (analysis.py:230-249): mean of each channel of a channel-major array. */
int ms_channel_means(const double* d_src, int64_t stride, int32_t n_channels, int64_t n, double* d_mean, void* stream);
/* rms (analysis.py:435-507): sqrt(np.convolve((x - mean)^2, ones(window) / window, "same")) per
 * channel; d_mean may be NULL (no centring).  window <= n. */
int ms_rms_envelope(const double* d_src, int64_t stride, int32_t n_channels, int64_t n, const double* d_mean,
                    int32_t window, double* d_out, int64_t out_stride, void* stream);
/* digital_filter (analysis.py:314-432): scipy.signal.sosfilt (zero_lag == 0: forward, from rest) or
 * sosfiltfilt (zero_lag != 0: odd extension by padlen samples, forward and backward runs started at
 * h_zi * first sample) along time, per channel.  h_sos: [n_sections][6] = b0 b1 b2 1 a1 a2 (scipy's
 * layout, host memory, n_sections <= 8); h_zi: [n_sections][2] = scipy.signal.sosfilt_zi(sos) (host;
 * only read when zero_lag); padlen: sosfiltfilt's (n > padlen), 0 when zero_lag == 0.
 * linear_envelope (analysis.py:252-311) is the same call with the rectification fused into the loads:
 * the filter input is x - d_mean[channel] (d_mean NULL: x), and its absolute value when rectify != 0.
 * d_work: ms_sosfilt_workspace_bytes(n, n_channels, padlen, zero_lag) bytes of device memory. */
size_t ms_sosfilt_workspace_bytes(int64_t n, int32_t n_channels, int64_t padlen, int32_t zero_lag);
int ms_sosfilt(const double* d_src, int64_t stride, int32_t n_channels, int64_t n, const double* h_sos,
               int32_t n_sections, const double* h_zi, int64_t padlen, int32_t zero_lag, const double* d_mean,
               int32_t rectify, double* d_out, int64_t out_stride, void* d_work, void* stream);
/* time_normalize (analysis.py:551-594, linear) of rows [start_w, stop_w) onto reduce_to points,
 * then (normalize != 0) normalize (analysis.py:510-525): divide by the column max |.|.
 * d_out: [n_windows][reduce_to][n_channels] (samples x muscles, the orientation NMF takes). */
int ms_time_normalize_windows(const double* d_env, int64_t stride, int32_t n_channels, const int64_t* d_starts,
                              const int64_t* d_stops, int32_t n_windows, int32_t reduce_to, int32_t normalize,
                              double* d_out, void* stream);

/* ---- NMF by multiplicative updates (extension; not a reference-parity claim) --------------- */

/* What analysis.py:862-863 asks scikit-learn for with solver="mu", beta_loss="frobenius":
 *   W <- W * (X H^T) / (W (H H^T));  H <- H * (W^T X) / ((W^T W) H);  zero denominators -> float32 eps;
 *   every check_every iterations (tol > 0) stop when (previous_error - error) / error_at_init < tol.
 * One launch runs a whole batch of problems on the same X (rank sweep x restarts), fp32,
 * X / W / H resident in shared memory.  d_X: one or more [n][m] row-major matrices (samples x
 * muscles); h_x_index[p] (NULL = all 0) selects the matrix of problem p, so a launch can also
 * cover many gait cycles.  h_ranks[p]: rank of problem p (1..16).  d_W / d_H: initial factors
 * packed problem after problem (W_p [n][k_p], H_p [k_p][m], row-major); results overwrite them.
 * d_work: n_problems * 32 bytes.  Outputs per problem: d_n_iter, d_err = ||X - W H||_F,
 * d_vaf [m + 1] = 1 - SS_res / SS_tot overall, then per column (analysis.py:642-667). */
int32_t ms_nmf_resident_max_rows(int32_t m, int32_t kmax);
int ms_nmf_mu_batched(const float* d_X, int32_t n, int32_t m, const int32_t* h_ranks, const int32_t* h_x_index,
                      int32_t n_problems,
                      float* d_W, float* d_H, int32_t max_iter, float tol, int32_t check_every, void* d_work,
                      int32_t* d_n_iter, float* d_err, float* d_vaf, void* stream);

/* The same launch without the host-to-device copy of the problem table and the wait behind it: ms_nmf_plan writes
 * the table (32 bytes per problem) to host memory the caller owns and returns the largest rank (or MS_E_*); the caller
 * keeps a device copy for as long as it runs that sweep (one launch per trial in pipeline.py) and passes it, with
 * that rank, to ms_nmf_mu_batched_planned, which only queues the kernel. */
int32_t ms_nmf_plan(int32_t n, int32_t m, const int32_t* h_ranks, const int32_t* h_x_index, int32_t n_problems, void* h_table);
int ms_nmf_mu_batched_planned(const float* d_X, int32_t n, int32_t m, const void* d_table, int32_t n_problems, int32_t kmax,
                              float* d_W, float* d_H, int32_t max_iter, float tol, int32_t check_every,
                              int32_t* d_n_iter, float* d_err, float* d_vaf, void* stream);

/* Same contract for X of any length: X [n][m] and W [n][k] stream from HBM once per iteration
 * (algorithmic bytes per iteration and problem: 4 n m + 8 n k); W^T X and W^T W are reduced per
 * CTA and accumulated with atomics; the objective needs no extra pass over X.
 * d_work: ms_nmf_stream_workspace_bytes(m, n_problems). */
int64_t ms_nmf_stream_workspace_bytes(int32_t m, int32_t n_problems);
int ms_nmf_mu_stream(const float* d_X, int64_t n, int32_t m, const int32_t* h_ranks, const int32_t* h_x_index,
                     int32_t n_problems, float* d_W, float* d_H, int32_t max_iter, float tol, int32_t check_every,
                     void* d_work, int32_t* d_n_iter, float* d_err, float* d_vaf, void* stream);

/* ---- NMF by coordinate descent, NNDSVD initialisation (extension; fp64) ----------------------- */

/* scikit-learn's default solver="cd" (shuffle=False, no regularisation; _nmf.py _fit_coordinate_descent,
 * _cdnmf_fast.pyx) for a batch of problems, in fp64: per iteration a coordinate sweep of W with H H^T and X H^T of the
 * current H, then of H with W^T W and X^T W of the updated W; the summed projected-gradient violation of iteration 1
 * is violation_init, and a problem stops when that is 0 or violation / violation_init <= tol (tol = 0: max_iter
 * iterations).  Same batch description as the MU entries: d_X one or more [n][m] row-major fp64 matrices, d_table
 * the 32-byte problem table of ms_nmf_plan in device memory (ranks 1..16, m <= 64), d_W / d_H the initial factors
 * packed problem after problem (fp64), overwritten with the results.  Outputs per problem: d_n_iter, d_err =
 * ||X - W H||_F, d_vaf [m + 1] = 1 - SS_res / SS_tot overall, then per column (analysis.py:642-667), all fp64.
 * ms_nmf_cd_batched_planned keeps each problem in the shared memory of one CTA (n <= ms_nmf_cd_resident_max_rows). */
int32_t ms_nmf_cd_resident_max_rows(int32_t m, int32_t kmax);
int ms_nmf_cd_batched_planned(const double* d_X, int32_t n, int32_t m, const void* d_table, int32_t n_problems,
                              int32_t kmax, double* d_W, double* d_H, int32_t max_iter, double tol, int32_t* d_n_iter,
                              double* d_err, double* d_vaf, void* stream);

/* Same contract for X of any length: per iteration one pass over X [n][m] and W [n][k] in HBM (the W step, W^T W,
 * X^T W and the violation; algorithmic bytes 8 n m + P * 16 n k when every problem shares one X), then one small
 * kernel per problem for the H step and the stop test.  Synchronises `stream` every 64 iterations to stop once every
 * problem has converged.  d_work: ms_nmf_cd_stream_workspace_bytes(m, n_problems), 256-byte aligned. */
int64_t ms_nmf_cd_stream_workspace_bytes(int32_t m, int32_t n_problems);
int ms_nmf_cd_stream(const double* d_X, int64_t n, int32_t m, const void* d_table, int32_t n_problems, int32_t kmax,
                     double* d_W, double* d_H, int32_t max_iter, double tol, void* d_work, int32_t* d_n_iter,
                     double* d_err, double* d_vaf, void* stream);

/* _initialize_nmf(X, k, init="nndsvd" (variant 0) or "nndsvda" (variant 1)) for every problem of a batch, written to
 * the packed d_W / d_H (fp64).  The singular triplets are exact (X^T X, cyclic Jacobi eigensolver, U = X V S^-1),
 * one SVD per matrix of the stack (n_matrices [n][m] matrices in d_X); scikit-learn's come from a randomized SVD, so
 * its random_state has no counterpart here.  kmax <= min(n, m).  *d_status (device) is set non-zero when the init
 * would divide by zero: a singular value needed is 0 (at most m * eps * the largest one) or the chosen part of a
 * singular vector pair is empty; the factors are then meaningless.  d_work: ms_nndsvd_workspace_bytes(m, n_matrices). */
int64_t ms_nndsvd_workspace_bytes(int32_t m, int32_t n_matrices);
int ms_nndsvd_init(const double* d_X, int64_t n, int32_t m, int32_t n_matrices, const void* d_table, int32_t n_problems,
                   int32_t kmax, int32_t variant, void* d_work, double* d_W, double* d_H, int32_t* d_status, void* stream);

/* NMF with fixed synergies, what sklearn's NMF.transform does (update_H=False), for a batch of problems in fp64:
 * problem p fits W_p >= 0 to the matrix x_off of its ms_nmf_plan table entry with H_p (d_H, packed, k_p x m) held fixed.
 * solver 0 = "cd" (coordinate descent; d_W must hold zeros), 1 = "mu" (multiplicative updates, beta 2; d_W must hold
 * sqrt(mean(X) / k_p)); d_W receives the result.  X element (i, j) of a matrix is at d_X[x_off + i * row_stride +
 * j * col_stride]: a row-major [n][m] matrix (m, 1) and a channel-major [m][n] one (1, n) are read in place.  Outputs
 * per problem as for ms_nmf_cd_batched_planned: d_n_iter, d_err = ||X - W H||_F, d_vaf [m + 1].
 * regime 0 (n <= ms_nmf_fixed_h_resident_max_rows(m, kmax)): one CTA per problem, all of it in shared memory, d_work
 * unused.  regime 1 (any n): X is read once to form X H^T, then rows iterate in registers in chunks; synchronises
 * `stream` every 64 iterations to stop once every problem has stopped.  d_work: ms_nmf_fixed_h_workspace_bytes(n, m,
 * n_problems, kmax), 256-byte aligned.  Ranks 1..16, m <= 64; reductions have a fixed order (results are reproducible
 * bit for bit), and at tol = 0 both regimes give the same W bit for bit. */
int32_t ms_nmf_fixed_h_resident_max_rows(int32_t m, int32_t kmax);
int64_t ms_nmf_fixed_h_workspace_bytes(int64_t n, int32_t m, int32_t n_problems, int32_t kmax);
int ms_nmf_fixed_h(const double* d_X, int64_t n, int32_t m, int64_t row_stride, int64_t col_stride, const void* d_table,
                   int32_t n_problems, int32_t kmax, double* d_W, const double* d_H, int32_t solver, int32_t max_iter,
                   double tol, int32_t regime, void* d_work, int32_t* d_n_iter, double* d_err, double* d_vaf,
                   void* stream);

/* β-divergence NMF by multiplicative updates, fp64: scikit-learn's solver="mu" with beta_loss = beta != 2 (1: Kullback-
 * Leibler, 0: Itakura-Saito, any other float), no regularisation.  update_H = 1: fit W (n x k_p) and H (k_p x m) from
 * the given d_W / d_H (ms_nmf_plan's table, as for ms_nmf_cd_batched_planned); update_H = 0: sklearn's transform, H
 * fixed, from the given W (sklearn starts it at sqrt(mean(X) / k_p)).  X as for ms_nmf_fixed_h (row_stride,
 * col_stride).  Outputs per problem: d_n_iter, d_err = sqrt(2 D_beta(X | W H)) (sklearn's reconstruction_err_), d_vaf
 * [m + 1] (Frobenius VAF, overall then per column).  regime 0 (n <= ms_nmf_beta_resident_max_rows(m, kmax)): one CTA
 * per problem, d_work unused.  regime 1 (any n): one pass over X per iteration; synchronises `stream` every 64
 * iterations when tol > 0 to stop once every problem has stopped.  d_work: ms_nmf_beta_workspace_bytes(n, m,
 * n_problems, kmax), 256-byte aligned.  Ranks 1..16, m <= 64; beta = 2 is refused (MS_E_INVALID).  Reductions have a
 * fixed order: results are reproducible bit for bit. */
int32_t ms_nmf_beta_resident_max_rows(int32_t m, int32_t kmax);
int64_t ms_nmf_beta_workspace_bytes(int64_t n, int32_t m, int32_t n_problems, int32_t kmax);
int ms_nmf_beta(const double* d_X, int64_t n, int32_t m, int64_t row_stride, int64_t col_stride, const void* d_table,
                int32_t n_problems, int32_t kmax, double* d_W, double* d_H, double beta, int32_t update_H,
                int32_t max_iter, double tol, int32_t regime, void* d_work, int32_t* d_n_iter, double* d_err,
                double* d_vaf, void* stream);

/* ---- synergy comparison (extension; fp64) --------------------------------------------------- */

/* One synergy set of a packed array: rows [offset, offset + k * m) of d_H are its k synergy vectors (row-major). */
typedef struct ms_synergy_set {
    int64_t offset;   /* element offset of the set's first row in d_H */
    int32_t k;        /* rank: rows of the set, 1..kmax */
    int32_t reserved;
} ms_synergy_set;

/* Matched cosine similarity of pairs of synergy sets of equal rank, the standard comparison of synergies between
 * cycles, trials or subjects.  For pair p = (a, b) = d_pairs[2p], d_pairs[2p + 1] (int32 indices into d_sets, device
 * memory, 8-byte aligned): S[i][j] = <a_i, b_j> / (||a_i|| ||b_j||) (0 where a row's norm is 0 or its squared norm
 * overflows), then the exact
 * maximum-weight perfect matching on S that scipy.optimize.linear_sum_assignment(S, maximize=True) finds (shortest
 * augmenting paths, O(k^3); among equal tentative distances the lowest column is taken).  Writes d_mean[p], the mean
 * matched similarity; d_pairs NULL: every pair a < b of the table, in np.triu_indices(n_sets, 1) order (the kernel
 * decodes p; n_pairs must be n_sets (n_sets - 1) / 2).  d_perm[p * kmax + i] (int8), the row of b paired with row i of a, and d_sim[p * kmax + i], that
 * similarity, both for i < k and -1 / NaN for k <= i < kmax; d_perm and d_sim may be NULL.  kmax: the largest rank in
 * the table, 1..16; m: 1..64.  d_work: ms_synergy_match_workspace_bytes(n_sets) bytes (the norms, once per set).  A
 * set whose rank is outside 1..kmax, a pair index outside the table or a pair of unequal ranks is found on the device:
 * the entry then returns MS_E_INVALID (that pair's outputs are NaN / -1).  Synchronises `stream` to read that check.
 * No floating-point atomics: repeated calls are bit-identical. */
int64_t ms_synergy_match_workspace_bytes(int32_t n_sets);
int ms_synergy_match(const double* d_H, int32_t m, const ms_synergy_set* d_sets, int32_t n_sets, int32_t kmax,
                     const int32_t* d_pairs, int64_t n_pairs, int8_t* d_perm, double* d_sim, double* d_mean,
                     void* d_work, int64_t work_bytes, void* stream);

/* ---- misc ------------------------------------------------------------------------------- */
/* The used part of a channel-major block (rows channels of width_bytes each, src_pitch_bytes apart) to host
 * memory as one 2-D copy on the DMA engine; asynchronous when h_dst is page-locked. */
int ms_copy_rows_to_host(void* h_dst, int64_t dst_pitch_bytes, const void* d_src, int64_t src_pitch_bytes,
                         int64_t width_bytes, int64_t rows, void* stream);
/* Host to host copy with non-temporal stores (no read of the destination's cache lines): what the file readers use to
 * move a mapped file out of the page cache into the pinned buffer the DMA engine reads (load_csv.py:29 opens the file;
 * everything after that is this library's). */
int ms_host_copy_stream(void* h_dst, const void* h_src, int64_t n_bytes);
/* Text of the last CUDA failure reported (MS_E_CUDA) to the calling thread. */
const char* ms_last_cuda_error(void);
const char* ms_version(void);
/* Number of kernels this library has launched in this process (bench.py gpu_launches). */
int64_t ms_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* MS_B200_H */
