/*
 * ncfa.h — C ABI of the B200-native nightcore front-end (libncfa.so).
 *
 * The reference (Tealdragon204/nightcore-to-flac-analyzer) is pure Python and has no FFI; its
 * boundary for this path is the Python module surface (SURVEY.md §8b).  These entry points are
 * what the drop-in `nightcore_analyzer` Python package binds through ctypes, one per kernel
 * family; each cites the reference interface it replaces (paths under
 * /root/reference/nightcore_analyzer/).
 *
 * Conventions
 *   - every pointer named d_* is DEVICE memory owned by the caller; h_* is host memory;
 *   - `stream` is a cudaStream_t passed as void*; nothing here synchronises or allocates;
 *   - workspaces are caller-provided; query the size with the paired *_workspace_bytes();
 *   - return 0 on success, a negative NCFA_E_* code otherwise; ncfa_last_error() gives the
 *     (thread-local) message.  No exceptions cross the boundary.
 *   - a "segment" is a contiguous run of samples inside one device audio buffer:
 *     d_seg_off[i] (int64 sample offset) and d_seg_len[i] (int32 samples).  Analysis windows
 *     (io.py:94-110) and whole tracks (tempo.py:158) are both segments.
 */
#ifndef NCFA_H
#define NCFA_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NCFA_OK 0
#define NCFA_E_INVALID (-1)   /* bad argument */
#define NCFA_E_CUDA (-2)      /* CUDA runtime error (no device, launch failure, ...) */
#define NCFA_E_WORKSPACE (-3) /* workspace too small */
#define NCFA_E_OVERFLOW (-4)  /* internal capacity exceeded (reported, never silent) */

#define NCFA_N_FFT 2048
#define NCFA_N_MELS 128

int ncfa_version(void);
const char *ncfa_last_error(void);

/* Optional per-kernel timing for bench.py: while enabled, every kernel launch is bracketed by CUDA
 * events on its stream; ncfa_profile_report() waits for them and writes "name,launches,total_ms"
 * lines into buf, then forgets them. */
void ncfa_profile_enable(int on);
int ncfa_profile_report(char *buf, size_t cap);
/* Same records as a timeline: "name,stream,t0_ms,t1_ms" per launch, relative to the first record (diagnostics:
 * where concurrent host workers leave the device idle).  Clears the records. */
int ncfa_profile_timeline(char *buf, size_t cap);

/* Build and upload the constant tables (Hann, FFT twiddles, Slaney mel bank for `sr`) on the
 * current device.  Idempotent and thread-safe; the other entry points call it lazily. */
int ncfa_init_tables(int sr);

/* Small parameter uploads (segment tables, priors, bootstrap values) that must not queue behind a
 * bulk host->device copy on the DMA engine: a kernel on `stream` reads `nbytes` from PINNED host
 * memory (cudaHostAlloc / torch pin_memory; checked with cudaHostGetDevicePointer) and writes
 * them to d_dst.  h_pinned_src must stay untouched until the stream has passed this call. */
int ncfa_param_upload(void *d_dst, const void *h_pinned_src, size_t nbytes, void *stream);

/* ---- io.py:38-40,94-110  _rms_db / slice_windows --------------------------------------------
 * d_meansq[i] = mean(x^2) of segment i accumulated in float64 (host finishes 20·log10(sqrt)). */
int ncfa_window_energy(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len, int n_seg,
                       double *d_meansq, void *stream);

/* ---- io.py:58-79 strip_silence → librosa.effects.trim; xcorr.py:210 librosa.feature.rms -------
 * d_rms[f] = sqrt(mean(frame^2)), centred frames of `frame_length`, zero padded, hop `hop`;
 * n_frames = 1 + n/hop.  float32 like librosa for float32 input. */
int ncfa_rms_frames(const float *d_audio, int64_t n, int frame_length, int hop, float *d_rms, void *stream);

/* Batched io.strip_silence bounds (io.py:58-79 → librosa.effects.trim(top_db), frame 2048 / hop 512): for every
 * segment d_bounds[2i] = start, d_bounds[2i+1] = end (samples, relative to the segment; (0, 0) when no frame is
 * above −top_db relative to the loudest frame).  One pass over the samples (512-sample block sums in float64). */
size_t ncfa_trim_workspace_bytes(int n_seg, int max_seg_len);
int ncfa_trim_bounds_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len, int n_seg,
                             int max_seg_len, double top_db, int64_t *d_bounds, void *d_workspace,
                             size_t workspace_bytes, void *stream);

/* ---- tempo.py:44,158  librosa.onset.onset_strength(y, sr, hop_length) -----------------------------
 * For each segment: STFT(2048, hop, periodic Hann, centred, zero pad) → |.|^2 → Slaney mel(128)
 * → 10·log10(max(1e-10,.)) → clamp to (max over the segment − 80 dB) → positive first difference
 * → mean over mels → left-pad 1 + 1024/hop zeros → n_frames = 1 + len/hop values.
 * d_onset_off[i] is the float offset of segment i's envelope inside d_onset.
 * Workspace: log-mel spectrogram of every segment + per-segment maxima. */
size_t ncfa_onset_workspace_bytes(int n_seg, int max_seg_len, int hop);
int ncfa_onset_strength_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len,
                                int n_seg, int max_seg_len, int hop, int sr, float *d_onset,
                                const int64_t *d_onset_off, void *d_workspace, size_t workspace_bytes,
                                void *stream);

/* ---- tempo.py:63-66  librosa.feature.tempo(onset_envelope, sr, hop_length, start_bpm) ----------
 * Mean over frames of the inf-normalised Hann-windowed autocorrelation tempogram
 * (win_length = floor(8·sr/hop)), log-normal prior around d_start_bpm[i] (std 1 octave), lags
 * with bpm >= 320 masked; d_lag[i] = argmax lag (bpm = 60·sr/(hop·lag)); 0 for an all-zero
 * envelope (beat_track returns (0.0, [])). */
size_t ncfa_tempo_workspace_bytes(int n_seg, int max_env_len, int win_length);
int ncfa_tempo_lag_batched(const float *d_onset, const int64_t *d_onset_off, const int32_t *d_env_len, int n_seg,
                           int max_env_len, int hop, int sr, const double *d_start_bpm, int32_t *d_lag,
                           void *d_workspace, size_t workspace_bytes, void *stream);

/* ---- tempo.py:45-49,159-164  librosa.beat.beat_track(onset_envelope, sr, hop_length, start_bpm) --
 * Dynamic-programming beat tracker with frames-per-beat = d_lag[i] <= max_lag (tightness 100, trim=True;
 * max_lag = the tempogram win_length floor(8·sr/hop) bounds every lag ncfa_tempo_lag_batched returns).
 * d_beats holds max_beats int32 frames per segment (ascending); d_n_beats[i] the count
 * (NCFA_E_OVERFLOW is flagged in d_n_beats[i] = -1 if max_beats is too small; the row then holds the first max_beats
 * beats).  A segment with d_lag[i] < 2, d_lag[i] > max_lag or d_env_len[i] < 2 gets d_n_beats[i] = 0 and its row of
 * d_beats is not written. */
size_t ncfa_beat_workspace_bytes(int n_seg, int max_env_len, int max_lag);
int ncfa_beat_track_batched(const float *d_onset, const int64_t *d_onset_off, const int32_t *d_env_len, int n_seg,
                            int max_env_len, const int32_t *d_lag, int max_lag, int32_t *d_beats, int max_beats,
                            int32_t *d_n_beats, void *d_workspace, size_t workspace_bytes, void *stream);

/* ---- consensus.py:243-267 _bootstrap_ratio, :270-312 compute_ibi_ratio, pitch.py:143-150 ---------
 * Job j resamples a_j (drawn FIRST) then b_j with numpy's Generator(PCG64).choice semantics
 * (32-bit Lemire bounded draws, low half of each 64-bit output first, high half buffered
 * across calls), n_boot times, starting from the PCG64 state {state_hi,state_lo,inc_hi,inc_lo}.
 *   boot[i] = median(a*) / median(b*)      (b_len = 0: boot[i] = median(a*))
 *   d_out[3j+0] = median(a)/median(b) (or median(a)),  [3j+1], [3j+2] = np.percentile(boot, q_lo/q_hi)
 * consensus._bootstrap_ratio(nc, src): a = nc, b = src.  compute_ibi_ratio(nc, src): a = src, b = nc.
 * d_boot (optional, n_jobs·n_boot doubles) receives the bootstrap replicates;
 * d_idx (optional, only when n_jobs == 1) receives every bounded draw in order (int32). */
size_t ncfa_bootstrap_workspace_bytes(int n_jobs, int max_a, int max_b, int n_boot);
int ncfa_bootstrap_ratio_batched(const double *d_a, const int64_t *d_a_off, const int32_t *d_a_len,
                                 const double *d_b, const int64_t *d_b_off, const int32_t *d_b_len, int n_jobs,
                                 int max_a, int max_b, int n_boot, const uint64_t h_pcg_state[4], double q_lo,
                                 double q_hi, double *d_out, double *d_boot, int32_t *d_idx, void *d_workspace,
                                 size_t workspace_bytes, void *stream);

/* ---- pitch.py:55-64 _mean_chroma → librosa.feature.chroma_cqt(y, sr, bins_per_octave=36, hop_length=512).mean(axis=1)
 * Step 1 (librosa.estimate_tuning inside cqt): STFT(2048, 512) magnitudes → piptrack peaks in
 * 150..4000 Hz → peaks at or above the segment's median magnitude → 100-bin histogram of the
 * 1/36-octave residual → d_tuning_idx[i] = first fullest bin j; tuning = −0.5 + j/100 (50 when the
 * segment has no peak, i.e. tuning 0.0). */
size_t ncfa_tuning_workspace_bytes(int n_seg, int max_seg_len);
int ncfa_tuning_estimate_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len, int n_seg,
                                 int max_seg_len, int sr, int32_t *d_tuning_idx, void *d_workspace,
                                 size_t workspace_bytes, void *stream);

/* Step 2: 7-octave, 36-bins/octave CQT from C1·2^(tuning/36) (rectangular 1024-sample frames, hop
 * 512 >> octave, 2:1 half-band decimation ×√2 between octaves, 1 %-sparsified FFT basis folded with
 * the DFT into one real 72×1024 matrix per tuning), |·|, fold to 12 chroma (3 bins per semitone,
 * rolled −1), inf-norm per frame, mean over frames → d_chroma[12·i .. 12·i+11] (float64).
 * sr must be 22050 (the layout the reference always uses: io.SAMPLE_RATE, io.py:19). */
size_t ncfa_chroma_workspace_bytes(int n_seg, int max_seg_len);
int ncfa_chroma_mean_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len, int n_seg,
                             int max_seg_len, int sr, const int32_t *d_tuning_idx, double *d_chroma,
                             void *d_workspace, size_t workspace_bytes, void *stream);

/* ---- pitch.py:67-85 _cyclic_xcorr_peak: d_lag[p] = first argmax_k dot(src_p, roll(nc_p, −k)),
 * wrapped to (−n_bins/2, n_bins/2]; d_src / d_nc hold n_pairs vectors of n_bins float64. */
int ncfa_cyclic_xcorr_batched(const double *d_src, const double *d_nc, int n_pairs, int n_bins, int32_t *d_lag,
                              void *stream);

/* ---- xcorr.py:113-148 candidate search of estimate_speed_xcorr.  Reference window w is
 * d_a[d_a_pos[w] .. +win); its candidates are d_b[d_b_lo[w] + j·stride .. +win), j < d_n_cand[w]
 * (the host applies xcorr.py:95-111,121-125 to produce these tables).  c = dot/(‖wa‖‖wb‖) with the
 * reference's float32 roundings of dot and norms; d_best_j[w] = first j with the largest c when it
 * is > 0 and the window passes the RMS gate (xcorr.py:118) and the 1e-10 norm gates, else −1;
 * d_best_c[w] = that c (0 when none).  (win, stride) picks the block form (win/stride <= 4 blocks and a tail of at
 * most 16 samples) or the direct form; the workspace size is the larger of the two layouts, so it holds either.  Until
 * the direct form was sized too, one window with max_cand <= 3 got 512 bytes instead of 768. */
size_t ncfa_xcorr_workspace_bytes(int n_windows, int max_cand);
int ncfa_xcorr_search_batched(const float *d_a, const float *d_b, const int64_t *d_a_pos, const int64_t *d_b_lo,
                              const int32_t *d_n_cand, int n_windows, int max_cand, int win, int stride,
                              double rms_gate, int32_t *d_best_j, double *d_best_c, void *d_workspace,
                              size_t workspace_bytes, void *stream);

/* ---- xcorr.py:165-259 find_content_offset (pipeline.run(auto_align=True)) -----------------------
 * ncfa_decimate2: librosa.resample(orig_sr = 2·target_sr) stand-in — 127-tap Kaiser half-band, no
 *   scaling, n_out = ceil(n_in/2) (soxr_hq is not reproducible; documented deviation).
 * ncfa_f32_to_f64: the .astype(np.float64) of the RMS envelopes (xcorr.py:210-211).
 * ncfa_align_search: for each candidate speed s: stretched = np.interp(linspace(0,1,n_stretched[s]),
 *   linspace(0,1,n_nc), nc_env); corr = np.correlate(src_env, stretched, 'valid')[:n_lags[s]];
 *   d_peak_idx[s] = first argmax; d_score[s] = corr[peak]/sqrt(Σ src_env[peak:peak+n]²·Σ stretched²)
 *   (0 when the denominator is <= 1e-12).  n_lags[s] <= 0 marks a speed the reference skips: its d_peak_idx is −1,
 *   its d_score 0, and its n_stretched is ignored (it may exceed max_stretched).  Every other speed needs
 *   1 <= n_stretched[s] <= max_stretched, n_lags[s] <= max_lags and n_stretched[s] + n_lags[s] − 1 <= n_src;
 *   n_stretched = 1 is the single point np.linspace(0, 1, 1) = [0], i.e. nc_env[0]. */
int ncfa_decimate2(const float *d_in, int64_t n_in, float *d_out, void *stream);
int ncfa_f32_to_f64(const float *d_in, int64_t n, double *d_out, void *stream);
size_t ncfa_align_workspace_bytes(int n_speeds, int max_stretched, int max_lags);
int ncfa_align_search(const double *d_src_env, int n_src, const double *d_nc_env, int n_nc,
                      const int32_t *d_n_stretched, const int32_t *d_n_lags, int n_speeds, int max_stretched,
                      int max_lags, int32_t *d_peak_idx, double *d_score, void *d_workspace, size_t workspace_bytes,
                      void *stream);

/* ---- spectral.py:54-96 spectral.analyze (SURVEY §8f row 3): whole-file statistics of |STFT(2048, 512, Hann)| --------
 * d_stats[16·i + s]: s = 0 Σ_frames spectral_centroid (Hz), 1 Σ_frames spectral_rolloff(0.85) (Hz), 2..6 Σ of |STFT| over
 * the bins of the bands 20–80, 80–250, 250–2000, 2000–6000, 6000–20000 Hz and all frames, 7 number of frames,
 * 8 max |STFT|.  d_bin_db_mean[1025·i + k] = mean over frames of amplitude_to_db(|STFT|, ref=max, top_db=80)[k].
 * Means are formed by the caller (centroid / frames, band sum / (bins·frames)). */
size_t ncfa_spectral_workspace_bytes(int n_seg);
int ncfa_spectral_stats_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len, int n_seg, int sr,
                                double *d_stats, float *d_bin_db_mean, void *d_workspace, size_t workspace_bytes,
                                void *stream);

/* ---- workflow.py:117 `sox SRC HQNC speed X`: band-limited speed change (the HQNC render) -------------------------
 * Output m of segment i is the segment evaluated at input time t = m·R, R = ratio[i] (sox `speed R`: pitch and tempo
 * both × R at the same sample rate), through a Kaiser-windowed sinc table T of Z zero crossings × L entries each:
 *   T[j] = sinc(j/L)·I0(β·sqrt(1 − (j/(Z·L))²))/I0(β), j < Z·L;  T[Z·L] = 0   (float64, built on the host)
 *   c = ρ/max(1, R), half = Z/c (input samples), n_out = ncfa_render_out_len(len, R) = len ? floor((len−1)/R) + 1 : 0
 *   per output, in float64 and in this order: t = (double)m·R; n0 = floor(t − half) + 1; for k = 0 .. ceil(2·half),
 *   n = n0 + k: d = (|t − n|·c)·L, i = floor(d), f = d − i; if i < Z·L and 0 <= n < len:
 *   acc += (T[i] + f·(T[i+1] − T[i]))·(double)x[n];  y[m] = (float)(acc·c).
 * Samples outside the segment count as zero.  Output i goes to d_out[d_out_off[i] ..  + n_out).  The ratios are passed
 * twice: d_ratio is what the kernel reads, h_ratio (host memory, the same values) is checked before the launch (finite,
 * in [0.25, 4]) so that a bad ratio is an NCFA_E_INVALID rather than a device-side condition.  max_seg_len bounds every
 * d_seg_len[i] and sizes the grid; n_seg <= 65535 per call.  No workspace. */
#define NCFA_RENDER_ZEROS 32
#define NCFA_RENDER_PHASES 512
#define NCFA_RENDER_BETA 10.0
#define NCFA_RENDER_ROLLOFF 0.95
int64_t ncfa_render_out_len(int32_t len, double ratio);
int ncfa_render_batched(const float *d_audio, const int64_t *d_seg_off, const int32_t *d_seg_len, const double *d_ratio,
                        const double *h_ratio, int n_seg, int max_seg_len, const int64_t *d_out_off, float *d_out,
                        void *stream);

/* Host-side constant-table builders (no GPU needed; used by the CPU test-suite):
 * h_K[1024][72] = the CQT contraction matrix of tuning index j; h_taps[127] = the half-band FIR. */
int ncfa_host_cqt_matrix(int sr, int tuning_index, float *h_K);
int ncfa_host_halfband_taps(double *h_taps);
/* h_table[Z·L + 1] = the float64 sinc table ncfa_render_batched reads (see above). */
int ncfa_host_render_table(double *h_table);
/* Lane-transposed Slaney mel bank of the STFT kernels: h_lane_bin0 int32[4][32] first bin read by lane l of
 * group q (bands l, 63-l, 64+l, 127-l), h_qw int32[4] rows per group, h_wt float32[128][32] weights
 * (row = group offset + i, column = lane; zero outside a band's support). */
int ncfa_host_mel_lanes(int sr, int32_t *h_lane_bin0, int32_t *h_qw, float *h_wt);

#ifdef __cplusplus
}
#endif
#endif /* NCFA_H */
