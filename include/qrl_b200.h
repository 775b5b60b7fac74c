/*
 * qrl_b200.h -- C ABI of libqrl_b200.so: batched-channel, B200-native replacements for the per-mode
 * GNU Radio hier-blocks that QRadioLink's gr_demod_base / gr_mod_base connect between the SDR
 * source/sink and the gr_*_sink / gr_*_source boundary blocks.
 *
 * Every entry point returns 0 on success or a negative QRL_E* code; no C++ exception crosses the ABI.
 * qrl_last_error() gives the message for the last failure on a handle (or the process-wide one for
 * create failures when handle == NULL).  One caller thread per handle (same contract as a GNU Radio
 * block's work(): /root/reference/src/gr/gr_bit_sink.h:36-38).
 *
 * What each entry point replaces in the reference:
 *   qrl_rx_create      make_gr_demod_nbfm / make_gr_demod_4fsk / make_gr_demod_qpsk ... factories
 *                      (src/gr/gr_demod_4fsk.h:51-53, gr_demod_qpsk.h:48-50, gr_demod_nbfm.h:38-39) as
 *                      instantiated by gr_demod_base.cpp:203-228, for n_channels independent channels.
 *   qrl_rx_work        the flattened hier-block's work()/general_work() calls for one chunk of the
 *                      1 Msps gr_complex stream (gr_demod_base.cpp:180 "demod_valve" -> hier block),
 *                      including the rotator_cc carrier shift (gr_demod_base.cpp:57,1220-1225).
 *   qrl_rx_read_port   what gr_const_sink / gr_audio_sink / gr_bit_sink (src/gr/gr_bit_sink.cpp:45-84,
 *                      gr_audio_sink.cpp:49-90) receive on output ports 0..3 of the hier block.
 *   qrl_rx_set_param   set_squelch / set_filter_width / set_agc_attack ... (gr_demod_nbfm.h:47-49).
 *   qrl_tx_create/work make_gr_mod_4fsk ... (src/gr/gr_mod_4fsk.h:46-48; gr_mod_base.cpp:155-180) fed by
 *                      gr_byte_source (src/gr/gr_byte_source.cpp:54-106).
 */
#ifndef QRL_B200_H
#define QRL_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QRL_OK 0
#define QRL_EINVAL (-22)      /* bad argument / unsupported mode */
#define QRL_ENOMEM (-12)
#define QRL_ECUDA (-5)        /* CUDA runtime error, see qrl_last_error */
#define QRL_ERANGE (-34)      /* chunk larger than the handle was created for */
#define QRL_ENODEV (-19)      /* no CUDA device: this library has no CPU fallback */

/* hier-block kinds: one per reference file src/gr/gr_demod_<x>.cpp / gr_mod_<x>.cpp */
enum qrl_kind {
    QRL_DEMOD_NBFM = 1, QRL_DEMOD_4FSK = 2, QRL_DEMOD_QPSK = 3, QRL_DEMOD_BPSK = 4, QRL_DEMOD_2FSK = 5,
    QRL_DEMOD_SSB = 6,
    QRL_DEMOD_AM = 7,         /* gr_demod_am.cpp:28-82 (SURVEY 8f row 3); ports: IQ, float audio at 8 ksps */
    QRL_DEMOD_M17 = 10,       /* gr_demod_m17.cpp:30-113 (SURVEY 8f row 3); ports: IQ at 24 ksps, symbols, hard bits (2 per symbol) */
    QRL_DEMOD_DMR = 11,       /* gr_demod_dmr.cpp:32-112 (SURVEY 8f row 3); qrl_rx_create ignores carrier_freq / filter_width / flag; ports: IQ at
                                 24 ksps, symbols, hard bits (2 per symbol), FLOAT symbol filter output (one per port-0 sample) */
    QRL_DEMOD_DSSS = 12,      /* gr_demod_dsss.cpp:32-124 (SURVEY 8f row 3; make_gr_demod_dsss(25, 1e6, 1700, 150)): Barker-13 BPSK at 16 symbols/s;
                                 ports: IQ at 5200 sps, symbols, decoded bits of the two decoders (4 ports like BPSK).  The despreader's
                                 look-back beyond its declared history is DEFINED as the stream's own older items (zeros at the start) */
    QRL_DEMOD_WBFM = 9,       /* gr_demod_wbfm.cpp:28-70 (SURVEY 8f row 3); ports: IQ at 200 ksps, float audio at 8 ksps */
    QRL_DEMOD_GMSK = 8,       /* gr_demod_gmsk.cpp:30-134 (SURVEY 8f row 3); sps 10 / 5 / 1 = GMSK1K / 2K / 10K; 4 ports like 2FSK */
    QRL_MOD_4FSK = 101, QRL_MOD_QPSK = 102, QRL_MOD_NBFM = 103, QRL_MOD_BPSK = 104, QRL_MOD_2FSK = 105,
    QRL_MOD_SSB = 106,
    QRL_MOD_GMSK = 107,       /* gr_mod_gmsk.cpp:30-100 (sps 50 / 100 / 10 = GMSK2K / 1K / 10K) */
    QRL_MOD_M17 = 108,        /* gr_mod_m17.cpp:30-95 (sps = 125: x125 / 3 from 24 ksps); items: frame bytes, 4 symbols each */
    QRL_MOD_DSSS = 110,       /* gr_mod_dsss.cpp:27-93 (make_gr_mod_dsss(25, 1e6, 1700, 200), gr_mod_base.cpp:170): one input byte = 208 chips = 10^6 output items, so
                                 max_items is small (the output buffer holds max_items x 8 MB per channel) */
    QRL_MOD_AM = 111,         /* gr_mod_am.cpp:25-72 (make_gr_mod_am(125, 1e6, 1700, 5000), gr_mod_base.cpp:167): float audio at 8 ksps in, like NBFM / SSB */
    QRL_MOD_DMR = 109         /* gr_mod_dmr.cpp:27-93 (the M17 modulator's structure with the DMR pulse, deviation 0.85 and
                                 gr_zero_idle_bursts in place of the IF low-pass; see qrl_tx_zero_samples) */
};

/* runtime parameters (qrl_rx_set_param / qrl_tx_set_param) */
enum qrl_param {
    QRL_PARAM_CARRIER_OFFSET_HZ = 1,  /* rotator_cc phase increment, gr_demod_base.cpp:1220-1225 */
    QRL_PARAM_SQUELCH_DB = 2,         /* gr_demod_nbfm::set_squelch */
    QRL_PARAM_FILTER_WIDTH = 3,       /* set_filter_width of gr_demod_nbfm / _ssb / _am / _wbfm (gr_demod_nbfm.cpp:82-90, gr_demod_ssb.cpp:89-101, ...);
                                         through qrl_tx_set_param: gr_mod_nbfm / _ssb / _am::set_filter_width (gr_mod_nbfm.cpp:78-93, gr_mod_ssb.cpp:85-100,
                                         gr_mod_am.cpp:75-85), mid-stream */
    QRL_PARAM_BB_GAIN = 4,            /* gr_mod_*::set_bb_gain */
    QRL_PARAM_CTCSS = 7,              /* gr_demod_nbfm::set_ctcss (gr_demod_nbfm.cpp:97-121): 0 = no tone squelch; f = analog::ctcss_squelch_ff(8000, f, 0.01,
                                         8000, 160, gate) in front of the audio filter (the audio stream shrinks while the tone is absent);
                                         through qrl_tx_set_param: gr_mod_nbfm::set_ctcss (gr_mod_nbfm.cpp:101-139) */
    QRL_PARAM_AGC_ATTACK = 8,         /* gr_demod_ssb::set_agc_attack / gr_demod_am::set_agc_attack (gr_demod_ssb.cpp:108-111, gr_demod_am.cpp:94-97) */
    QRL_PARAM_AGC_DECAY = 9,          /* gr_demod_ssb::set_agc_decay / gr_demod_am::set_agc_decay */
    QRL_PARAM_GAIN = 10,              /* gr_demod_ssb::set_gain (gr_demod_ssb.cpp:118-121): the IF gain in front of the side-band filter */
    QRL_PARAM_RSSI = 6,               /* 1: keep the RSSI tap of rssi_block.cpp:25-45 on port 0 up to date (read with qrl_rx_rssi) */
    QRL_PARAM_OVERLAP_CALLS = 5       /* 1: the loop / FEC tail of qrl_rx_work call k runs under the parallel stages of call
                                         k+1 (streaming use).  Output ports are double-buffered; the results of a call are
                                         ordered on the caller's stream only after qrl_rx_join (or qrl_rx_sync /
                                         qrl_rx_read_port, which wait on the host).  Supported for 4FSK (fm) blocks. */
};

typedef struct qrl_rx qrl_rx;
typedef struct qrl_tx qrl_tx;

/* library / device */
int  qrl_device_count(void);
const char* qrl_version(void);
const char* qrl_last_error(const void* handle);

/* ---- RX ----
 * kind, sps, samp_rate, carrier_freq, filter_width, flag: exactly the arguments of the reference factory
 *   (flag = `fm` for 4FSK/2FSK, `sb` for SSB, ignored otherwise).
 * n_channels independent channels; max_samples = largest T a single qrl_rx_work call will carry. */
int qrl_rx_create(int kind, int sps, int samp_rate, int carrier_freq, int filter_width, int flag,
                  int n_channels, long max_samples, int device, qrl_rx** out);
int qrl_rx_destroy(qrl_rx* h);
/* run all kernels of this handle on an existing CUDA stream (cudaStream_t); NULL = the handle's own stream */
int qrl_rx_set_stream(qrl_rx* h, void* cuda_stream);
int qrl_rx_set_param(qrl_rx* h, int channel /* -1 = all */, int key, double value);
int qrl_rx_reset(qrl_rx* h);
/* iq: [n_channels][T] interleaved float (re,im) = gr_complex; channel stride = `stride` complex samples.
 * on_device != 0: iq is a device pointer (already in HBM). Otherwise host memory (pinned or pageable);
 * the copy to the device is part of the call.  Asynchronous on the handle's stream. */
int qrl_rx_work(qrl_rx* h, const float* iq, long T, long stride, int on_device);
/* The same call fed with the SDR's wire format: interleaved int16 I/Q (UHD / SoapySDR "sc16": 4 bytes per sample, half the PCIe
 * traffic of gr_complex).  Each component becomes float(v) * scale on the device -- one rounding, the arithmetic of the host-side
 * converter that sits in front of the reference's uhd / osmosdr source blocks (gr_demod_base.cpp:166-196; UHD's sc16 -> fc32
 * scale is 1 / 32767) -- and the chain then runs exactly as qrl_rx_work on that gr_complex stream.  stride in int16 pairs. */
int qrl_rx_work_sc16(qrl_rx* h, const short* iq, long T, long stride, float scale, int on_device);
/* the same for 8-bit front ends (HackRF and other int8 sources of gr-osmosdr, 2 bytes per sample): float(v) * scale, stride in int8 pairs */
int qrl_rx_work_sc8(qrl_rx* h, const signed char* iq, long T, long stride, float scale, int on_device);
/* wait for everything submitted so far */
/* RSSI tap (SURVEY 8f row 4): per channel the value probe_signal_f holds behind rssi_block (|x|^2 -> moving_average(2000) ->
 * single_pole_iir(0.04) -> 10 log10 -> + level; /root/reference/src/gr/rssi_block.cpp:25-45, gr_demod_base.cpp:199-200) after the
 * last qrl_rx_work; rssi_db_host [n_channels]; needs QRL_PARAM_RSSI = 1 */
int qrl_rx_rssi(qrl_rx*, float level, float* rssi_db_host);
/* QRL_PARAM_OVERLAP_CALLS: make the handle's stream wait (on the device, without blocking the host) for everything the
 * calls so far have started; a no-op otherwise */
int qrl_rx_join(qrl_rx*);
int qrl_rx_sync(qrl_rx* h);
/* number of output ports (2 for analog blocks, 3 for 4FSK/QPSK, 4 for BPSK/2FSK) and item size in bytes */
int qrl_rx_num_ports(const qrl_rx* h);
int qrl_rx_port_itemsize(const qrl_rx* h, int port);
/* copy what the last qrl_rx_work call produced on `port` into dst[n_channels][cap] (items), and the
 * per-channel item counts into counts[n_channels].  dst_on_device selects a device destination. Syncs. */
int qrl_rx_read_port(qrl_rx* h, int port, void* dst, long cap, int* counts, int dst_on_device);
/* device-resident view of a port (no copy): pointer to [n_channels][*cap] items and the int counts array */
int qrl_rx_port_device(qrl_rx* h, int port, void** data, long* cap, int** counts);
/* kernels launched by this handle so far (for bench accounting) */
long qrl_rx_launch_count(const qrl_rx* h);
/* per-stage device timing: when enabled, every qrl_rx_work brackets each stage's kernels with CUDA events on
 * the handle's stream.  qrl_rx_profile_read syncs and returns the accumulated milliseconds and launch count of
 * `stage` (0 = stage-1 decimating FIR, 1 = channel filter, 2 = demod/shaping, 3 = loops/symbol sync, 4 = FEC)
 * since the last qrl_rx_profile(h, 1) call. */
/* SM partition in use: SMs reserved for the sequential loop/FEC kernels and SMs left to the parallel stages
 * (both 0 when the driver refused green contexts and plain priority streams are used instead) */
int qrl_rx_sm_partition(const qrl_rx* h, int* loop_sms, int* parallel_sms);
int qrl_rx_profile(qrl_rx* h, int enable);
int qrl_rx_profile_read(qrl_rx* h, int stage, double* ms_total, long* n_launches);

/* ---- TX ---- */
int qrl_tx_create(int kind, int sps, int samp_rate, int carrier_freq, int filter_width, int flag,
                  int n_channels, long max_items, int device, qrl_tx** out);
int qrl_tx_destroy(qrl_tx* h);
int qrl_tx_set_stream(qrl_tx* h, void* cuda_stream);
int qrl_tx_set_param(qrl_tx* h, int channel, int key, double value);
/* in: [n_channels][n] bytes (digital) ; produces [n_channels][n_out] gr_complex at 1 Msps */
int qrl_tx_work(qrl_tx* h, const void* in, long n, long stride, int on_device);
int qrl_tx_sync(qrl_tx* h);
int qrl_tx_read(qrl_tx* h, float* dst, long cap, long* n_out, int dst_on_device);
int qrl_tx_out_device(qrl_tx* h, float** data, long* stride, long* n_out);
long qrl_tx_launch_count(const qrl_tx* h);
/* QRL_MOD_DMR only: the "zero_samples" stream tag of gr_dmr_source.cpp:148 / gr_mmdvm_source.cpp:264, attached to byte
 * `byte_offset` (absolute position in the channel's input stream since create) with value n_samples; channel = -1: every channel.
 * At gr_zero_idle_bursts (gr_zero_idle_bursts.cpp:45-82) the tag sits on 24 ksps item 20 * byte_offset; `delay` = 62 items earlier
 * the block loads its counter with n_samples and clears one output item per count (a later tag overrides a running count; of two
 * tags on one item the first registered wins).  The block's history also delays the stream by 2 * 720 - 1 items (60 ms).
 * Register a tag before the qrl_tx_work call that feeds byte (byte_offset - 4): a tag whose start item has already been produced
 * clears only what is left of its count.  Deviation from the reference, on purpose: the reference drops a tag that falls into
 * the first 62 items of a scheduler window (its lookup is bounded by the current window); here results do not depend on chunking. */
int qrl_tx_zero_samples(qrl_tx* h, int channel, long long byte_offset, long n_samples);
/* per-stage device timing of the modulator (like qrl_rx_profile): stage 0 = bit chain (scrambler / encoder / mapper),
 * 1 = pulse shaping + frequency modulator, 2 = final interpolating FIR (the HBM-write-bound kernel) */
int qrl_tx_profile(qrl_tx* h, int enable);
int qrl_tx_profile_read(qrl_tx* h, int stage, double* ms_total, long* n_launches);

/* ---- front end at device rates >= 2 Msps ------------------------------------------------------------------------------------------
 * gr_demod_base::set_samp_rate (/root/reference/src/gr/gr_demod_base.cpp:1303-1362): when the device delivers samp_rate >= 2 Msps the
 * reference puts rational_resampler_ccf(1, samp_rate / 1e6, low_pass(1, samp_rate, 480000, 100000, BLACKMAN_HARRIS)) behind the
 * rotator (which then runs at the device rate, :1220-1225,1358) and in front of the demodulators.  This object is that pair for a batch
 * of channels: [n_channels][T] gr_complex at samp_rate in, [n_channels][T / N] at 1 Msps out -- the device-resident input layout of
 * qrl_rx_work.  Streaming (any chunking), phase-continuous retunes. */
typedef struct qrl_frontend qrl_frontend;
int  qrl_frontend_create(int samp_rate /* multiple of 1e6, >= 2e6 */, int n_channels, long max_in, int device, qrl_frontend** out);
int  qrl_frontend_destroy(qrl_frontend*);
int  qrl_frontend_set_stream(qrl_frontend*, void* cuda_stream);
int  qrl_frontend_set_carrier_offset(qrl_frontend*, int channel /* -1 = all */, double offset_hz);
int  qrl_frontend_work(qrl_frontend*, const float* iq, long T, long stride, int on_device, long* n_out);
int  qrl_frontend_out_device(qrl_frontend*, float** data, long* stride, long* n_out);
int  qrl_frontend_read(qrl_frontend*, float* dst /* [n_channels][cap] gr_complex */, long cap);
long qrl_frontend_launch_count(const qrl_frontend*);

/* ---- TX front end: 1 Msps -> device rate ------------------------------------------------------------------------------------------
 * gr_mod_base (/root/reference/src/gr/gr_mod_base.cpp:38,211-290,799-805) always runs mod -> rotator_cc(2 pi offset / 1e6) and, when
 * the sink runs at samp_rate >= 2 Msps, rational_resampler_ccf(N, 1, low_pass(N, samp_rate, 480000, 20000, BLACKMAN_HARRIS)) with
 * N = samp_rate / 1e6 in front of the sink (below 2 Msps the rotator feeds the sink directly).  This object is that pair for a batch
 * of channels: [n_channels][n] gr_complex at 1 Msps in (e.g. qrl_tx_out_device's buffer, on_device = 1), [n_channels][N n] items at
 * samp_rate out.  Definition: tests/txfront_ref.py -- exact Q32 NCO with phase = base + inc (n - n_base), inc = rint(offset / 1e6 2^32),
 * phase-continuous retunes; each output one sequential fma chain over the arm, oldest sample first.  Streaming: any chunking gives the
 * same stream.  samp_rate is 1e6 or a multiple of 1e6 in [2e6, 56e6]; anything else is QRL_EINVAL.
 * QRL_TXFRONT_SC16 stores per component (short) clamp(rintf(x * sc16_scale), -32768, 32767), interleaved I/Q: the arithmetic of a
 * SIMD fc32 -> sc16 converter with UHD's scale 32767.  That is a definition chosen here (UHD's converter is not in the reference tree
 * to pin it), like qrl_rx_work_sc16's.  It halves the HBM writes and the bytes that cross PCIe to the SDR. */
enum { QRL_TXFRONT_FC32 = 0, QRL_TXFRONT_SC16 = 1 };
typedef struct qrl_txfront qrl_txfront;
int  qrl_txfront_create(int samp_rate /* 1e6, or a multiple of 1e6 in [2e6, 56e6] */, int n_channels, long max_in /* 1 Msps items per call */,
                        int out_format, float sc16_scale, int device, qrl_txfront** out);
int  qrl_txfront_destroy(qrl_txfront*);
int  qrl_txfront_set_stream(qrl_txfront*, void* cuda_stream);
int  qrl_txfront_set_carrier_offset(qrl_txfront*, int channel /* -1 = all */, double offset_hz);
int  qrl_txfront_work(qrl_txfront*, const float* iq /* [C][stride] gr_complex at 1 Msps */, long n, long stride, int on_device, long* n_out);
int  qrl_txfront_out_device(qrl_txfront*, void** data, long* stride, long* n_out);
int  qrl_txfront_read(qrl_txfront*, void* dst /* [C][cap] items of the output format */, long cap);
long qrl_txfront_launch_count(const qrl_txfront*);

/* ---- design helpers (host only; the gr::filter::firdes calls the reference makes at construction /
 *      in set_filter_width, e.g. gr_demod_nbfm.cpp:82-90).  Return tap count or negative error. ---- */
int qrl_firdes_low_pass(double gain, double fs, double fc, double tw, int window, float* out, int cap);
int qrl_firdes_low_pass_2(double gain, double fs, double fc, double tw, double att_db, int window, float* out, int cap);
int qrl_firdes_band_pass(double gain, double fs, double lo, double hi, double tw, int window, float* out, int cap);
int qrl_firdes_complex_band_pass(double gain, double fs, double lo, double hi, double tw, int window, float* out, int cap);
int qrl_firdes_root_raised_cosine(double gain, double fs, double symrate, double alpha, int ntaps, float* out, int cap);
int qrl_firdes_gaussian(double gain, double spb, double bt, int ntaps, float* out, int cap);
int qrl_design_table(const char* name /* "atan","tanh","mmse","fxpt_sine" */, float* out, int cap);
int qrl_design_deemph(int fs, double tau, double* a2, double* b2);

/* ---- polyphase channelizer / synthesizer (SURVEY.md section 8f row 1) -------------------------------------------
 * Replaces gr::filter::pfb_channelizer_ccf::make(M, taps, 1.0) fed by blocks::stream_to_streams(M)
 * (/root/reference/src/gr/gr_demod_mmdvm_multi2.cpp:98-107) and gr::filter::pfb_synthesizer_ccf::make(M, taps, false)
 * (/root/reference/src/gr/gr_mod_mmdvm_multi2.cpp:90-92).  Streaming: history and samples that do not fill a frame
 * of M stay in the handle, results do not depend on chunking.  Channel c of the channelizer is centred on
 * +c*fs/M (ports M/2.. are the negative frequencies, the order both reference wirings rely on,
 * gr_demod_mmdvm_multi2.cpp:110-124).  The channelizer output [M][stride] gr_complex is exactly the device-resident
 * input layout of qrl_rx_work.
 * Commutator / timing (GNU Radio itself is not part of /root/reference, so this is restated, not pinned): with oversample rate 1.0
 * pfb_channelizer_ccf::general_work keeps its filter index at M-1 on every iteration, so stream j (sample x[mM + j] of
 * stream_to_streams) is filtered by branch M-1-j, taps[(M-1-j) + tM], at in[n] for every j and lands in FFT bin M-1-j of a backward
 * (e^{+j...}) FFT: u_k[m] = sum_t taps[k + tM] x[(m-t)M + (M-1-k)], out_c[m] = sum_k u_k[m] e^{+j 2 pi k c / M}.  Output column m
 * therefore needs wideband samples up to mM + M-1: the first column is produced once M samples have arrived.  A caller that
 * assumes a different commutator phase sees the same channels delayed / advanced by up to M-1 WIDEBAND samples (less than one
 * channel-rate sample), which the symbol-timing loops downstream absorb. */
enum { QRL_PFB_CHANNELIZER = 201, QRL_PFB_SYNTHESIZER = 202 };
typedef struct qrl_pfb qrl_pfb;
/* max_in: channelizer = wideband samples per call; synthesizer = columns (samples per channel) per call */
int  qrl_pfb_create(int kind, int M, const float* taps, int ntaps, long max_in, int device, qrl_pfb** out);
int  qrl_pfb_destroy(qrl_pfb*);
int  qrl_pfb_set_stream(qrl_pfb*, void* cuda_stream);
/* channelizer: in = n_in wideband gr_complex (in_stride ignored); *n_out = new samples per channel.
 * synthesizer: in = [M][in_stride] gr_complex, n_in columns; *n_out = n_in*M wideband samples.
 * in_on_device = 0: host memory (copied inside the call), 1: device pointer. Asynchronous on the handle's stream. */
int  qrl_pfb_work(qrl_pfb*, const void* in, long n_in, long in_stride, int in_on_device, long* n_out);
int  qrl_pfb_sync(qrl_pfb*);
/* device view of the last call's output: channelizer [M][*stride] gr_complex (*items valid columns),
 * synthesizer [*items] gr_complex; valid until the next qrl_pfb_work */
int  qrl_pfb_out_device(qrl_pfb*, void** data, long* stride, long* items);
/* copy the last call's output to host (channelizer: row c at host_dst + c*dst_stride items) and synchronise */
int  qrl_pfb_read(qrl_pfb*, void* host_dst, long dst_stride);
long qrl_pfb_launch_count(qrl_pfb*);

/* ---- MMDVM multi-channel front end: the per-channel chains either side of the filter bank ------------------------------------------
 * gr_demod_mmdvm_multi2 (/root/reference/src/gr/gr_demod_mmdvm_multi2.cpp:56-126; MMDVM_SAMPLE_RATE 250000, src/config_mmdvm.h:4) behind
 * qrl_pfb's channelizer: for channel c, row rows[c] of the [n_rows][stride] gr_complex slab at 25 ksps (NULL rows = identity; the
 * reference's port map is channels 0..3 on ports 0..3, 4.. on 9, 8, ..) -> rational_resampler_ccf(24, 25, low_pass_2(1, 600k, fw, 2000,
 * 60, BH)) -> low_pass_2(1, 24k, fw, 2000, 60, BH) -> rssi_tag_block (one dB value per 300 items, rssi_tag_block.cpp:42-63) ->
 * quadrature_demod_cf(24000 / (2 pi 12500)) -> x1.0 -> float_to_short(1, 32767): int16 [n_channels][*n_out] at 24 ksps, what
 * gr_mmdvm_sink takes.  No feedback loop anywhere: one thread per item in every stage; results are chunk invariant.
 * gr_mod_mmdvm_multi2 (gr_mod_mmdvm_multi2.cpp:47-126) in front of the synthesizer: int16 [n_channels][n] at 24 ksps -> short_to_float
 * (x (float)(1 / 32767): VOLK's SIMD form) -> x1.0 -> frequency_modulator_fc(2 pi 12500 / 24000) (Q32 phase, as the other modulators) ->
 * low_pass_2(1, 24k, ...) -> x0.8 -> rational_resampler_ccf(25, 24, low_pass_2(25, 600k, ...)) -> rows rows[c] of a zeroed [n_rows][stride]
 * slab at 25 ksps (the synthesizer's input; unused rows are the reference's null_source).  qrl_mmdvm_tx_finish applies what follows
 * the synthesizer, multiply_const_cc(1 / n_channels) and multiply_const_cc(bb_gain), in place on the wideband device buffer.
 * gr_zero_idle_bursts(0) (gr_mod_mmdvm_multi2.cpp:88,108-117; gr_mod_mmdvm.cpp:51-58) = qrl_mmdvm_tx_zero_samples below.
 * Not built: the MMDVM protocol sink / source (ZeroMQ, out of scope). */
typedef struct qrl_mmdvm_rx qrl_mmdvm_rx;
typedef struct qrl_mmdvm_tx qrl_mmdvm_tx;
/* variant 0: the per-channel chains of gr_demod_mmdvm_multi2 / gr_mod_mmdvm_multi2 described above (25 ksps <-> 24 ksps).
 * variant 1: the single-channel blocks gr_demod_mmdvm (gr_demod_mmdvm.cpp:30-64) / gr_mod_mmdvm (gr_mod_mmdvm.cpp:28-70) at
 * MMDVM_SAMPLE_RATE = 250 ksps: rational_resampler_ccf(12, 125, low_pass_2(12, 3 MHz, fw, 2000, 60, BH)), the RSSI tags taken in FRONT of the
 * channel filter, quadrature_demod_cf(24000 / (2 pi 10000)); TX: ... -> x0.8 -> x bb_gain -> rational_resampler_ccf(125, 12) (qrl_mmdvm_tx_finish
 * is not used there); n_channels independent streams are processed at once. */
int  qrl_mmdvm_rx_create(int variant, int n_channels, const int* rows, int n_rows, int filter_width, long max_in, int device, qrl_mmdvm_rx** out);
int  qrl_mmdvm_rx_destroy(qrl_mmdvm_rx*);
int  qrl_mmdvm_rx_set_stream(qrl_mmdvm_rx*, void* cuda_stream);
int  qrl_mmdvm_rx_calibrate_rssi(qrl_mmdvm_rx*, float level);              /* rssi_tag_block::calibrate_rssi */
int  qrl_mmdvm_rx_work(qrl_mmdvm_rx*, const float* iq, long n, long stride, int on_device, long* n_out);
int  qrl_mmdvm_rx_sync(qrl_mmdvm_rx*);
/* device views of the last call: int16 [n_channels][*stride], RSSI dB [n_channels][*rssi_stride] (*n_rssi values, the first one
 * belongs to 24 ksps item *first_rssi_item, the next ones follow every 300 items) */
int  qrl_mmdvm_rx_out_device(qrl_mmdvm_rx*, short** data, long* stride, long* n_out, float** rssi_db, long* rssi_stride, int* n_rssi,
                             long long* first_rssi_item);
int  qrl_mmdvm_rx_read(qrl_mmdvm_rx*, short* dst, long dst_stride, float* rssi_db, long rssi_cap, int* n_rssi, long long* first_rssi_item);
long qrl_mmdvm_rx_launch_count(qrl_mmdvm_rx*);
int  qrl_mmdvm_tx_create(int variant, int n_channels, const int* rows, int n_rows, int filter_width, long max_in, int device, qrl_mmdvm_tx** out);
int  qrl_mmdvm_tx_destroy(qrl_mmdvm_tx*);
int  qrl_mmdvm_tx_set_stream(qrl_mmdvm_tx*, void* cuda_stream);
int  qrl_mmdvm_tx_set_bb_gain(qrl_mmdvm_tx*, float gain);                   /* gr_mod_mmdvm_multi2::set_bb_gain */
/* The "zero_samples" stream tag of gr_mmdvm_source.cpp:264 as gr_zero_idle_bursts(0) consumes it (gr_zero_idle_bursts.cpp:47-86): from item
 * `item_offset` of the zero-idle block's OWN stream on, n_samples outputs of `channel` (-1: all) are cleared; a later tag overrides what is
 * left of a running count; counts carry across calls.  The block's stream is the 24 ksps stream behind the FM modulator for variant 1
 * (gr_mod_mmdvm: every block in front of it is 1:1, so item_offset is the index of the tagged int16 sample) and the 25 ksps stream behind
 * the x25/24 resampler for variant 0 (gr_mod_mmdvm_multi2: GNU Radio's scheduler moves a tag on input sample k across the resampler to item
 * floor(k * 25 / 24 + 1/2); the adapter applies that mapping, qradiolink_b200.mmdvm_tag_item does).  Register a tag before the
 * qrl_mmdvm_tx_work call that produces its item; one registered later clears what is left of its count. */
int  qrl_mmdvm_tx_zero_samples(qrl_mmdvm_tx*, int channel, long long item_offset, long n_samples);
int  qrl_mmdvm_tx_work(qrl_mmdvm_tx*, const short* in, long n, long stride, int on_device, long* n_out);
int  qrl_mmdvm_tx_sync(qrl_mmdvm_tx*);
int  qrl_mmdvm_tx_out_device(qrl_mmdvm_tx*, float** data, long* stride, long* n_out);      /* [n_rows][*stride] gr_complex */
int  qrl_mmdvm_tx_read(qrl_mmdvm_tx*, float* dst, long dst_stride);
int  qrl_mmdvm_tx_finish(qrl_mmdvm_tx*, float* wideband_dev, long n);
long qrl_mmdvm_tx_launch_count(qrl_mmdvm_tx*);

/* ---- display spectrum on the device (SURVEY.md section 8f row 4) -----------------------------------------------------------------
 * rx_fft_c (/root/reference/src/gr/rx_fft.cpp:44-129; gr_demod_base.cpp:166: 32768 points, Blackman-Harris; get_FFT_data :978-986) for
 * n_streams streams at once (the wideband source of a GPU, or every channel of a batch: [n_streams][stride] gr_complex like
 * qrl_rx_work).  One qrl_spectrum_work call is one rx_fft_c::work call: while disabled (the initial state) or while a finished spectrum
 * has not been fetched the whole call is dropped; otherwise samples x window fill the buffer and the first sample AFTER it filled
 * runs the forward FFT and volk_32fc_s32f_power_spectrum_32f(points, fft, N, N) (dB of |X / N|^2).  qrl_spectrum_get copies the points
 * fft-shifted (DC in the middle), *fft_size = N, or *fft_size = 0 when no spectrum is ready, and re-arms the block.
 * The FFT is hand-written (four-step, radix-2 stages in shared memory; no cuFFT).  Float result against the oracle's double-precision
 * definition: within 2e-4 dB on bins less than 40 dB below the strongest line, every bin's amplitude within 2e-6 of the peak
 * amplitude (FFTW's rounding cannot be reproduced either way).
 * fft_size: power of two in [256, 65536]; window_type: gr::fft::window::win_type (0 Hamming, 1 Hann, 2 Blackman, 3 rectangular,
 * 5 Blackman-Harris; out of range -> Hamming as rx_fft.cpp:176-179; Kaiser / Bartlett / flat-top are not built). */
typedef struct qrl_spectrum qrl_spectrum;
int  qrl_spectrum_create(int fft_size, int window_type, int n_streams, long max_samples, int device, qrl_spectrum** out);
int  qrl_spectrum_destroy(qrl_spectrum*);
int  qrl_spectrum_set_stream(qrl_spectrum*, void* cuda_stream);
int  qrl_spectrum_set_enabled(qrl_spectrum*, int enabled);            /* rx_fft_c::set_enabled */
int  qrl_spectrum_set_fft_size(qrl_spectrum*, int fft_size);          /* rx_fft_c::set_fft_size: buffer and ready flag reset */
int  qrl_spectrum_work(qrl_spectrum*, const float* iq, long T, long stride, int on_device);
int  qrl_spectrum_get(qrl_spectrum*, float* dst, long dst_stride, int dst_on_device, unsigned* fft_size);
long qrl_spectrum_launch_count(qrl_spectrum*);

/* ---- layer-1 deframer on the device (SURVEY.md section 8f row 2) -------------------------------------------------
 * Replaces gr_modem::synchronize / findSync / packBytes (/root/reference/src/gr_modem.cpp:1119-1282, 980-994) for a
 * batch of channels; sync words /root/reference/src/layer1framing.h:8-24.  sync_class: 4 = M17 (0x55F7 / 0xFF5D / 32-bit 0x555D555D,
 * gr_modem.cpp:1187-1207; bit_buf_len 46 * 8, rx_frame_length 46), 1 = "1K" modes (0xB5),
 * 2 = narrow modes (0xED89 voice + 24-bit text / proto / video / callsign / end), 3 = wide modes QPSK250K /
 * QPSKVideo / 4FSK100K (IP / video / end).  bit_buf_len / rx_frame_length as gr_modem::toggleRxMode sets them
 * (gr_modem.cpp:203-322), e.g. 64 / 7 for 4FSK-2k, 1517*8 / 1516 for QPSK-250k.  Input: one decoded bit per byte,
 * [n_channels][stride] with a per-channel count -- exactly qrl_rx_port_device(handle, 2, ...).  Output: per channel
 * up to max_frames records of qrl_deframer_record_bytes() bytes { uint32 frame_type (the sync word), uint32 nbytes,
 * payload }, the arguments of gr_modem::processReceivedData.  State (partial frames, shift register, _modem_sync)
 * carries across calls. */
typedef struct qrl_deframer qrl_deframer;
int  qrl_deframer_create(int sync_class, int bit_buf_len, int rx_frame_length, int n_channels, long max_bits, int max_frames,
                         int device, qrl_deframer** out);
int  qrl_deframer_destroy(qrl_deframer*);
int  qrl_deframer_set_stream(qrl_deframer*, void* cuda_stream);
/* bits [n_channels][stride], counts [n_channels]; on_device = 1: both are device pointers (e.g. from qrl_rx_port_device) */
int  qrl_deframer_work(qrl_deframer*, const unsigned char* bits, const int* counts, long stride, int on_device);
int  qrl_deframer_record_bytes(qrl_deframer*);
/* records_host [n_channels][max_frames][record_bytes] (may be NULL), frame_counts_host [n_channels],
 * modem_sync_host [n_channels] (may be NULL); synchronises */
int  qrl_deframer_read(qrl_deframer*, unsigned char* records_host, int* frame_counts_host, int* modem_sync_host);
int  qrl_deframer_out_device(qrl_deframer*, void** records, int** frame_counts);
int  qrl_deframer_sync(qrl_deframer*);
long qrl_deframer_launch_count(qrl_deframer*);
/* two candidate streams per channel (the two gr_deframer_bb outputs of a dual-decoder mode): like gr_modem::demodulate
 * (/root/reference/src/gr_modem.cpp:1066-1085) the LONGER one of a call is deframed, the first on a tie; same stride for both */
int  qrl_deframer_work2(qrl_deframer*, const unsigned char* bits_a, const int* counts_a, const unsigned char* bits_b, const int* counts_b,
                        long stride, int on_device);
/* frames found beyond max_frames since creation, per channel (they are not stored; frame_counts saturates at max_frames) */
int  qrl_deframer_dropped(qrl_deframer*, int* dropped_host);

/* ---- TX framing: gr_modem::frame (/root/reference/src/gr_modem.cpp:904-961) for a batch of channels -----------------------------------
 * payload [n_channels][payload_stride] with per-channel lengths and frame types (the sync words of layer1framing.h:8-24) ->
 * out [n_channels][out_stride] + lengths: [10 x 0xAA for an IP frame when burst_ip] + sync word (voice: 0xB5 when one_k_mode, else 0xED89
 * + reserved 0xAA; text / video / IP / proto: 24-bit word; other types: none) + payload -- the bytes qrl_tx_work takes.  on_device = 1:
 * all pointers are device pointers, the call is asynchronous on cuda_stream; 0: host pointers, synchronous. */
int  qrl_frame_build(int n_channels, const unsigned char* payload, long payload_stride, const int* payload_len, const unsigned* frame_type,
                     int one_k_mode, int burst_ip, unsigned char* out, long out_stride, int* out_len, int on_device, int device, void* cuda_stream);

/* ---- gr_deframer_bb on the device (/root/reference/src/gr/gr_deframer_bb.cpp:83-185) --------------------------------------------
 * The bit deframer behind ports 2 / 3 of the dual-decoder modes (BPSK, 2FSK, GMSK: gr_demod_base wires _deframer1/2 = type 1,
 * _deframer_700_1/2 = type 2, _deframer_10k_1/2 = type 3).  Input as qrl_deframer_work: one bit per byte, [n_channels][stride] with
 * per-channel counts -- exactly qrl_rx_port_device(handle, 2 or 3, ...).  Output: the stream get_data() hands to gr_modem: for every
 * sync word found, the word itself MSB first (16 bits, 24 for the End word, 8 for type 2) and the next 64 / 32 / 384 input bits;
 * [n_channels][out_stride] with per-channel counts, valid until the next call; feed it to qrl_deframer_work(2) on the device. */
typedef struct qrl_dfbb qrl_dfbb;
int  qrl_dfbb_create(int modem_type /* 1, 2, 3 */, int n_channels, long max_bits, int device, qrl_dfbb** out);
int  qrl_dfbb_destroy(qrl_dfbb*);
int  qrl_dfbb_set_stream(qrl_dfbb*, void* cuda_stream);
int  qrl_dfbb_work(qrl_dfbb*, const unsigned char* bits, const int* counts, long stride, int on_device);
int  qrl_dfbb_out_device(qrl_dfbb*, void** bits, long* stride, int** counts);
int  qrl_dfbb_read(qrl_dfbb*, unsigned char* out_host /* [n_channels][cap] */, long cap, int* counts_host);
int  qrl_dfbb_sync(qrl_dfbb*);
long qrl_dfbb_launch_count(qrl_dfbb*);

/* ---- stand-alone kernels exposed for tests / micro-benchmarks ---- */
/* batched decimating FIR (stage 1 alone): x [C][T] device, y [C][ceil(T/D)] device; zero history */
int qrl_fir_decim_ccf_device(const float* taps, int ntaps, int D, const float* x_dev, long T, long x_stride,
                             float* y_dev, long y_stride, int C, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif
