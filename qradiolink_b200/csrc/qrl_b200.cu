// qrl_b200.cu -- handles, stage orchestration and the C ABI (include/qrl_b200.h) of libqrl_b200.so.
//
// One qrl_rx handle = n_channels independent instances of ONE reference demod hier-block
// (/root/reference/src/gr/gr_demod_{nbfm,4fsk,qpsk}.cpp) running as batched CUDA kernels.  All
// per-channel DSP state (FIR history, resampler phase, loop filters, Viterbi start state, LFSR)
// lives in HBM between qrl_rx_work calls, so results do not depend on how the stream is chunked.
// There is NO CPU fallback: without a CUDA device every create call fails with QRL_ENODEV.
#include "../../include/qrl_b200.h"
#include "qrl_design.hpp"
#include "qrl_kernels.cuh"
#include "qrl_handle.hpp"

#include <cuda.h>

#include <algorithm>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

using namespace qrl;

namespace {

thread_local std::string g_err;
std::mutex g_tables_mu;
bool g_tables_done[16] = { false };     // per device ordinal (mod 16): lookup tables uploaded

#define CK(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e__ = (call);                                                                    \
        if (e__ != cudaSuccess) {                                                                    \
            set_err(h, std::string(#call) + ": " + cudaGetErrorString(e__));                         \
            return QRL_ECUDA;                                                                        \
        }                                                                                            \
    } while (0)

struct Ring {
    void* d = nullptr;
    unsigned mask = 0;
    long long stride = 0;   // items per channel (= capacity)
};

unsigned pow2_at_least(long long n)
{
    unsigned long long c = 64;
    while (c < static_cast<unsigned long long>(n)) c <<= 1;
    return static_cast<unsigned>(c);
}

using HandleBase = QrlHandleBase;       // qrl_handle.hpp: shared by every handle type of the library

void set_err(HandleBase* h, const std::string& s)
{
    g_err = s;
    if (h) h->err = s;
}

// a device pointer handed to a *_work call must live on the handle's device (a pointer from another GPU would fault inside a kernel
// long after the call returned)
int check_device_ptr(HandleBase* h, const void* p, const char* who)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return QRL_OK; }
    if (a.type == cudaMemoryTypeDevice && a.device != h->device) {
        set_err(h, std::string(who) + ": the device pointer belongs to GPU " + std::to_string(a.device) + ", the handle to GPU " + std::to_string(h->device));
        return QRL_EINVAL;
    }
    return QRL_OK;
}

int upload_tables(HandleBase* h)
{
    std::lock_guard<std::mutex> lk(g_tables_mu);
    if (g_tables_done[h->device & 15]) return QRL_OK;
    auto at = atan_table(); auto th = tanh_table(); auto mm = mmse_table(); auto sn = fxpt_sine_table();
    cudaError_t e = cudaMemcpyToSymbol(d_atan_tab, at.data(), at.size() * 4);
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(d_tanh_tab, th.data(), th.size() * 4);
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(d_mmse_tab, mm.data(), mm.size() * 4);
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(d_sine_tab, sn.data(), sn.size() * 4);
    if (e != cudaSuccess) { set_err(h, std::string("table upload: ") + cudaGetErrorString(e)); return QRL_ECUDA; }   // retried by the next create
    g_tables_done[h->device & 15] = true;
    return QRL_OK;
}

template <class T>
int dev_alloc(HandleBase* h, T** p, size_t n_items, bool zero = true)
{
    void* q = nullptr;
    size_t bytes = std::max<size_t>(n_items * sizeof(T), 16);
    cudaError_t e = cudaMalloc(&q, bytes);
    if (e != cudaSuccess) { set_err(h, std::string("cudaMalloc: ") + cudaGetErrorString(e)); return QRL_ENOMEM; }
    if (zero) {
        e = cudaMemsetAsync(q, 0, bytes, h->stream);
        if (e != cudaSuccess) { set_err(h, std::string("cudaMemset: ") + cudaGetErrorString(e)); return QRL_ECUDA; }
    }
    h->allocs.push_back(q);
    *p = static_cast<T*>(q);
    return QRL_OK;
}

int upload_floats(HandleBase* h, float** p, const std::vector<float>& v)
{
    int rc = dev_alloc(h, p, v.size(), false);
    if (rc) return rc;
    cudaError_t e = cudaMemcpy(*p, v.data(), v.size() * 4, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { set_err(h, std::string("tap upload: ") + cudaGetErrorString(e)); return QRL_ECUDA; }
    return QRL_OK;
}

}  // namespace

// =====================================================================================================
struct qrl_rx : HandleBase {
    int kind = 0, sps = 0, samp_rate = 0, carrier_freq = 0, filter_width = 0, flag = 0, C = 0;
    long Tmax = 0;
    int nports = 3;
    // stage 1 (rational_resampler_ccf(1, D))
    int D1 = 1, L1 = 1, Q1 = 1, ntaps1 = 0, H = 0, hist_cur = 0;
    float* d_taps1 = nullptr;
    float2* d_hist[2] = { nullptr, nullptr };
    float2* d_in_staging = nullptr;
    short2* d_in_sc16 = nullptr;        // qrl_rx_work_sc16 with a host buffer: the int16 slab as it arrived over PCIe
    long long n_in = 0, n1 = 0;       // stage-1 progress (absolute input samples consumed / outputs produced)
    long long n_in_s = 0, n1_s = 0;   // progress of the per-slice stages behind it (equal to the above between calls)
    bool fir_group_forced = false;     // QRL_FIR_GROUP given: keep it in overlap mode too
    int fir_group = 4;                 // stage-1 launches cover this many slices (bigger launches, same pipeline depth)
    Ring r1;
    // stage 2: channel / shaping filter on the complex stream (port 0)
    float* d_taps2 = nullptr; int ntaps2 = 0; size_t taps2_cap = 0;     // floats allocated for d_taps2 (set_filter_width redesigns)
    float if_gain = 0.9f;              // gr_demod_ssb: multiply_const_cc(0.9) in front of the side-band filter (set_gain)
    Ring r2;
    float2* d_port0 = nullptr; long port0_cap = 0; long port0_n = 0;
    // stage 3: quadrature demod + RRC (4FSK-FM)
    float* d_taps3 = nullptr; int ntaps3 = 0; float qd_gain = 0;
    Ring r4;
    // PSK chains: agc2 + costas "PLL" loop stage (per sample), output ring r3 (interleaved)
    AgcCostasParams acp{};
    AgcCostasState* d_ac = nullptr;
    // NBFM: de-emphasis recurrence in its own kernel on s_loop2 (overlaps the next slice's squelch recurrence)
    NbfmDeemphState* d_nb2 = nullptr; Ring raud; bool nbfm_split = false;
    // NBFM: stream between the 2/5 resampler and the audio filter (copy, or ctcss_squelch_ff after set_ctcss(f))
    Ring rq; NbfmCtcss ctc{}; double* d_cenv = nullptr;
    // gr_demod_dsss: one chain kernel behind stage 1 (dsss_chain_kernel)
    DsssParams dsp{}; DsssState* d_ds = nullptr; float* d_ds_arms = nullptr; float2* d_ds_taps = nullptr;
    Ring ds_a, ds_c, ds_d; long long ds_o_call0 = 0;
    Ring r3;
    int sym_sps = 0;
    // BPSK / 2FSK: fll_band_edge_cc + second (delayed) decoder
    FllParams fllp{};
    FllState* d_fll = nullptr; float2* d_fll_hist = nullptr; float* d_fll_taps = nullptr;
    Ring rf;                       // FLL output (channel-major complex)
    ViterbiState* d_vs2 = nullptr;
    unsigned char* d_port3 = nullptr; int* d_port3_cnt = nullptr;
    // front-end rotator (carrier offset)
    std::vector<RotState> rot; RotState* d_rot = nullptr; bool rot_active = false; float2* d_rot_buf = nullptr;
    bool rot_fused = false;            // this call: the rotator runs inside the stage-1 kernel (register-tiled shapes)
    // non-FM FSK detectors: band-pass bank + symbol filter
    float* d_bank_taps = nullptr; int nt_bank = 0;
    float* d_symf_taps = nullptr; int nt_symf = 0;
    Ring rbank;                    // bank output (complex for 4FSK, float for 2FSK), channel-major
    // SSB audio chain
    SsbParams ssbp{};
    SsbState* d_ssb = nullptr;
    Ring rclip, rstr;
    float* d_taps2c = nullptr;     // complex side-band filter taps
    // NBFM audio chain
    NbfmParams nbp{};
    NbfmState* d_nb = nullptr;
    Ring rg, rd, rr;
    float* d_env = nullptr; float* d_arm_taps = nullptr; float* d_audio_taps = nullptr;
    float* d_port1f = nullptr;
    int tsr = 0;
    std::vector<std::pair<void*, size_t>> zero_list;   // buffers qrl_rx_reset clears
    // symbol sync
    SymSyncParams ssp{};
    SymSyncState* d_ss = nullptr;
    float* d_ss_scratch = nullptr; int* d_ss_hdr = nullptr; long long ss_chunk_cap = 0, ss_chunk_off = 0;   // external symbol-sync epilogue
    cudaStream_t s_epi = nullptr;                        // wide-partition stream of the external epilogue
    bool gmsk = false;                                   // 2FSK code path running as gr_demod_gmsk (no FLL)
    bool m17 = false;                                    // 4FSK (fm) code path running as gr_demod_m17 (x3/125 front end, hard bits)
    int nt_arm1 = 0;                                     // taps per arm of a generic rational stage 1 (L1 > 1)
    bool dmr = false;                                    // M17 code path running as gr_demod_dmr (plain M&M detector, x0.9, float port 3)
    float* d_port3f = nullptr;                           // gr_demod_dmr port 3: symbol filter output, [C][port0_cap] floats
    // RSSI tap on port 0 (QRL_PARAM_RSSI): ring of |x|^2, carried IIR value, latest dB value per channel
    bool rssi_on = false; float* d_rssi_ring = nullptr; float* d_rssi_y = nullptr; float* d_rssi_db = nullptr; long long rssi_n = 0;
    // QRL_PARAM_OVERLAP_CALLS: the loop / FEC tail of call k runs under the parallel stages of call k+1.  Output ports
    // are double-buffered (alt_* = the buffers of the previous call), ring reuse is fenced slice by slice.
    bool many = false;                                   // many-channel geometry of the loop kernels (small windows, no SM partition)
    bool overlap = false;
    float2* alt_port0 = nullptr; float2* alt_port1 = nullptr; unsigned char* alt_port2 = nullptr; unsigned char* alt_port3 = nullptr;
    int *alt_port1_cnt = nullptr, *alt_port2_cnt = nullptr, *alt_port3_cnt = nullptr;
    long alt_port0_n = 0;
    cudaEvent_t ev_v[16] = { nullptr };                  // Viterbi of slice i done (kMaxSub entries)
    cudaEvent_t ev_tail[2][3] = { { nullptr } };         // s_loop / s_fec / s_epi at the end of a call, by call parity
    int call_parity = 0;
    long prev_T = -1;                  // length of the previous overlapped call (a change of length joins the tail, see qrl_rx_work)
    long long prev_k1[16] = { 0 }, cur_k1[16] = { 0 }; int prev_nsub = 0;      // stage-1 sample index at the end of each slice
    int ss_ch = 256;                                     // rows per symbol-sync window (256 x 3 stages or 512 x 2)
    float2* d_port1 = nullptr; long port1_cap = 0; int* d_port1_cnt = nullptr;
    Ring r5;   // soft bits (u8)
    ViterbiState* d_vs = nullptr;
    unsigned char* d_port2 = nullptr; long port2_cap = 0; int* d_port2_cnt = nullptr;
    long n1max = 0;
    // software pipeline inside one work() call: parallel stages on `stream`, loop stages on s_loop, FEC on s_fec
    static constexpr int kMaxSub = 16;
    int nsub = 12;
    bool nsub_forced = false;          // QRL_NSUB given
    cudaStream_t s_loop = nullptr, s_loop2 = nullptr, s_fec = nullptr;
    cudaEvent_t ev_start = nullptr, ev_a[kMaxSub] = { nullptr }, ev_b[kMaxSub] = { nullptr }, ev_c[kMaxSub] = { nullptr },
                ev_loop_done = nullptr, ev_loop2_done = nullptr, ev_fec_done = nullptr;
    long long* d_nsoft = nullptr;   // [kMaxSub][C] soft-bit write index snapshots
    // static SM partition (CUDA green contexts): the sequential loop / FEC kernels get a small private set of SMs so
    // their single dependent instruction streams never arbitrate with the FMA-bound FIR warps; the parallel stages
    // run on the remaining SMs through s_par.  Falls back to plain streams when the driver refuses.
    CUgreenCtx g_loop = nullptr, g_par = nullptr;
    cudaStream_t s_par = nullptr;
    cudaEvent_t ev_par_done = nullptr;
    int sm_loop = 0, sm_par = 0;
    cudaStream_t par() const { return s_par ? s_par : stream; }
    // optional per-stage device timing (qrl_rx_profile)
    bool prof = false;
    struct ProfRec { int stage; cudaEvent_t a, b; };
    std::vector<ProfRec> prof_recs; size_t prof_used = 0;
    double prof_ms[8] = { 0 }; long prof_n[8] = { 0 };
    cudaStream_t prof_stream = nullptr;
    cudaEvent_t prof_begin(int stage, cudaStream_t on = nullptr)
    {
        prof_stream = on ? on : stream;
        if (!prof) return nullptr;
        if (prof_used == prof_recs.size()) {
            ProfRec r{ stage, nullptr, nullptr };
            cudaEventCreate(&r.a); cudaEventCreate(&r.b);
            prof_recs.push_back(r);
        }
        ProfRec& r = prof_recs[prof_used];
        r.stage = stage;
        cudaEventRecord(r.a, prof_stream);
        return r.b;
    }
    void prof_end(cudaEvent_t b) { if (b) { cudaEventRecord(b, prof_stream); prof_used++; } }
};

namespace {

template <int D, int Q, int K, int NOUT, int NWARPS>
int launch_fir_poly(qrl_rx* h, const float2* iq, long long stride, long long T, long long k0, long long k1)
{
    constexpr int W = (NOUT + Q - 1) * D;
    const size_t smem = sizeof(float2) * ((W + 3) & ~1);
    static bool attr_done[16] = { false };
    if (!attr_done[h->device & 15]) {
        CK(cudaFuncSetAttribute(fir_decim_poly_kernel<D, Q, K, NOUT, NWARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[h->device & 15] = true;
    }
    const long long nout = k1 - k0;
    dim3 grid(static_cast<unsigned>((nout + NOUT - 1) / NOUT), h->C);
    fir_decim_poly_kernel<D, Q, K, NOUT, NWARPS><<<grid, NWARPS * 32, smem, h->par()>>>(
        iq, stride, T, h->d_hist[h->hist_cur], h->H, h->d_taps1,
        static_cast<float2*>(h->r1.d), h->r1.mask, h->r1.stride, h->n_in, k0, k1, h->rot_fused ? h->d_rot : nullptr);
    h->launches++;
    CK(cudaGetLastError());
    return QRL_OK;
}

template <int NTP, int K, int NTHREADS>
int launch_fir_d2(qrl_rx* h, const float2* iq, long long stride, long long T, long long k0, long long k1)
{
    constexpr int NOUT = NTHREADS * K;
    constexpr int W = 2 * (NOUT - 1) + NTP;
    const size_t smem = sizeof(float2) * (W + W / (2 * K) + 2);
    const long long nout = k1 - k0;
    dim3 grid(static_cast<unsigned>((nout + NOUT - 1) / NOUT), h->C);
    fir_decim2_kernel<NTP, K, NTHREADS><<<grid, NTHREADS, smem, h->par()>>>(
        iq, stride, T, h->d_hist[h->hist_cur], h->H, h->d_taps1,
        static_cast<float2*>(h->r1.d), h->r1.mask, h->r1.stride, h->n_in, k0, k1);
    h->launches++;
    CK(cudaGetLastError());
    return QRL_OK;
}

int launch_fir_resamp_2_25(qrl_rx* h, const float2* iq, long long stride, long long T, long long k0, long long k1)
{
    constexpr int L = 2, M = 25, NT = 105, NOUT = 512;
    constexpr int SPAN = (NOUT * M + L - 1) / L + NT + 1;
    const size_t smem = sizeof(float2) * SPAN;
    static bool attr_done[16] = { false };    // per device: function attributes belong to the device's context
    if (!attr_done[h->device & 15]) { CK(cudaFuncSetAttribute(fir_resamp_ccf_kernel<L, M, NT, NOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); attr_done[h->device & 15] = true; }
    dim3 grid(static_cast<unsigned>((k1 - k0 + NOUT - 1) / NOUT), h->C);
    fir_resamp_ccf_kernel<L, M, NT, NOUT><<<grid, 256, smem, h->par()>>>(iq, stride, T, h->d_hist[h->hist_cur], h->H, h->d_taps1,
        static_cast<float2*>(h->r1.d), h->r1.mask, h->r1.stride, h->n_in, k0, k1);
    h->launches++;
    CK(cudaGetLastError());
    return QRL_OK;
}

int stage1(qrl_rx* h, const float2* iq, long long stride, long long T, long long k0, long long k1)
{
    if (k1 <= k0) return QRL_OK;
    if (h->L1 == 2 && h->D1 == 25 && h->ntaps1 <= 210) return launch_fir_resamp_2_25(h, iq, stride, T, k0, k1);
    if (h->L1 > 2) {       // shape-generic rational resampler (M17: x3 / 125)
        const long long nout = k1 - k0;
        dim3 grid(static_cast<unsigned>((nout + 127) / 128), h->C);
        fir_resamp_hist_generic_kernel<<<grid, 128, 0, h->par()>>>(iq, stride, T, h->d_hist[h->hist_cur], h->H, h->d_taps1, h->nt_arm1,
            h->L1, h->D1, static_cast<float2*>(h->r1.d), h->r1.mask, h->r1.stride, h->n_in, k0, k1);
        h->launches++;
        CK(cudaGetLastError());
        return QRL_OK;
    }
    if (h->L1 != 1) { set_err(h, "stage-1 resampler shape not built"); return QRL_EINVAL; }
    if (h->D1 == 50 && h->Q1 == 9) return launch_fir_poly<50, 9, 8, 128, 8>(h, iq, stride, T, k0, k1);
    if (h->D1 == 100 && h->Q1 == 9) return launch_fir_poly<100, 9, 8, 64, 8>(h, iq, stride, T, k0, k1);     // 837 taps (4FSK-1k, QPSK-2k shape)
    if (h->D1 == 25 && h->Q1 == 9) return launch_fir_poly<25, 9, 8, 256, 8>(h, iq, stride, T, k0, k1);      // 209 taps (2FSK-2k)
    if (h->D1 == 125 && h->Q1 == 9) return launch_fir_poly<125, 9, 8, 48, 6>(h, iq, stride, T, k0, k1);     // 1045 taps (SSB)
    if (h->D1 == 25 && h->Q1 == 28) return launch_fir_poly<25, 28, 8, 192, 8>(h, iq, stride, T, k0, k1);    // 681 taps (QPSK-20k)
    if (h->D1 == 100 && h->Q1 == 28) return launch_fir_poly<100, 28, 8, 32, 4>(h, iq, stride, T, k0, k1);   // 2727 taps (QPSK-2k)
    if (h->D1 == 2 && h->ntaps1 <= 56) return launch_fir_d2<56, 8, 128>(h, iq, stride, T, k0, k1);
    if (h->L1 == 1) {      // no register-tiled instance for this shape: one thread per output, same order, same history
        const long long nout = k1 - k0;
        dim3 grid(static_cast<unsigned>((nout + 127) / 128), h->C);
        fir_decim_hist_generic_kernel<<<grid, 128, 0, h->par()>>>(iq, stride, T, h->d_hist[h->hist_cur], h->H, h->d_taps1, h->ntaps1, h->D1,
            static_cast<float2*>(h->r1.d), h->r1.mask, h->r1.stride, h->n_in, k0, k1);
        h->launches++;
        CK(cudaGetLastError());
        return QRL_OK;
    }
    set_err(h, "stage-1 resampler shape not built (L=" + std::to_string(h->L1) + ", D=" + std::to_string(h->D1) + ", taps=" + std::to_string(h->ntaps1) + ")");
    return QRL_EINVAL;
}

template <class F>
F drv(const char* name)
{
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult st;
    if (cudaGetDriverEntryPoint(name, &fn, cudaEnableDefault, &st) != cudaSuccess || st != cudaDriverEntryPointSuccess) return nullptr;
    return reinterpret_cast<F>(fn);
}

// split the device into {loop_sms} + {rest} and create the three internal streams; false -> caller falls back
bool make_sm_partition(qrl_rx* h, unsigned loop_sms, int prio, bool fec_on_par_default)
{
    if (const char* e = getenv("QRL_NO_SM_PARTITION")) { if (e[0] == '1') return false; }
    auto pDeviceGet = drv<CUresult (*)(CUdevice*, int)>("cuDeviceGet");
    auto pGetRes = drv<CUresult (*)(CUdevice, CUdevResource*, CUdevResourceType)>("cuDeviceGetDevResource");
    auto pSplit = drv<CUresult (*)(CUdevResource*, unsigned int*, const CUdevResource*, CUdevResource*, unsigned int, unsigned int)>("cuDevSmResourceSplitByCount");
    auto pDesc = drv<CUresult (*)(CUdevResourceDesc*, CUdevResource*, unsigned int)>("cuDevResourceGenerateDesc");
    auto pCreate = drv<CUresult (*)(CUgreenCtx*, CUdevResourceDesc, CUdevice, unsigned int)>("cuGreenCtxCreate");
    auto pStream = drv<CUresult (*)(CUstream*, CUgreenCtx, unsigned int, int)>("cuGreenCtxStreamCreate");
    if (!pDeviceGet || !pGetRes || !pSplit || !pDesc || !pCreate || !pStream) return false;
    CUdevice dev;
    if (pDeviceGet(&dev, h->device) != CUDA_SUCCESS) return false;
    CUdevResource all{}, grp{}, rest{};
    if (pGetRes(dev, &all, CU_DEV_RESOURCE_TYPE_SM) != CUDA_SUCCESS) return false;
    unsigned nb = 1;
    if (pSplit(&grp, &nb, &all, &rest, 0, loop_sms) != CUDA_SUCCESS || nb < 1) return false;
    CUdevResourceDesc d_loop, d_par;
    if (pDesc(&d_loop, &grp, 1) != CUDA_SUCCESS || pDesc(&d_par, &rest, 1) != CUDA_SUCCESS) return false;
    if (pCreate(&h->g_loop, d_loop, dev, CU_GREEN_CTX_DEFAULT_STREAM) != CUDA_SUCCESS) return false;
    if (pCreate(&h->g_par, d_par, dev, CU_GREEN_CTX_DEFAULT_STREAM) != CUDA_SUCCESS) return false;
    CUstream a = nullptr, b = nullptr, c = nullptr, d = nullptr;
    if (pStream(&a, h->g_loop, CU_STREAM_NON_BLOCKING, prio) != CUDA_SUCCESS) return false;
    // FEC (Viterbi) stream.  Up to 64 channels the step is the latency of the lone recurrence warps and the decoder runs on the wide
    // partition, off their SMs (64 ch x 2^22: 0.925 ms per call against 0.941 next to the loop kernels); with more channels the step is
    // the sum of the parallel stages and the decoder stays in the loop partition, out of their way (256 ch: 2.23 ms against 2.35).
    // profiles/r02_y_256ch_stage_times.txt; QRL_FEC_ON_PAR=0/1 forces either.
    bool fec_on_par = fec_on_par_default;
    if (const char* e = getenv("QRL_FEC_ON_PAR")) fec_on_par = e[0] == '1';
    if (pStream(&b, fec_on_par ? h->g_par : h->g_loop, CU_STREAM_NON_BLOCKING, prio) != CUDA_SUCCESS) return false;
    if (pStream(&d, h->g_loop, CU_STREAM_NON_BLOCKING, prio) != CUDA_SUCCESS) return false;
    if (pStream(&c, h->g_par, CU_STREAM_NON_BLOCKING, 0) != CUDA_SUCCESS) return false;
    CUstream e2 = nullptr;
    if (pStream(&e2, h->g_par, CU_STREAM_NON_BLOCKING, prio) != CUDA_SUCCESS) return false;
    h->s_loop = a; h->s_fec = b; h->s_par = c; h->s_loop2 = d; h->s_epi = e2;
    h->sm_loop = static_cast<int>(grp.sm.smCount); h->sm_par = static_cast<int>(rest.sm.smCount);
    return true;
}

// interleaved = channel-interleaved layout [ceil(C/32)][slots][32] (allocated for the padded channel count)
// digital::fll_band_edge_cc::design_filter restated: returns lower[2N] | upper[2N] (complex, stored reversed)
std::vector<float> fll_design(float sps, float rolloff, int N)
{
    auto sinc = [](double x) { return x == 0 ? 1.0 : std::sin(kPi * x) / (kPi * x); };
    std::vector<float> bb(N), t(4 * N);
    const int M = static_cast<int>(std::rint(N / sps));
    float power = 0;
    for (int i = 0; i < N; i++) {
        const float k = static_cast<float>(-M + i * 2.0 / sps);
        const float tap = static_cast<float>(sinc(rolloff * k - 0.5) + sinc(rolloff * k + 0.5));
        power += tap; bb[i] = tap;
    }
    const int Nh = static_cast<int>((N - 1.0) / 2.0);
    for (int i = 0; i < N; i++) {
        const float tap = bb[i] / power;
        const float k = static_cast<float>((-Nh + i) / (2.0 * sps));
        const float ang = static_cast<float>(2.0 * kPi * (1 + rolloff) * k);
        t[2 * (N - i - 1)] = tap * cosf(-ang); t[2 * (N - i - 1) + 1] = tap * sinf(-ang);
        t[2 * N + 2 * (N - i - 1)] = tap * cosf(ang); t[2 * N + 2 * (N - i - 1) + 1] = tap * sinf(ang);
    }
    return t;
}

int make_ring(qrl_rx* h, Ring* r, size_t isz, long long min_items, bool interleaved = false)
{
    unsigned cap = pow2_at_least(min_items);
    r->mask = cap - 1;
    r->stride = cap;
    unsigned char* p = nullptr;
    const size_t nch = interleaved ? static_cast<size_t>((h->C + 31) / 32) * 32 : static_cast<size_t>(h->C);
    const size_t bytes = static_cast<size_t>(cap) * isz * nch;
    int rc = dev_alloc(h, &p, bytes, true);
    r->d = p;
    if (!rc) h->zero_list.emplace_back(p, bytes);
    return rc;
}

// low-rate stream filters: register-tiled instances for real calls, the one-thread-per-output kernels for slivers
int launch_fir_ccf_c(HandleBase* h, int C, cudaStream_t st, const float2* in, unsigned in_mask, long long in_stride, float2* out, unsigned out_mask, long long out_stride,
                     const float* taps, int ntaps, long long a0, long long a1, float2* lin, long long lin_stride, long long lin_base, int interleaved);
int launch_fir_ccf(qrl_rx* h, cudaStream_t st, const float2* in, unsigned in_mask, long long in_stride, float2* out, unsigned out_mask, long long out_stride,
                   const float* taps, int ntaps, long long a0, long long a1, float2* lin, long long lin_stride, long long lin_base, int interleaved)
{
    return launch_fir_ccf_c(h, h->C, st, in, in_mask, in_stride, out, out_mask, out_stride, taps, ntaps, a0, a1, lin, lin_stride, lin_base, interleaved);
}
int launch_fir_ccf_c(HandleBase* h, int C_, cudaStream_t st, const float2* in, unsigned in_mask, long long in_stride, float2* out, unsigned out_mask, long long out_stride,
                     const float* taps, int ntaps, long long a0, long long a1, float2* lin, long long lin_stride, long long lin_base, int interleaved)
{
    struct CShim { int C; } hc{ C_ }; CShim* hC = &hc;
    const long long n = a1 - a0;
    if (n <= 0) return QRL_OK;
    constexpr int K = 8, NT = 128, TILE = K * NT;
    const int span = TILE + ntaps - 1;
    const size_t smem = sizeof(float) * ((ntaps + 1) & ~1) + sizeof(float2) * (span + (span >> 4) + 2);
    if (smem > 48 * 1024 && smem <= 100 * 1024) {            // long filters (gr_mod_am's 4545-tap output filter): opt in to the larger window once per device
        static bool big_attr[16] = { false };
        if (!big_attr[h->device & 15]) { CK(cudaFuncSetAttribute(fir_ccf_ring_tiled_kernel<K, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024)); big_attr[h->device & 15] = true; }
    }
    if (n >= 256 && smem <= 100 * 1024 && ntaps >= K) {      // (the tiled kernel's head / tail phases assume at least K taps)
        dim3 g(static_cast<unsigned>((n + TILE - 1) / TILE), hC->C);
        fir_ccf_ring_tiled_kernel<K, NT><<<g, NT, smem, st>>>(in, in_mask, in_stride, out, out_mask, out_stride, taps, ntaps, a0, a1, lin, lin_stride, lin_base, interleaved);
    } else {
        dim3 g(static_cast<unsigned>((n + 255) / 256), hC->C);
        fir_ccf_ring_kernel<<<g, 256, sizeof(float) * ntaps, st>>>(in, in_mask, in_stride, out, out_mask, out_stride, taps, ntaps, a0, a1, lin, lin_stride, lin_base, interleaved);
    }
    h->launches++;
    CK(cudaGetLastError());
    return QRL_OK;
}
int launch_qdemod_fir(qrl_rx* h, cudaStream_t st, const float2* in, unsigned in_mask, long long in_stride, float* out, unsigned out_mask, long long out_stride,
                      const float* taps, int ntaps, float gain, long long a0, long long a1)
{
    const long long n = a1 - a0;
    if (n <= 0) return QRL_OK;
    constexpr int K = 8, NT = 128, TILE = K * NT;
    const int span = TILE + ntaps - 1;
    const size_t smem = sizeof(float) * (ntaps + span + (span >> 5) + 2);
    if (n >= 256 && smem <= 48 * 1024 && ntaps >= K) {
        dim3 g(static_cast<unsigned>((n + TILE - 1) / TILE), h->C);
        qdemod_fir_fff_tiled_kernel<K, NT><<<g, NT, smem, st>>>(in, in_mask, in_stride, out, out_mask, out_stride, taps, ntaps, gain, a0, a1);
    } else {
        dim3 g(static_cast<unsigned>((n + 255) / 256), h->C);
        qdemod_fir_fff_kernel<<<g, 256, sizeof(float) * (2 * ntaps + 256), st>>>(in, in_mask, in_stride, out, out_mask, out_stride, taps, ntaps, gain, a0, a1, nullptr, 0);
    }
    h->launches++;
    CK(cudaGetLastError());
    return QRL_OK;
}

}  // namespace

// =====================================================================================================
// last-error hook for the other translation units of the library (qrl_pfb.cu)
void qrl_internal_set_err(const std::string& s) { g_err = s; }

extern "C" {

int qrl_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}
const char* qrl_version(void) { return "qrl_b200 0.1 (sm_100a)"; }
const char* qrl_last_error(const void* handle)
{
    if (handle) return static_cast<const HandleBase*>(handle)->err.c_str();
    return g_err.c_str();
}

int qrl_rx_create(int kind, int sps, int samp_rate, int carrier_freq, int filter_width, int flag,
                  int n_channels, long max_samples, int device, qrl_rx** out)
{
    if (!out || n_channels <= 0 || max_samples <= 0) { set_err(nullptr, "qrl_rx_create: bad argument"); return QRL_EINVAL; }
    *out = nullptr;
    if (qrl_device_count() <= device) { set_err(nullptr, "qrl_rx_create: no CUDA device (this library has no CPU fallback)"); return QRL_ENODEV; }
    // gr_demod_gmsk.cpp:30-134 is the 2FSK (fm) chain without the band-edge FLL, with a plain low-pass as symbol filter and its
    // own clock-loop constants: it runs through the 2FSK code path
    const bool gmsk = (kind == QRL_DEMOD_GMSK);
    if (gmsk) { kind = QRL_DEMOD_2FSK; flag = 1; }
    // gr_demod_m17.cpp:30-113 is the 4FSK (fm) chain behind a x3 / 125 rational resampler (24 ksps, 5 samples per symbol) with a
    // hard-decision bit tail instead of the FEC: it runs through the 4FSK code path
    // gr_demod_dmr.cpp:32-112 is that M17 chain again with its own stage-1 taps, no IF filter, a 0.2 roll-off symbol filter tapped as
    // (float) port 3, the PLAIN Mueller & Mueller detector in the symbol sync and x0.9 in front of the phase modulator
    const bool dmr = (kind == QRL_DEMOD_DMR);
    const bool m17 = (kind == QRL_DEMOD_M17) || dmr;
    if (m17) { kind = QRL_DEMOD_4FSK; flag = 1; }
    if (dmr) { carrier_freq = 0; filter_width = 5000; }
    qrl_rx* h = new qrl_rx();
    h->kind = kind; h->sps = sps; h->samp_rate = samp_rate; h->carrier_freq = carrier_freq;
    h->filter_width = filter_width; h->flag = flag; h->C = n_channels; h->Tmax = max_samples; h->device = device;
    h->gmsk = gmsk; h->m17 = m17; h->dmr = dmr;
    auto fail = [&](int rc) { std::string e = h->err; qrl_rx_destroy(h); g_err = e; return rc; };
    if (cudaSetDevice(device) != cudaSuccess) { set_err(h, "cudaSetDevice failed"); return fail(QRL_ECUDA); }
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { set_err(h, "stream create failed"); return fail(QRL_ECUDA); }
    h->own_stream = true;
    int rc = upload_tables(h);
    if (rc) return fail(rc);

    std::vector<float> taps1, taps2, taps3;
    int tsr = 0, sym_sps = 0;
    if (kind == QRL_DEMOD_4FSK) {
        // gr_demod_4fsk.cpp:46-84 (sps ladder), :98-107 (resampler), :108-109 (filter), :125-131 (demod, RRC, sync)
        int decimation = 1, interpolation = 1, nfilts = 0;
        if (dmr) { tsr = 24000; sym_sps = 5; decimation = 125; interpolation = 3; nfilts = 25 * sym_sps; }           // gr_demod_dmr.cpp:38-45
        else if (m17) { tsr = 24000; sym_sps = 5; decimation = 125; interpolation = 3; nfilts = 50 * sym_sps; }      // gr_demod_m17.cpp:37-48
        else if (sps == 1) { tsr = 80000; sym_sps = sps * 8; decimation = 25; interpolation = 2; nfilts = 32 * sym_sps; }
        else if (sps == 5) { tsr = 20000; sym_sps = sps * 2; decimation = 50; nfilts = 25 * sym_sps; }
        else if (sps == 10) { tsr = 10000; sym_sps = sps; decimation = 100; nfilts = 25 * sym_sps; }
        else if (sps == 2) { decimation = 2; sym_sps = 5; tsr = 500000; nfilts = 50 * sym_sps; }
        else { set_err(h, "make_gr_demod_4fsk: unsupported sps"); return fail(QRL_EINVAL); }
        if ((nfilts % 2) == 0) nfilts += 1;
        taps1 = dmr ? low_pass_2(3, 3.0 * samp_rate, 5000, 2000, 60, WIN_BLACKMAN_HARRIS)              // gr_demod_dmr.cpp:54-55
                    : low_pass(interpolation, static_cast<double>(interpolation) * samp_rate, tsr / 2, tsr / 2, WIN_BLACKMAN_HARRIS);
        h->D1 = decimation; h->L1 = interpolation;
        taps2 = dmr ? std::vector<float>{ 1.0f }                // no IF filter in gr_demod_dmr: the stage runs as a 1-tap pass-through
              : m17 ? low_pass(1, tsr, filter_width, filter_width, WIN_BLACKMAN_HARRIS)                 // gr_demod_m17.cpp:58-59
                    : low_pass(1, tsr, filter_width, filter_width / 2, WIN_BLACKMAN_HARRIS);
        taps3 = dmr ? root_raised_cosine(1, tsr, tsr / sym_sps, 0.2, nfilts)                            // gr_demod_dmr.cpp:61-62
                    : root_raised_cosine(1.5, tsr, tsr / sym_sps, m17 ? 0.5 : 0.2, nfilts);
        const float m17_rate = static_cast<float>(tsr) / static_cast<float>(sym_sps);
        h->qd_gain = dmr ? static_cast<float>(tsr / (kPi / 2 * m17_rate))                               // gr_demod_dmr.cpp:71
                         : static_cast<float>(sym_sps / (1 * kPi));
        const float dev = dmr ? 0.06f : (m17 ? 500.0f / m17_rate : 0.05f);                              // gr_demod_m17.cpp:67-70, gr_demod_dmr.cpp:68
        clock_loop_gains(dmr ? static_cast<float>(2 * kPi / 100.0f)
                             : (m17 ? static_cast<float>(2 * kPi / (m17_rate / 50)) : static_cast<float>(2 * kPi / 200.0f)), 1.0f, 0.2869f,
                         h->ssp.alpha, h->ssp.beta);
        if (dmr) h->ssp.sym_scale = 0.9f;                                                               // gr_demod_dmr.cpp:72
        h->ssp.sps = static_cast<float>(sym_sps);
        h->ssp.max_period = h->ssp.sps + dev; h->ssp.min_period = h->ssp.sps - dev;
        h->ssp.lookahead = 8 + static_cast<int>(ceilf(h->ssp.max_period)) + 1;
        h->ssp.pm_sens = static_cast<float>(kPi / 2);
        h->ssp.soft_scale = 128.0f;
        h->ssp.n0 = static_cast<int>(floorf(h->ssp.min_period - fabsf(h->ssp.alpha)));
        h->ssp.fl0 = static_cast<float>(h->ssp.n0);
        h->nports = dmr ? 4 : 3;
        if (!flag) {     // gr_demod_4fsk.cpp:110-124: four complex band-pass filters + discriminator + symbol filter
            int rs = 0, bw = 0;
            if (sps == 1) { rs = 10000; bw = 4000; } else if (sps == 5) { rs = 2000; bw = 4000; } else if (sps == 10) { rs = 1000; bw = 2000; }
            else { set_err(h, "make_gr_demod_4fsk: non-FM variant needs sps 1, 5 or 10"); return fail(QRL_EINVAL); }
            const int fw = filter_width;
            const double lo[4] = { double(-fw), double(-fw + rs), 0.0, double(fw - rs) }, hi[4] = { double(-fw + rs), 0.0, double(fw - rs), double(fw) };
            std::vector<float> bank;
            for (int b = 0; b < 4; b++) {
                std::vector<float> t = complex_band_pass(1, tsr, lo[b], hi[b], bw, WIN_BLACKMAN_HARRIS);
                h->nt_bank = static_cast<int>(t.size() / 2);
                bank.insert(bank.end(), t.begin(), t.end());
            }
            if ((rc = upload_floats(h, &h->d_bank_taps, bank))) return fail(rc);
            std::vector<float> sf = low_pass(1.0, tsr, tsr / sym_sps, tsr / sym_sps / 20, WIN_BLACKMAN_HARRIS);
            h->nt_symf = static_cast<int>(sf.size());
            if ((rc = upload_floats(h, &h->d_symf_taps, sf))) return fail(rc);
        }
    } else if (kind == QRL_DEMOD_QPSK) {
        // gr_demod_qpsk.cpp:46-71 (sps ladder), :98-103 (resampler), :106-110 (RRC), :104,113-118 (agc, sync, costas)
        int decimation; float costas_bw = static_cast<float>(kPi / 200);
        if (sps > 4 && sps < 125) { decimation = 25; sym_sps = sps * 4 / 25; tsr = 40000; }
        else if (sps >= 125) { decimation = 100; sym_sps = sps / 25; tsr = 10000; }
        else { decimation = 2; sym_sps = sps; tsr = 500000; costas_bw = static_cast<float>(kPi / 400); }
        if (sps > 4) {      // gr_demod_qpsk.cpp:105,130-134: FLL between the resampler and the shaping filter
            h->fllp.N = 32;
            control_loop_gains(static_cast<float>(2 * kPi / 100), h->fllp.alpha, h->fllp.beta);
            h->fllp.max_freq = static_cast<float>(2.0 * kPi * (2.0 / sym_sps)); h->fllp.min_freq = -h->fllp.max_freq;
        }
        taps1 = low_pass_2(1, static_cast<double>(samp_rate), tsr / 2, tsr / 10, 60, WIN_BLACKMAN_HARRIS);
        h->D1 = decimation;
        taps2 = root_raised_cosine(sym_sps, sym_sps, 1, 0.35, 11 * sym_sps);
        h->acp.attack = 1.0f; h->acp.decay = 1e-1f; h->acp.ref = 1.0f; h->acp.max_gain = 65536.0f;
        control_loop_gains(static_cast<float>(kPi / 200 / sym_sps), h->acp.alpha, h->acp.beta);
        h->acp.order = 4; h->acp.use_snr = 1;
        const float symbol_rate = static_cast<float>(tsr) / static_cast<float>(sym_sps);
        const float sps_dev = 200.0f / symbol_rate;
        clock_loop_gains(static_cast<float>(2 * kPi / (symbol_rate / 10)), 1.0f, 0.2869f, h->ssp.alpha, h->ssp.beta);
        h->ssp.sps = static_cast<float>(sym_sps);
        h->ssp.max_period = h->ssp.sps + sps_dev; h->ssp.min_period = h->ssp.sps - sps_dev;
        h->ssp.lookahead = 8 + static_cast<int>(ceilf(h->ssp.max_period)) + 1;
        control_loop_gains(costas_bw, h->ssp.costas_alpha, h->ssp.costas_beta);
        const float th = static_cast<float>(-3 * kPi / 4);
        h->ssp.rot_r = cosf(th); h->ssp.rot_i = sinf(th);
        h->ssp.soft_scale = 48.0f;
        h->ssp.n0 = static_cast<int>(floorf(h->ssp.min_period - fabsf(h->ssp.alpha)));
        h->ssp.fl0 = static_cast<float>(h->ssp.n0);
        h->nports = 3;
    } else if (kind == QRL_DEMOD_2FSK) {
        // gr_demod_2fsk.cpp:39-130 (fm variant)
        int decim, nfilts, interp = 1;
        if (sps == 10) { tsr = 20000; sym_sps = sps; decim = 50; nfilts = 35 * sym_sps; }
        else if (sps >= 5) { tsr = 40000; sym_sps = sps * 2; decim = 25; nfilts = 35 * sym_sps; }
        else if (sps == 1) { tsr = 80000; sym_sps = 4; decim = 25; interp = 2; nfilts = 125 * sym_sps; }
        else { set_err(h, "make_gr_demod_2fsk: unsupported sps"); return fail(QRL_EINVAL); }
        h->L1 = interp;
        if ((nfilts % 2) == 0) nfilts += 1;
        if (!flag) {     // gr_demod_2fsk.cpp:88-100: upper (-fw,0) / lower (0,fw) band filters, ratio detector, symbol filter
            std::vector<float> bank = complex_band_pass(1, tsr, -filter_width, 0, filter_width, WIN_BLACKMAN_HARRIS);
            std::vector<float> lower = complex_band_pass(1, tsr, 0, filter_width, filter_width, WIN_BLACKMAN_HARRIS);
            h->nt_bank = static_cast<int>(bank.size() / 2);
            bank.insert(bank.end(), lower.begin(), lower.end());
            if ((rc = upload_floats(h, &h->d_bank_taps, bank))) return fail(rc);
            std::vector<float> sf = low_pass(1.0, tsr, tsr / sym_sps, tsr / sym_sps, WIN_HAMMING);
            h->nt_symf = static_cast<int>(sf.size());
            if ((rc = upload_floats(h, &h->d_symf_taps, sf))) return fail(rc);
        }
        taps1 = low_pass(interp, static_cast<double>(interp) * samp_rate, tsr / 2, tsr / 2, WIN_BLACKMAN_HARRIS);
        h->D1 = decim;
        taps2 = low_pass(1, tsr, filter_width, filter_width, WIN_BLACKMAN_HARRIS);
        taps3 = gmsk ? low_pass(1, tsr, tsr / sym_sps, tsr / sym_sps, WIN_HAMMING)            // gr_demod_gmsk.cpp:88-90
                     : root_raised_cosine(1, tsr, tsr / sym_sps, 0.2, nfilts);
        h->qd_gain = static_cast<float>(sym_sps / (1 * kPi / 2));
        const float symbol_rate = static_cast<float>(tsr) / static_cast<float>(sym_sps);
        const float sps_dev = gmsk ? 0.05f : 200.0f / symbol_rate;                                    // gr_demod_gmsk.cpp:79-84
        clock_loop_gains(gmsk ? static_cast<float>(2 * kPi / 200.0f) : static_cast<float>(2 * kPi / (symbol_rate / 10)), 1.0f, 0.2869f,
                         h->ssp.alpha, h->ssp.beta);
        h->ssp.sps = static_cast<float>(sym_sps);
        h->ssp.max_period = h->ssp.sps + sps_dev; h->ssp.min_period = h->ssp.sps - sps_dev;
        h->ssp.lookahead = 8 + static_cast<int>(ceilf(h->ssp.max_period)) + 1;
        h->ssp.soft_scale = 128.0f;
        h->ssp.n0 = static_cast<int>(floorf(h->ssp.min_period - fabsf(h->ssp.alpha)));
        h->ssp.fl0 = static_cast<float>(h->ssp.n0);
        h->fllp.N = 16;
        control_loop_gains(static_cast<float>(24 * kPi / 100), h->fllp.alpha, h->fllp.beta);
        h->fllp.max_freq = static_cast<float>(2.0 * kPi * (2.0 / sym_sps)); h->fllp.min_freq = -h->fllp.max_freq;
        h->nports = 4;
    } else if (kind == QRL_DEMOD_BPSK) {
        // gr_demod_bpsk.cpp:40-76
        tsr = 20000; sym_sps = sps;
        taps1 = low_pass(1, samp_rate, tsr / 2, tsr / 2, WIN_BLACKMAN_HARRIS);
        h->D1 = 50;
        taps2 = root_raised_cosine(sps, sps, 1, 0.35, 15 * sps);
        h->acp.attack = 1e-1f; h->acp.decay = 1e-1f; h->acp.ref = 1.0f; h->acp.max_gain = 65536.0f; h->acp.order = 0;
        const float gain_mu = 0.05f, gain_omega = 0.005f;
        h->ssp.loop_kind = LOOP_CRMM;
        h->ssp.sps = static_cast<float>(sps);
        h->ssp.gain_omega = gain_omega * gain_omega; h->ssp.gain_mu = gain_mu;
        h->ssp.omega_mid = static_cast<float>(sps); h->ssp.omega_lim = 0.001f * static_cast<float>(sps);
        h->ssp.lookahead = 24;
        h->ssp.max_period = static_cast<float>(sps) + 1.0f; h->ssp.min_period = static_cast<float>(sps) - 1.0f;   // bounds for buffer sizing only
        h->ssp.alpha = 0.0f;
        control_loop_gains(static_cast<float>(2 * kPi / 200), h->ssp.costas_alpha, h->ssp.costas_beta);
        h->ssp.soft_scale = 64.0f;
        h->fllp.N = 32;
        control_loop_gains(static_cast<float>(8 * kPi / 100), h->fllp.alpha, h->fllp.beta);
        h->fllp.max_freq = static_cast<float>(2.0 * kPi * (2.0 / sps)); h->fllp.min_freq = -h->fllp.max_freq;
        h->nports = 4;
    } else if (kind == QRL_DEMOD_DSSS) {
        // gr_demod_dsss.cpp:32-124 (instance gr_demod_base.cpp:218: make_gr_demod_dsss(25, 1e6, 1700, 150)); sps = items per chip at 5200 sps
        tsr = 20000; sym_sps = 2;
        taps1 = low_pass(1, samp_rate, tsr / 2, tsr / 2, WIN_BLACKMAN_HARRIS);
        h->D1 = 50;
        const std::vector<float> tif = low_pass(1, 20000, 5200 / 2, 5200 / 2, WIN_BLACKMAN_HARRIS);       // rational_resampler_ccf(13, 50)
        taps2 = low_pass(1, 5200, filter_width, 1200, WIN_BLACKMAN_HARRIS);
        DsssParams& d = h->dsp;
        d.nt_arm = (static_cast<int>(tif.size()) + 12) / 13; d.nt2 = static_cast<int>(taps2.size());
        d.N = sps * 13; d.ntaps = d.N + 11 * sps;
        if (sps < 1 || d.nt_arm > 8 || d.nt2 > 64 || d.ntaps > 640 || d.N + d.ntaps - 1 > kDsssChunk) {
            set_err(h, "make_gr_demod_dsss: sps / filter_width outside what the chain kernel holds in shared memory"); return fail(QRL_EINVAL);
        }
        std::vector<float> arms(static_cast<size_t>(13) * d.nt_arm, 0.0f);
        for (int p = 0; p < 13; p++) for (int k = 0; k < d.nt_arm; k++) { const size_t j = p + static_cast<size_t>(k) * 13; if (j < tif.size()) arms[p * d.nt_arm + k] = tif[j]; }
        if ((rc = upload_floats(h, &h->d_ds_arms, arms))) return fail(rc);
        {   // dsss_decoder_cc_impl.cc:60-96: reversed Barker-13, `sps` items per chip, shaped by RRC(1, sps, 1, 0.35f, 11 sps); the block's
            // fir_filter_ccc keeps the taps reversed (what is uploaded)
            static const int barker_13[13] = { 1, 1, 1, 1, 1, 0, 0, 1, 1, 0, 1, 0, 1 };
            const int extra = 11 * sps, total = d.N + 2 * extra;
            std::vector<float> cs(total, 0.0f);
            for (int i = 0; i < 13; i++) { const float cv = barker_13[13 - (i + 1)] == 0 ? -1.0f : 1.0f; for (int k = 0; k < sps; k++) cs[extra + i * sps + k] = cv; }
            const std::vector<float> rrc = root_raised_cosine(1, sps, 1.0, static_cast<double>(0.350f), extra);
            const int nr = static_cast<int>(rrc.size());
            std::vector<float> t(2 * static_cast<size_t>(d.ntaps));
            for (int i = 0; i < d.ntaps; i++) {
                float acc = 0.0f, acci = 0.0f;
                for (int k = 0; k < nr; k++) { acc = acc + cs[i + k] * rrc[nr - 1 - k]; acci = acci + 0.0f * rrc[nr - 1 - k]; }
                t[2 * (d.ntaps - 1 - i)] = acc; t[2 * (d.ntaps - 1 - i) + 1] = acci;
            }
            float* tp = nullptr;
            if ((rc = upload_floats(h, &tp, t))) return fail(rc);
            h->d_ds_taps = reinterpret_cast<float2*>(tp);
        }
        control_loop_gains(static_cast<float>(kPi / 200), d.pll_alpha, d.pll_beta);
        control_loop_gains(static_cast<float>(2 * kPi / 100), d.costas_alpha, d.costas_beta);
        d.agc_attack = 1e-1f; d.agc_decay = 1e-1f; d.agc_ref = 1.0f; d.agc_max = 65536.0f;
        const float gain_mu = 0.05f, gain_omega = 0.005f;
        d.gain_omega = gain_omega * gain_omega; d.gain_mu = gain_mu; d.omega_mid = 1.0f; d.omega_lim = 0.005f * 1.0f; d.soft_scale = 64.0f;
        h->ssp.lookahead = 0; h->ssp.sps = 2.0f;
        h->nports = 4;
    } else if (kind == QRL_DEMOD_SSB) {
        // gr_demod_ssb.cpp:37-61; flag = sb (0 USB, 1 LSB); sps = decimation (125)
        tsr = 8000; sym_sps = 2;
        taps1 = low_pass(1, samp_rate, tsr / 2, tsr / 2, WIN_BLACKMAN_HARRIS);
        h->D1 = sps;
        taps2 = flag ? complex_band_pass_2(1, tsr, -filter_width, -200, 200, 90, WIN_BLACKMAN_HARRIS)
                     : complex_band_pass_2(1, tsr, 200, filter_width, 200, 90, WIN_BLACKMAN_HARRIS);
        h->nports = 2;
    } else if (kind == QRL_DEMOD_WBFM) {
        // gr_demod_wbfm.cpp:35-54
        tsr = 200000; sym_sps = 2;
        taps1 = low_pass(1, samp_rate, tsr / 2, tsr / 2, WIN_BLACKMAN_HARRIS);
        h->D1 = 5;
        taps2 = low_pass_2(1, tsr, filter_width, 600, 90, WIN_BLACKMAN_HARRIS);
        h->qd_gain = static_cast<float>(tsr / (2 * kPi * filter_width));
        h->nports = 2;
    } else if (kind == QRL_DEMOD_AM) {
        // gr_demod_am.cpp:35-56
        tsr = 20000; sym_sps = 2;
        taps1 = low_pass(1, samp_rate, tsr / 2, tsr / 2, WIN_BLACKMAN_HARRIS);
        h->D1 = 50;
        taps2 = complex_band_pass_2(1, tsr, -filter_width, filter_width, 200, 90, WIN_BLACKMAN_HARRIS);
        h->nports = 2;
    } else if (kind == QRL_DEMOD_NBFM) {
        // gr_demod_nbfm.cpp:39-66
        tsr = 20000; sym_sps = 2;
        taps1 = low_pass(1, samp_rate, tsr / 2, tsr / 2, WIN_BLACKMAN_HARRIS);
        h->D1 = 50;
        taps2 = low_pass_2(1, tsr, filter_width, 3500, 60, WIN_BLACKMAN_HARRIS);
        h->qd_gain = static_cast<float>(tsr / (4 * kPi * filter_width));
        h->nports = 2;
    } else {
        set_err(h, "qrl_rx_create: demod kind " + std::to_string(kind) + " not built");
        return fail(QRL_EINVAL);
    }
    h->sym_sps = sym_sps; h->tsr = tsr;

    // ---- stage 1 buffers
    h->ntaps1 = static_cast<int>(taps1.size());
    h->Q1 = (h->ntaps1 + h->D1 - 1) / h->D1;
    int padded = std::max(h->Q1 * h->D1, h->D1 == 2 ? 56 : 0);
    std::vector<float> tp(padded, 0.0f);
    std::copy(taps1.begin(), taps1.end(), tp.begin());
    if (h->L1 == 2) {       // rational_resampler arms: arm[p][k] = taps[p + k L], 105 taps per arm
        const int nt = 105;
        tp.assign(2 * nt, 0.0f);
        for (int p = 0; p < 2; p++) for (int k = 0; k < nt; k++) { const size_t j = p + 2 * k; if (j < taps1.size()) tp[p * nt + k] = taps1[j]; }
        padded = 128;       // history samples kept
    } else if (h->L1 > 2) {   // shape-generic rational resampler: arm[p][k] = taps[p + k L]
        const int nt = (static_cast<int>(taps1.size()) + h->L1 - 1) / h->L1;
        tp.assign(static_cast<size_t>(h->L1) * nt, 0.0f);
        for (int p = 0; p < h->L1; p++) for (int k = 0; k < nt; k++) { const size_t j = p + static_cast<size_t>(k) * h->L1; if (j < taps1.size()) tp[p * nt + k] = taps1[j]; }
        h->nt_arm1 = nt;
        padded = nt + 8;
    }
    if ((rc = upload_floats(h, &h->d_taps1, tp))) return fail(rc);
    h->H = padded;
    if ((rc = dev_alloc(h, &h->d_hist[0], static_cast<size_t>(h->H) * h->C))) return fail(rc);
    if ((rc = dev_alloc(h, &h->d_hist[1], static_cast<size_t>(h->H) * h->C))) return fail(rc);
    h->n1max = h->Tmax * h->L1 / h->D1 + 2;
    // ---- rings
    h->ntaps2 = static_cast<int>(taps2.size()) / ((kind == QRL_DEMOD_SSB || kind == QRL_DEMOD_AM) ? 2 : 1);
    h->ntaps3 = static_cast<int>(taps3.size());
    {
        std::vector<float> t2(std::max<size_t>(taps2.size(), 512), 0.0f);     // room for set_filter_width redesigns
        std::copy(taps2.begin(), taps2.end(), t2.begin());
        if ((rc = upload_floats(h, &h->d_taps2, t2))) return fail(rc);
        h->taps2_cap = t2.size();
    }
    if (!taps3.empty() && (rc = upload_floats(h, &h->d_taps3, taps3))) return fail(rc);
    if ((rc = make_ring(h, &h->r1, sizeof(float2), h->n1max + std::max(512, static_cast<int>(taps2.size())) + 8))) return fail(rc);
    if (kind == QRL_DEMOD_SSB) {
        if ((rc = make_ring(h, &h->r2, sizeof(float2), h->n1max + 64))) return fail(rc);
        std::vector<float> audio_f = band_pass_2(1, tsr, 200, filter_width, 200, 90, WIN_BLACKMAN_HARRIS);
        if ((rc = upload_floats(h, &h->d_audio_taps, audio_f))) return fail(rc);
        h->ssbp.sq_alpha = 0.01; h->ssbp.sq_threshold = std::pow(10.0, -140 / 10.0);
        h->ssbp.attack = 1e-1f; h->ssbp.decay = 1e-1f; h->ssbp.ref = 0.25f; h->ssbp.max_gain = 65536.0f;
        h->ssbp.clip = 0.95f; h->ssbp.emax = static_cast<float>(1 / (std::sqrt(0.5) / 2)); h->ssbp.out_gain = 1.333f;
        h->ssbp.nt_audio = static_cast<int>(audio_f.size());
        if ((rc = make_ring(h, &h->rclip, sizeof(float2), h->n1max + 16))) return fail(rc);
        if ((rc = make_ring(h, &h->rstr, sizeof(float), h->n1max + h->ssbp.nt_audio + 16))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_ssb, h->C))) return fail(rc);
    } else if (kind == QRL_DEMOD_WBFM) {
        // gr_demod_wbfm.cpp:39-64: the analog audio kernel in mode 2
        if ((rc = make_ring(h, &h->r2, sizeof(float2), h->n1max + 64))) return fail(rc);
        std::vector<float> audio_rs = low_pass(1, tsr, 4000, 2000, WIN_BLACKMAN_HARRIS);
        if ((rc = upload_floats(h, &h->d_audio_taps, audio_rs))) return fail(rc);
        if ((rc = upload_floats(h, &h->d_arm_taps, std::vector<float>{ 0.0f, 0.0f }))) return fail(rc);
        if ((rc = upload_floats(h, &h->d_env, std::vector<float>{ 1.0f, 1.0f }))) return fail(rc);
        double a[2], b[2];
        deemph_taps(8000, 50e-6, a, b);                        // the reference designs them for 8 kHz (:39) and runs them at 200 ksps
        h->nbp.sq_alpha = 0.01; h->nbp.sq_threshold = std::pow(10.0, -140 / 10.0); h->nbp.sq_ramp = 0; h->nbp.sq_gate = 1;
        h->nbp.qd_gain = h->qd_gain; h->nbp.nt_arm = 1; h->nbp.nt_audio = static_cast<int>(audio_rs.size());
        h->nbp.b0 = b[0]; h->nbp.b1 = b[1]; h->nbp.a1 = a[1]; h->nbp.out_gain = 1.0f;
        h->nbp.mode = 2; h->nbp.am_gain = 0.9f;
        if ((rc = make_ring(h, &h->rg, sizeof(float2), h->n1max + 16))) return fail(rc);
        if ((rc = make_ring(h, &h->rd, sizeof(float), h->n1max + 16))) return fail(rc);
        if ((rc = make_ring(h, &h->rr, sizeof(float), h->n1max + h->nbp.nt_audio + 16))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_nb, h->C))) return fail(rc);
    } else if (kind == QRL_DEMOD_AM) {
        // gr_demod_am.cpp:41-70: the NBFM audio kernel in detector mode 1
        if ((rc = make_ring(h, &h->r2, sizeof(float2), h->n1max + 64))) return fail(rc);
        std::vector<float> audio_rs = low_pass(2, 2 * tsr, 3600, 600, WIN_BLACKMAN_HARRIS);
        std::vector<float> audio_f = low_pass(1, 8000, 3600, 300, WIN_BLACKMAN_HARRIS);
        const int nt_arm = (static_cast<int>(audio_rs.size()) + 1) / 2;
        std::vector<float> arms(2 * nt_arm, 0.0f);
        for (int pp = 0; pp < 2; pp++)
            for (int k = 0; k < nt_arm; k++) { const size_t j = pp + 2 * k; arms[pp * nt_arm + k] = j < audio_rs.size() ? audio_rs[j] : 0.0f; }
        if ((rc = upload_floats(h, &h->d_arm_taps, arms))) return fail(rc);
        if ((rc = upload_floats(h, &h->d_audio_taps, audio_f))) return fail(rc);
        if ((rc = upload_floats(h, &h->d_env, std::vector<float>{ 1.0f, 1.0f }))) return fail(rc);
        h->nbp.sq_alpha = 0.01; h->nbp.sq_threshold = std::pow(10.0, -140 / 10.0); h->nbp.sq_ramp = 0; h->nbp.sq_gate = 1;
        h->nbp.qd_gain = 0.0f; h->nbp.nt_arm = nt_arm; h->nbp.nt_audio = static_cast<int>(audio_f.size());
        h->nbp.b0 = 1.0; h->nbp.b1 = -1.0; h->nbp.a1 = -0.9999; h->nbp.out_gain = 1.0f;      // iir_filter_ffd({1,-1},{0,0.9999}), old style
        h->nbp.mode = 1; h->nbp.agc_attack = 1e-1f; h->nbp.agc_decay = 1e-1f; h->nbp.agc_ref = 1.0f; h->nbp.agc_max = 65536.0f; h->nbp.am_gain = 0.99f;
        if ((rc = make_ring(h, &h->rg, sizeof(float2), 64))) return fail(rc);
        if ((rc = make_ring(h, &h->rd, sizeof(float), h->n1max + nt_arm + 16))) return fail(rc);
        if ((rc = make_ring(h, &h->rr, sizeof(float), h->n1max * 2 / 5 + h->nbp.nt_audio + 16))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_nb, h->C))) return fail(rc);
    } else if (kind == QRL_DEMOD_NBFM) {
        if ((rc = make_ring(h, &h->r2, sizeof(float2), h->n1max + 64))) return fail(rc);
        std::vector<float> audio_rs = low_pass_2(2, 2 * tsr, 3600, 250, 60, WIN_BLACKMAN_HARRIS);
        std::vector<float> audio_f = low_pass_2(1, 8000, 3500, 200, 35, WIN_BLACKMAN_HARRIS);
        const int nt_arm = (static_cast<int>(audio_rs.size()) + 1) / 2;
        std::vector<float> arms(2 * nt_arm, 0.0f);
        for (int pp = 0; pp < 2; pp++)
            for (int k = 0; k < nt_arm; k++) { const size_t j = pp + 2 * k; arms[pp * nt_arm + k] = j < audio_rs.size() ? audio_rs[j] : 0.0f; }
        if ((rc = upload_floats(h, &h->d_arm_taps, arms))) return fail(rc);
        if ((rc = upload_floats(h, &h->d_audio_taps, audio_f))) return fail(rc);
        const int ramp = 320;
        std::vector<float> env(ramp + 1);
        for (int k = 0; k <= ramp; k++) env[k] = static_cast<float>(0.5 - std::cos(kPi * k / ramp) / 2.0);
        if ((rc = upload_floats(h, &h->d_env, env))) return fail(rc);
        double a[2], b[2];
        deemph_taps(tsr, 50e-6, a, b);
        h->nbp.sq_alpha = 0.01; h->nbp.sq_threshold = std::pow(10.0, -140 / 10.0); h->nbp.sq_ramp = ramp; h->nbp.sq_gate = 1;
        h->nbp.qd_gain = h->qd_gain; h->nbp.nt_arm = nt_arm; h->nbp.nt_audio = static_cast<int>(audio_f.size());
        h->nbp.b0 = b[0]; h->nbp.b1 = b[1]; h->nbp.a1 = a[1]; h->nbp.out_gain = 2.0f;
        if ((rc = make_ring(h, &h->rg, sizeof(float2), h->n1max + 16))) return fail(rc);
        if ((rc = make_ring(h, &h->rd, sizeof(float), h->n1max + nt_arm + 16))) return fail(rc);
        if ((rc = make_ring(h, &h->rr, sizeof(float), h->n1max * 2 / 5 + h->nbp.nt_audio + 16))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_nb, h->C))) return fail(rc);
        if (kind == QRL_DEMOD_NBFM) {
            // analog::ctcss_squelch_ff::make(8000, 88.5, 0.01, 8000, 160, true) (gr_demod_nbfm.cpp:60), out of the graph until set_ctcss(f)
            if ((rc = make_ring(h, &h->rq, sizeof(float), h->n1max * 2 / 5 + h->nbp.nt_audio + 64))) return fail(rc);
            h->ctc.on = 0; h->ctc.len = 8000; h->ctc.ramp = 160; h->ctc.gate = 1; h->ctc.level = 0.01f;
            std::vector<double> ce(h->ctc.ramp + 1);
            for (int k = 0; k <= h->ctc.ramp; k++) ce[k] = 0.5 - std::cos(kPi * k / h->ctc.ramp) / 2.0;       // squelch_base_ff envelope (double)
            if ((rc = dev_alloc(h, &h->d_cenv, ce.size(), false))) return fail(rc);
            if (cudaMemcpy(h->d_cenv, ce.data(), sizeof(double) * ce.size(), cudaMemcpyHostToDevice) != cudaSuccess) { set_err(h, "envelope upload failed"); return fail(QRL_ECUDA); }
        }
        // (an FP64 instruction occupies an SM's FP64 pipe for ~64 cycles whatever its lane count, so two recurrences only overlap on
        // DIFFERENT SMs: both kernels then ask for more than half an SM's shared memory, which keeps their CTAs one per SM and apart, and
        // the split is used while 2 C CTAs fit the machine)
        if (kind == QRL_DEMOD_NBFM && 2 * h->C <= 140 && !getenv("QRL_NBFM_NO_SPLIT")) {
            if ((rc = make_ring(h, &h->raud, sizeof(float), h->n1max * 2 / 5 + 64))) return fail(rc);
            if ((rc = dev_alloc(h, &h->d_nb2, h->C))) return fail(rc);
            h->zero_list.emplace_back(h->d_nb2, sizeof(NbfmDeemphState) * h->C);
            h->nbfm_split = true;
        }
    } else if (kind == QRL_DEMOD_DSSS) {
        const long long n5 = h->n1max * 13 / 50 + 8;
        if ((rc = make_ring(h, &h->ds_a, sizeof(float2), n5 + 2048))) return fail(rc);
        if ((rc = make_ring(h, &h->ds_c, sizeof(float2), n5 + 2048))) return fail(rc);
        if ((rc = make_ring(h, &h->ds_d, sizeof(float2), n5 / h->dsp.N + 128))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_ds, h->C))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_vs2, h->C))) return fail(rc);
    } else if (kind == QRL_DEMOD_4FSK || kind == QRL_DEMOD_2FSK) {
        if ((rc = make_ring(h, &h->r2, sizeof(float2), h->n1max + h->ntaps3 + 64))) return fail(rc);
        // two calls deep when the block may run with overlapped calls (the producer of call k+1 must not wait for the
        // consumer of call k)
        if ((rc = make_ring(h, &h->r4, sizeof(float), (flag && kind == QRL_DEMOD_4FSK ? 2 : 1) * h->n1max + 600, true))) return fail(rc);
        if (flag && kind == QRL_DEMOD_4FSK) {
            // scratch of the external symbol-sync epilogue: [groups][chunks][maxs + 2][32] floats + a 128-int header per group
            // window size: 512 rows x 2 stages when the replicated interpolator bank still fits next to it, else 256 x 3
            {
                const int maxs512 = static_cast<int>((512 + 1) / (h->ssp.min_period - fabsf(h->ssp.alpha)) + 3);
                const size_t need512 = sizeof(float) * (2 * 512 * 32 + SYMSYNC_TAB_FLOATS + 2 * (maxs512 + 2) * 32) + sizeof(int) * 64 + 129 * 512;
                h->ss_ch = need512 <= 220 * 1024 ? 512 : 256;
            }
            if (const char* e = getenv("QRL_SS_CH")) { const int v = atoi(e); if (v == 512 || v == 256) h->ss_ch = v; }
            const int maxs = static_cast<int>((h->ss_ch + 1) / (h->ssp.min_period - fabsf(h->ssp.alpha)) + 3);
            h->ss_chunk_cap = h->n1max / symsync_stride(h->ss_ch, h->ssp.lookahead) + 4 + 3 * qrl_rx::kMaxSub;
            const size_t groups = (h->C + 31) / 32;
            if ((rc = dev_alloc(h, &h->d_ss_scratch, groups * h->ss_chunk_cap * (maxs + 2) * 32))) return fail(rc);
            if ((rc = dev_alloc(h, &h->d_ss_hdr, groups * 128 * qrl_rx::kMaxSub))) return fail(rc);
        }
        if (!flag) {
            if ((rc = make_ring(h, &h->rbank, kind == QRL_DEMOD_4FSK ? sizeof(float2) : sizeof(float), h->n1max + h->nt_symf + 16))) return fail(rc);
            if (kind == QRL_DEMOD_4FSK && (rc = make_ring(h, &h->r3, sizeof(float2), h->n1max + 600, true))) return fail(rc);
        }
    } else {   // QPSK / BPSK: shaping-filter output and loop output are channel-interleaved complex rings
        if ((rc = make_ring(h, &h->r2, sizeof(float2), h->n1max + 600, true))) return fail(rc);
        if ((rc = make_ring(h, &h->r3, sizeof(float2), h->n1max + 600, true))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_ac, h->C))) return fail(rc);
    }
    const bool has_fll = kind == QRL_DEMOD_BPSK || kind == QRL_DEMOD_2FSK || (kind == QRL_DEMOD_QPSK && sps > 4);
    if (has_fll) {
        const float fsps = static_cast<float>(sym_sps);
        std::vector<float> ft = fll_design(fsps, kind == QRL_DEMOD_2FSK ? 0.1f : 0.35f, h->fllp.N);
        if ((rc = upload_floats(h, &h->d_fll_taps, ft))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_fll, h->C))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_fll_hist, static_cast<size_t>(32) * h->C))) return fail(rc);
        h->zero_list.emplace_back(h->d_fll_hist, sizeof(float2) * 32 * h->C);
        h->zero_list.emplace_back(h->d_fll, sizeof(FllState) * h->C);
        if ((rc = make_ring(h, &h->rf, sizeof(float2), h->n1max + 512 + 8))) return fail(rc);
        if (kind != QRL_DEMOD_QPSK && (rc = dev_alloc(h, &h->d_vs2, h->C))) return fail(rc);
    }
    if ((rc = make_ring(h, &h->r5, 1, 2 * h->n1max + 1024))) return fail(rc);
    h->port0_cap = h->n1max;
    if ((rc = dev_alloc(h, &h->d_port0, static_cast<size_t>(h->port0_cap) * h->C))) return fail(rc);
    h->port1_cap = h->n1max / std::max(1, sym_sps - 1) + 64;
    if ((rc = dev_alloc(h, &h->d_port1, static_cast<size_t>(h->port1_cap) * h->C))) return fail(rc);
    h->d_port1f = reinterpret_cast<float*>(h->d_port1);
    if ((rc = dev_alloc(h, &h->d_port1_cnt, h->C))) return fail(rc);
    h->port2_cap = (h->m17 ? 2 : 1) * h->port1_cap + 160;      // M17: two hard bits per symbol, no rate-1/2 decoder behind them
    if ((rc = dev_alloc(h, &h->d_port2, static_cast<size_t>(h->port2_cap) * h->C))) return fail(rc);
    if ((rc = dev_alloc(h, &h->d_port2_cnt, h->C))) return fail(rc);
    if (h->dmr) {
        if ((rc = dev_alloc(h, &h->d_port3f, static_cast<size_t>(h->port0_cap) * h->C))) return fail(rc);
    } else if (h->nports == 4) {
        if ((rc = dev_alloc(h, &h->d_port3, static_cast<size_t>(h->port2_cap) * h->C))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_port3_cnt, h->C))) return fail(rc);
    }
    if ((rc = dev_alloc(h, &h->d_ss, h->C))) return fail(rc);
    if (h->ssp.lookahead > 0 && symsync_stride(128, h->ssp.lookahead) < 32 &&
        (kind == QRL_DEMOD_QPSK || kind == QRL_DEMOD_BPSK || (kind == QRL_DEMOD_4FSK && !flag))) {
        set_err(h, "symbol-sync lookahead does not fit the 128-row window of the complex-symbol kernels");
        return fail(QRL_EINVAL);
    }
    if ((rc = dev_alloc(h, &h->d_vs, h->C))) return fail(rc);
    if ((rc = dev_alloc(h, &h->d_nsoft, static_cast<size_t>(qrl_rx::kMaxSub) * h->C))) return fail(rc);
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        bool ok = true;
        // loop partition: one SM per big-shared-memory loop CTA (4FSK: symbol sync; QPSK: agc/costas + symbol sync)
        const int groups = (h->C + 31) / 32;
        // analog blocks: one CTA per channel whose thread 0 runs the double-precision recurrences (squelch power, de-emphasis): they want
        // an SM (its FP64 pipe) each, up to half the machine
        const bool analog_kind = kind == QRL_DEMOD_NBFM || kind == QRL_DEMOD_SSB || kind == QRL_DEMOD_AM || kind == QRL_DEMOD_WBFM;
        const int big_ctas = (kind == QRL_DEMOD_QPSK) ? 2 * groups : (analog_kind ? (h->nbfm_split ? 2 * h->C : std::min(h->C, 44)) : groups);
        unsigned loop_sms = static_cast<unsigned>(std::min(48, 8 * ((big_ctas + 4 + 7) / 8)));
        if (const char* e = getenv("QRL_LOOP_SMS")) { int v = atoi(e); if (v >= 8 && v <= 64) loop_sms = static_cast<unsigned>(v); }
        // Many channels (more loop CTAs than a 48-SM partition holds one per SM): the loop kernels have enough warps in flight to
        // hide their own latency, a private partition would only serialise them.  They then run with small windows (several CTAs
        // per SM) on all SMs, next to the parallel stages, on priority streams.
        h->many = big_ctas > 44 || (analog_kind && h->C > 64);
        if (const char* e = getenv("QRL_MANY_CHANNELS")) h->many = e[0] == '1';
        // QPSK (per-sample loops, 2 loop CTAs per 32 channels + a heavy Viterbi load): measured faster WITHOUT a private partition
        // (256 channels: 62.3 ms per 2^20-sample call on priority streams, 66.8 ms with a 24-SM partition -- the decoder gets the whole
        // machine (38.9 -> 12.9 ms) and the loop CTAs spread over more SMs); QRL_QPSK_PARTITION=1 brings the partition back.
        bool want_partition = kind != QRL_DEMOD_QPSK;
        if (const char* e = getenv("QRL_QPSK_PARTITION")) { if (kind == QRL_DEMOD_QPSK) want_partition = e[0] == '1'; }
        if (h->many || !want_partition || !make_sm_partition(h, loop_sms, hi, !analog_kind && groups <= 2)) {
            h->s_par = nullptr; h->sm_loop = 0; h->sm_par = 0;
            if (h->s_loop == nullptr)
                ok = cudaStreamCreateWithPriority(&h->s_loop, cudaStreamNonBlocking, hi) == cudaSuccess;
            if (h->s_loop2 == nullptr)
                ok = ok && cudaStreamCreateWithPriority(&h->s_loop2, cudaStreamNonBlocking, hi) == cudaSuccess;
            if (h->s_fec == nullptr)
                ok = ok && cudaStreamCreateWithPriority(&h->s_fec, cudaStreamNonBlocking, hi) == cudaSuccess;
            if (h->s_epi == nullptr)
                ok = ok && cudaStreamCreateWithPriority(&h->s_epi, cudaStreamNonBlocking, hi) == cudaSuccess;
        }
        auto mk = [&](cudaEvent_t* e) { ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess; };
        mk(&h->ev_start); mk(&h->ev_loop_done); mk(&h->ev_loop2_done); mk(&h->ev_fec_done); mk(&h->ev_par_done);
        for (int i = 0; i < qrl_rx::kMaxSub; i++) { mk(&h->ev_a[i]); mk(&h->ev_b[i]); mk(&h->ev_c[i]); }
        if (!ok) { set_err(h, "stream/event creation failed"); return fail(QRL_ECUDA); }
    }
    // QPSK: the call ends with the symbol sync + Viterbi of the last slice behind the per-sample loop (no overlapped calls for this
    // chain): the finest slicing the event arrays allow keeps that tail short
    if (kind == QRL_DEMOD_QPSK) h->nsub = qrl_rx::kMaxSub;
    if (const char* e = getenv("QRL_NSUB")) { int v = atoi(e); if (v >= 1 && v <= qrl_rx::kMaxSub) { h->nsub = v; h->nsub_forced = true; } }
    if (const char* e = getenv("QRL_FIR_GROUP")) { int v = atoi(e); if (v >= 1 && v <= qrl_rx::kMaxSub) { h->fir_group = v; h->fir_group_forced = true; } }
    if ((rc = qrl_rx_reset(h))) return fail(rc);
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) { set_err(h, "create sync failed"); return fail(QRL_ECUDA); }
    *out = h;
    return QRL_OK;
}

// host-side wait for everything a handle has in flight on its internal streams
static int rx_join_host(qrl_rx* h)
{
    if (h->s_loop) CK(cudaStreamSynchronize(h->s_loop));
    if (h->s_fec) CK(cudaStreamSynchronize(h->s_fec));
    if (h->s_loop2) CK(cudaStreamSynchronize(h->s_loop2));
    if (h->s_epi) CK(cudaStreamSynchronize(h->s_epi));
    if (h->s_par) CK(cudaStreamSynchronize(h->s_par));
    return QRL_OK;
}

int qrl_rx_reset(qrl_rx* h)
{
    if (!h) return QRL_EINVAL;
    if (h->s_loop) CK(cudaStreamSynchronize(h->s_loop));
    if (h->s_fec) CK(cudaStreamSynchronize(h->s_fec));
    if (h->s_loop2) CK(cudaStreamSynchronize(h->s_loop2));
    if (h->s_epi) CK(cudaStreamSynchronize(h->s_epi));
    if (h->s_par) CK(cudaStreamSynchronize(h->s_par));
    // all-zero history / rings; loop states at their constructor values
    std::vector<SymSyncState> ss(h->C);
    std::vector<ViterbiState> vs(h->C);
    for (int c = 0; c < h->C; c++) {
        std::memset(&ss[c], 0, sizeof(SymSyncState));
        ss[c].avg_period = h->ssp.sps; ss[c].inst_period = h->ssp.sps;
        ss[c].mu = (h->ssp.loop_kind == LOOP_CRMM) ? 0.5f : 0.0f;          // clock_recovery_mm_cc(omega, g_omega, mu = 0.5, ...)
        vs[c].rd = 0; vs[c].start_state = 0; vs[c].descr_reg = 0x7F;
    }
    CK(cudaMemcpyAsync(h->d_ss, ss.data(), sizeof(SymSyncState) * h->C, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_vs, vs.data(), sizeof(ViterbiState) * h->C, cudaMemcpyHostToDevice, h->stream));
    if (h->d_vs2) CK(cudaMemcpyAsync(h->d_vs2, vs.data(), sizeof(ViterbiState) * h->C, cudaMemcpyHostToDevice, h->stream));
    if (h->d_port3_cnt) CK(cudaMemsetAsync(h->d_port3_cnt, 0, sizeof(int) * h->C, h->stream));
    CK(cudaMemsetAsync(h->d_hist[0], 0, sizeof(float2) * h->H * h->C, h->stream));
    CK(cudaMemsetAsync(h->d_hist[1], 0, sizeof(float2) * h->H * h->C, h->stream));
    for (auto& z : h->zero_list) CK(cudaMemsetAsync(z.first, 0, z.second, h->stream));
    if (h->d_ds) {
        std::vector<DsssState> ds(h->C);
        for (int c = 0; c < h->C; c++) {
            std::memset(&ds[c], 0, sizeof(DsssState));
            ds[c].agc = 10.0f;                        // agc2_cc::make(1e-1, 1e-1, 1, 10): initial gain 10 (gr_demod_dsss.cpp:66)
            ds[c].omega = 1.0f; ds[c].mu = 0.5f;      // clock_recovery_mm_cc(1, ..., 0.5, ...)
        }
        CK(cudaMemcpyAsync(h->d_ds, ds.data(), sizeof(DsssState) * h->C, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        h->ds_o_call0 = 0;
    }
    std::vector<SsbState> sb(h->C);
    if (h->d_ssb) {
        for (int c = 0; c < h->C; c++) { std::memset(&sb[c], 0, sizeof(SsbState)); sb[c].sq_state = SQ_MUTED; sb[c].gain = 1.0f; }
        CK(cudaMemcpyAsync(h->d_ssb, sb.data(), sizeof(SsbState) * h->C, cudaMemcpyHostToDevice, h->stream));
    }
    std::vector<NbfmState> nb(h->C);
    if (h->d_nb) {
        for (int c = 0; c < h->C; c++) {
            std::memset(&nb[c], 0, sizeof(NbfmState));
            nb[c].sq_state = SQ_MUTED; nb[c].envelope = h->nbp.sq_ramp ? 0.0f : 1.0f; nb[c].agc_gain = 1.0f;
            nb[c].c_mute = 1; nb[c].c_state = SQ_MUTED; nb[c].c_env = h->ctc.ramp ? 0.0 : 1.0;      // ctcss_squelch_ff: d_mute(true), squelch_base_ff starts muted
        }
        CK(cudaMemcpyAsync(h->d_nb, nb.data(), sizeof(NbfmState) * h->C, cudaMemcpyHostToDevice, h->stream));
    }
    std::vector<AgcCostasState> ac(h->C);
    if (h->d_ac) {
        for (int c = 0; c < h->C; c++) { ac[c].pos = 0; ac[c].gain = 1.0f; ac[c].pll.phase = 0.0f; ac[c].pll.freq = 0.0f; }
        CK(cudaMemcpyAsync(h->d_ac, ac.data(), sizeof(AgcCostasState) * h->C, cudaMemcpyHostToDevice, h->stream));
    }
    CK(cudaMemsetAsync(h->d_port1_cnt, 0, sizeof(int) * h->C, h->stream));
    CK(cudaMemsetAsync(h->d_port2_cnt, 0, sizeof(int) * h->C, h->stream));
    CK(cudaStreamSynchronize(h->stream));   // the staging vectors above go out of scope
    h->n_in = 0; h->n1 = 0; h->n_in_s = 0; h->n1_s = 0; h->hist_cur = 0; h->port0_n = 0; h->prev_nsub = 0; h->rssi_n = 0;
    return QRL_OK;
}

int qrl_rx_destroy(qrl_rx* h)
{
    if (!h) return QRL_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->s_loop) { cudaStreamSynchronize(h->s_loop); cudaStreamDestroy(h->s_loop); }
    if (h->s_fec) { cudaStreamSynchronize(h->s_fec); cudaStreamDestroy(h->s_fec); }
    if (h->s_loop2) { cudaStreamSynchronize(h->s_loop2); cudaStreamDestroy(h->s_loop2); }
    if (h->s_epi) { cudaStreamSynchronize(h->s_epi); cudaStreamDestroy(h->s_epi); }
    if (h->s_par) { cudaStreamSynchronize(h->s_par); cudaStreamDestroy(h->s_par); }
    // every stream is idle now: the events recorded on them can go
    auto ev_free = [](cudaEvent_t e) { if (e) cudaEventDestroy(e); };
    for (cudaEvent_t e : { h->ev_start, h->ev_loop_done, h->ev_loop2_done, h->ev_fec_done, h->ev_par_done }) ev_free(e);
    for (int i = 0; i < qrl_rx::kMaxSub; i++) { ev_free(h->ev_a[i]); ev_free(h->ev_b[i]); ev_free(h->ev_c[i]); ev_free(h->ev_v[i]); }
    for (int q = 0; q < 2; q++) for (int j = 0; j < 3; j++) ev_free(h->ev_tail[q][j]);
    for (auto& r : h->prof_recs) { ev_free(r.a); ev_free(r.b); }
    if (h->g_loop || h->g_par) {
        auto pDestroy = drv<CUresult (*)(CUgreenCtx)>("cuGreenCtxDestroy");
        if (pDestroy) { if (h->g_loop) pDestroy(h->g_loop); if (h->g_par) pDestroy(h->g_par); }
    }
    for (void* p : h->allocs) cudaFree(p);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return QRL_OK;
}

int qrl_rx_set_stream(qrl_rx* h, void* s)
{
    if (!h) return QRL_EINVAL;
    CK(cudaStreamSynchronize(h->stream));
    if (h->own_stream && h->stream) { cudaStreamDestroy(h->stream); h->own_stream = false; }
    if (s) h->stream = static_cast<cudaStream_t>(s);
    else { CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); h->own_stream = true; }
    return QRL_OK;
}

int qrl_rx_set_param(qrl_rx* h, int channel, int key, double value)
{
    if (!h) return QRL_EINVAL;
    if (key == QRL_PARAM_RSSI) {
        if (value != 0.0 && !h->d_rssi_ring) {
            int rc;
            if ((rc = dev_alloc(h, &h->d_rssi_ring, static_cast<size_t>(4096) * h->C))) return rc;
            if ((rc = dev_alloc(h, &h->d_rssi_y, h->C))) return rc;
            if ((rc = dev_alloc(h, &h->d_rssi_db, h->C))) return rc;
            h->zero_list.emplace_back(h->d_rssi_ring, sizeof(float) * 4096 * h->C);
            h->zero_list.emplace_back(h->d_rssi_y, sizeof(float) * h->C);
            h->rssi_n = 0;
        }
        h->rssi_on = value != 0.0;
        return QRL_OK;
    }
    if (key == QRL_PARAM_OVERLAP_CALLS) {
        // only the path whose ring reuse is fenced for it: real-symbol 4FSK (external soft-bit epilogue)
        if (!(h->kind == QRL_DEMOD_4FSK && h->flag) || h->dmr) { set_err(h, "QRL_PARAM_OVERLAP_CALLS: not supported for this block"); return QRL_EINVAL; }
        CK(cudaStreamSynchronize(h->stream));
        { int rc = rx_join_host(h); if (rc) return rc; }
        const bool on = value != 0.0;
        if (on && !h->alt_port1) {
            int rc;
            if ((rc = dev_alloc(h, &h->alt_port0, static_cast<size_t>(h->port0_cap) * h->C))) return rc;
            if ((rc = dev_alloc(h, &h->alt_port1, static_cast<size_t>(h->port1_cap) * h->C))) return rc;
            if ((rc = dev_alloc(h, &h->alt_port2, static_cast<size_t>(h->port2_cap) * h->C))) return rc;
            if ((rc = dev_alloc(h, &h->alt_port1_cnt, h->C))) return rc;
            if ((rc = dev_alloc(h, &h->alt_port2_cnt, h->C))) return rc;
            if (h->d_port3) {
                if ((rc = dev_alloc(h, &h->alt_port3, static_cast<size_t>(h->port2_cap) * h->C))) return rc;
                if ((rc = dev_alloc(h, &h->alt_port3_cnt, h->C))) return rc;
            }
            for (int q = 0; q < 2; q++) for (int j = 0; j < 3; j++)
                if (!h->ev_tail[q][j]) CK(cudaEventCreateWithFlags(&h->ev_tail[q][j], cudaEventDisableTiming));
            for (int i = 0; i < qrl_rx::kMaxSub; i++)
                if (!h->ev_v[i]) CK(cudaEventCreateWithFlags(&h->ev_v[i], cudaEventDisableTiming));
            CK(cudaStreamSynchronize(h->stream));
        }
        h->overlap = on;
        return QRL_OK;
    }
    if (key == QRL_PARAM_CARRIER_OFFSET_HZ) {        // gr_demod_base::set_carrier_offset (:1220-1225): phase inc = 2 pi (-offset) / fs
        if (channel >= h->C) { set_err(h, "set_param: channel out of range"); return QRL_EINVAL; }
        if (h->rot.empty()) h->rot.assign(h->C, RotState{ 0u, 0u, 0 });
        const unsigned inc = static_cast<unsigned>(static_cast<int>(static_cast<long long>(std::rint(-value / h->samp_rate * 4294967296.0))));
        for (int c = 0; c < h->C; c++) {
            if (channel >= 0 && c != channel) continue;
            RotState& r = h->rot[c];
            r.base = r.base + r.inc * static_cast<unsigned>(h->n_in - r.n_base);     // keep the phase continuous
            r.n_base = h->n_in;
            r.inc = inc;
        }
        h->rot_active = false;
        for (auto& r : h->rot) if (r.inc != 0 || r.base != 0) h->rot_active = true;
        if (!h->d_rot) { int rc = dev_alloc(h, &h->d_rot, h->C); if (rc) return rc; }
        CK(cudaStreamSynchronize(h->stream));
        if (h->overlap) { int rc = rx_join_host(h); if (rc) return rc; }
        CK(cudaMemcpy(h->d_rot, h->rot.data(), sizeof(RotState) * h->C, cudaMemcpyHostToDevice));
        return QRL_OK;
    }
    // ---- run-time setters of the analog blocks.  Kernel parameters travel by value with every launch, so a plain host-side update is
    // enough for scalars; new taps are uploaded after everything in flight has drained and meet the true sample history (the rings)
    // from the next qrl_rx_work on.
    const bool nbfm = h->kind == QRL_DEMOD_NBFM, ssb = h->kind == QRL_DEMOD_SSB, am = h->kind == QRL_DEMOD_AM, wbfm = h->kind == QRL_DEMOD_WBFM;
    auto quiesce = [&]() -> int { CK(cudaStreamSynchronize(h->stream)); return rx_join_host(h); };
    auto upload = [&](float* dst, const std::vector<float>& t) -> int {
        int rc = quiesce(); if (rc) return rc;
        CK(cudaMemcpy(dst, t.data(), t.size() * 4, cudaMemcpyHostToDevice));
        return QRL_OK;
    };
    if (key == QRL_PARAM_SQUELCH_DB && (nbfm || ssb || am || wbfm)) {
        // gr_demod_nbfm::set_squelch (:92-95), gr_demod_ssb.cpp:103-106, gr_demod_am.cpp:104-107, gr_demod_wbfm.cpp:88-91: _squelch->set_threshold(dB)
        const double thr = std::pow(10.0, value / 10.0);
        if (ssb) h->ssbp.sq_threshold = thr; else h->nbp.sq_threshold = thr;
        return QRL_OK;
    }
    if (key == QRL_PARAM_AGC_ATTACK && (ssb || am)) {    // gr_demod_ssb::set_agc_attack (:108-111), gr_demod_am.cpp:94-97
        if (ssb) h->ssbp.attack = static_cast<float>(value); else h->nbp.agc_attack = static_cast<float>(value);
        return QRL_OK;
    }
    if (key == QRL_PARAM_AGC_DECAY && (ssb || am)) {     // gr_demod_ssb::set_agc_decay (:113-116), gr_demod_am.cpp:99-102
        if (ssb) h->ssbp.decay = static_cast<float>(value); else h->nbp.agc_decay = static_cast<float>(value);
        return QRL_OK;
    }
    if (key == QRL_PARAM_GAIN && ssb) { h->if_gain = static_cast<float>(value); return QRL_OK; }      // gr_demod_ssb::set_gain (:118-121): _if_gain->set_k
    if (key == QRL_PARAM_CTCSS && nbfm) {
        // gr_demod_nbfm::set_ctcss (:97-121).  0: tone squelch out of the graph, low-pass audio filter (only when it was in: the first
        // disconnect of :101 throws otherwise and the rest is skipped).  f: ctcss_squelch_ff::set_frequency(f) (new Goertzel filters at
        // the tone and its table neighbours, the block's squelch state is kept), and on the first switch the block goes in front of a
        // band-pass audio filter.
        if (value == 0.0) {
            if (!h->ctc.on) return QRL_OK;
            h->ctc.on = 0;
            return upload(h->d_audio_taps, low_pass_2(1, 8000, 3500, 200, 35, WIN_BLACKMAN_HARRIS));
        }
        static const float tones[38] = { 67.0f, 71.9f, 74.4f, 77.0f, 79.7f, 82.5f, 85.4f, 88.5f, 91.5f, 94.8f, 97.4f, 100.0f, 103.5f, 107.2f,
                                         110.9f, 114.8f, 118.8f, 123.0f, 127.3f, 131.8f, 136.5f, 141.3f, 146.2f, 151.4f, 156.7f, 162.2f, 167.9f,
                                         173.8f, 179.9f, 186.2f, 192.8f, 203.5f, 210.7f, 218.1f, 225.7f, 233.6f, 241.8f, 250.3f };
        const float freq = static_cast<float>(value);
        int idx = -1;
        for (int i = 0; i < 38; i++) if (tones[i] == freq) idx = i;
        const float fl = (idx == -1 || idx == 0) ? static_cast<float>(freq * 0.98) : tones[idx - 1];
        const float fr = (idx == -1 || idx == 37) ? static_cast<float>(freq * 1.02) : tones[idx + 1];
        auto gz = [](float f, float& wr, float& wi) { const float w = static_cast<float>(2.0 * kPi * f / 8000); wr = static_cast<float>(2.0 * std::cos(w)); wi = std::sin(w); };
        gz(fl, h->ctc.wr_l, h->ctc.wi_l); gz(freq, h->ctc.wr_c, h->ctc.wi_c); gz(fr, h->ctc.wr_r, h->ctc.wi_r);
        int rc = quiesce(); if (rc) return rc;
        {   // set_frequency makes new Goertzel objects: their running sums restart (the squelch state machine keeps its state)
            std::vector<NbfmState> stv(h->C);
            CK(cudaMemcpy(stv.data(), h->d_nb, sizeof(NbfmState) * h->C, cudaMemcpyDeviceToHost));
            for (auto& x : stv) { x.gl1 = x.gl2 = x.gc1 = x.gc2 = x.gr1 = x.gr2 = 0.0f; x.g_processed = 0; }
            CK(cudaMemcpy(h->d_nb, stv.data(), sizeof(NbfmState) * h->C, cudaMemcpyHostToDevice));
        }
        if (!h->ctc.on) {
            h->ctc.on = 1;
            return upload(h->d_audio_taps, band_pass_2(1, 8000, 300, 3500, 200, 35, WIN_BLACKMAN_HARRIS));
        }
        return QRL_OK;
    }
    if (key == QRL_PARAM_FILTER_WIDTH && (nbfm || ssb || am || wbfm)) {
        const int fw = static_cast<int>(value);
        if (fw <= 0) { set_err(h, "set_filter_width: out of range"); return QRL_EINVAL; }
        std::vector<float> t;
        if (nbfm || wbfm) t = low_pass(1, h->tsr, fw, 1200, WIN_BLACKMAN_HARRIS);                       // gr_demod_nbfm.cpp:82-90, gr_demod_wbfm.cpp:77-85
        else if (am) t = complex_band_pass(1, h->tsr, -fw, fw, 1200, WIN_BLACKMAN_HARRIS);              // gr_demod_am.cpp:84-92
        else t = h->flag ? complex_band_pass_2(1, h->tsr, -fw, -200, 200, 90, WIN_BLACKMAN_HARRIS)      // gr_demod_ssb.cpp:89-101
                         : complex_band_pass_2(1, h->tsr, 200, fw, 200, 90, WIN_BLACKMAN_HARRIS);
        if (t.size() > h->taps2_cap) { set_err(h, "set_filter_width: out of range (filter longer than the block was sized for)"); return QRL_EINVAL; }
        int rc = upload(h->d_taps2, t); if (rc) return rc;
        h->ntaps2 = static_cast<int>(t.size()) / ((ssb || am) ? 2 : 1);
        h->filter_width = fw;
        if (nbfm) h->qd_gain = static_cast<float>(h->tsr / (4 * kPi * fw));
        if (wbfm) h->qd_gain = static_cast<float>(h->tsr / (2 * kPi * fw));
        h->nbp.qd_gain = h->qd_gain;
        if (ssb) {          // the audio band-pass follows the filter width (gain 2 here, 1 in the constructor: the reference's)
            std::vector<float> a = band_pass_2(2, h->tsr, 200, fw, 200, 90, WIN_BLACKMAN_HARRIS);
            if (static_cast<int>(a.size()) != h->ssbp.nt_audio) { set_err(h, "set_filter_width: audio filter length changed"); return QRL_EINVAL; }
            if ((rc = upload(h->d_audio_taps, a))) return rc;
        }
        return QRL_OK;
    }
    set_err(h, "qrl_rx_set_param: key " + std::to_string(key) + " not supported for this block");
    return QRL_EINVAL;
}

static int rx_work_impl(qrl_rx* h, const void* iq_any, long T, long stride, int on_device, int sc16, float sc16_scale);

int qrl_rx_work(qrl_rx* h, const float* iq, long T, long stride, int on_device)
{
    return rx_work_impl(h, iq, T, stride, on_device, 0, 0.0f);
}
int qrl_rx_work_sc16(qrl_rx* h, const short* iq, long T, long stride, float scale, int on_device)
{
    return rx_work_impl(h, iq, T, stride, on_device, 2, scale);
}
int qrl_rx_work_sc8(qrl_rx* h, const signed char* iq, long T, long stride, float scale, int on_device)
{
    return rx_work_impl(h, iq, T, stride, on_device, 1, scale);
}

// sc16: 0 = gr_complex input, 2 = int16 pairs, 1 = int8 pairs (bytes per component)
static int rx_work_impl(qrl_rx* h, const void* iq_any, long T, long stride, int on_device, int sc16, float sc16_scale)
{
    const float* iq = static_cast<const float*>(iq_any);
    if (!h || !iq || T < 0) return QRL_EINVAL;
    if (T > h->Tmax) { set_err(h, "qrl_rx_work: T exceeds max_samples given at create"); return QRL_ERANGE; }
    if (T == 0) return QRL_OK;
    CK(cudaSetDevice(h->device));
    if (on_device) { int rc = check_device_ptr(h, iq, "qrl_rx_work"); if (rc) return rc; }
    const float2* x = reinterpret_cast<const float2*>(iq);
    long long xstride = stride;
    if (!on_device || sc16) {
        if (!h->d_in_staging) {
            int rc = dev_alloc(h, &h->d_in_staging, static_cast<size_t>(h->Tmax) * h->C, false);
            if (rc) return rc;
        }
    }
    if (sc16) {
        // the SDR's wire format (interleaved int16 I/Q, 4 B per sample: half the PCIe bytes of gr_complex); converted on the device
        // exactly like the host converter in front of the reference's source block: float(v) * scale, one rounding
        const short2* s = static_cast<const short2*>(iq_any);
        long long sstride = stride;
        const size_t isz = sc16 == 2 ? sizeof(short2) : sizeof(char2);
        if (!on_device) {
            if (!h->d_in_sc16) {
                int rc = dev_alloc(h, &h->d_in_sc16, static_cast<size_t>(h->Tmax) * h->C, false);
                if (rc) return rc;
            }
            CK(cudaMemcpy2DAsync(h->d_in_sc16, isz * h->Tmax, iq_any, isz * stride, isz * T, h->C, cudaMemcpyHostToDevice, h->stream));
            s = h->d_in_sc16; sstride = h->Tmax;
        }
        dim3 g(static_cast<unsigned>(std::min<long long>((T + 1023) / 1024, 65535)), h->C);
        if (sc16 == 2) sc16_to_fc32_kernel<<<g, 256, 0, h->stream>>>(s, sstride, h->d_in_staging, h->Tmax, T, sc16_scale);
        else sc8_to_fc32_kernel<<<g, 256, 0, h->stream>>>(reinterpret_cast<const char2*>(s), sstride, h->d_in_staging, h->Tmax, T, sc16_scale);
        h->launches++;
        x = h->d_in_staging;
        xstride = h->Tmax;
    } else if (!on_device) {
        CK(cudaMemcpy2DAsync(h->d_in_staging, sizeof(float2) * h->Tmax, iq, sizeof(float2) * stride,
                             sizeof(float2) * T, h->C, cudaMemcpyHostToDevice, h->stream));
        x = h->d_in_staging;
        xstride = h->Tmax;
    }
    // carrier offset: the register-tiled /50, /100, /25, /125 stage-1 instances rotate their window in shared memory (no extra pass over
    // HBM); the other stage-1 shapes take the rotator as a separate pass
    const bool poly_shape = h->L1 == 1 && ((h->D1 == 50 && h->Q1 == 9) || (h->D1 == 100 && (h->Q1 == 9 || h->Q1 == 28)) ||
                                           (h->D1 == 25 && (h->Q1 == 9 || h->Q1 == 28)) || (h->D1 == 125 && h->Q1 == 9));
    h->rot_fused = h->rot_active && poly_shape && !getenv("QRL_ROTATOR_PASS");
    if (h->rot_active && !h->rot_fused) {
        if (!h->d_rot_buf) { int rc = dev_alloc(h, &h->d_rot_buf, static_cast<size_t>(h->Tmax) * h->C, false); if (rc) return rc; }
        dim3 g(static_cast<unsigned>(std::min<long long>((T + 255) / 256, 4096)), h->C);
        rotator_kernel<<<g, 256, 0, h->stream>>>(h->d_rot, x, xstride, h->d_rot_buf, h->Tmax, T, h->n_in);
        h->launches++;
        x = h->d_rot_buf; xstride = h->Tmax;
    }
    if (h->overlap) {
        // this call writes the buffers call k-2 used: wait for that call's tail, then they are free
        h->call_parity ^= 1;
        for (int j = 0; j < 3; j++) CK(cudaStreamWaitEvent(h->stream, h->ev_tail[h->call_parity][j], 0));
        // The per-slice fences below (ev_v[i], ev_c[q]) pair slice i of this call with slice i of the previous one: that only
        // holds while both calls are cut the same way.  A call of a different length moves the slice boundaries, the symbol-sync
        // scratch regions and the number of slices, so it joins the previous call's tail first (no overlap across that one seam).
        if (h->prev_T != T && h->prev_T >= 0)
            for (int j = 0; j < 3; j++) CK(cudaStreamWaitEvent(h->stream, h->ev_tail[h->call_parity ^ 1][j], 0));
        std::swap(h->d_port0, h->alt_port0); std::swap(h->d_port1, h->alt_port1); std::swap(h->d_port2, h->alt_port2);
        std::swap(h->d_port1_cnt, h->alt_port1_cnt); std::swap(h->d_port2_cnt, h->alt_port2_cnt);
        if (h->d_port3) { std::swap(h->d_port3, h->alt_port3); std::swap(h->d_port3_cnt, h->alt_port3_cnt); }
        h->d_port1f = reinterpret_cast<float*>(h->d_port1);
    }
    CK(cudaMemsetAsync(h->d_port1_cnt, 0, sizeof(int) * h->C, h->stream));
    CK(cudaMemsetAsync(h->d_port2_cnt, 0, sizeof(int) * h->C, h->stream));
    if (h->d_port3_cnt) CK(cudaMemsetAsync(h->d_port3_cnt, 0, sizeof(int) * h->C, h->stream));

    // The call is cut into nsub time slices.  Per slice the parallel stages (decimating FIR, channel filter,
    // demod + RRC) run on the caller's stream; the sequential loop stage of slice i runs on s_loop and the
    // FEC stage on s_fec, overlapping the parallel stages of slices i+1.. (channels stay independent).
    CK(cudaEventRecord(h->ev_start, h->stream));
    CK(cudaStreamWaitEvent(h->s_loop, h->ev_start, 0));
    CK(cudaStreamWaitEvent(h->s_loop2, h->ev_start, 0));
    CK(cudaStreamWaitEvent(h->s_fec, h->ev_start, 0));
    if (h->s_par) CK(cudaStreamWaitEvent(h->s_par, h->ev_start, 0));
    cudaStream_t sp = h->par();
    // overlapped calls keep the pipeline full across calls: two big slices are enough and cost least (a symbol-sync launch has
    // ~20 us of start-up: measured 0.941 ms per 64 x 2^22 call with 2 slices, 0.963 with 3, 0.988 with 4, 1.45 with 1)
    int nsub = (h->overlap && !h->nsub_forced) ? 2 : h->nsub;
    if (T < 32768L * nsub) nsub = static_cast<int>(std::max<long>(1, T / 32768));
    const long long k_call0 = h->n1;
    h->port0_n = 0;
    for (int i = 0; i < nsub; i++) {
        // slice boundaries on multiples of 2*D: the slice base stays 16-byte aligned (TMA bulk fill) and every slice
        // produces the same number of stage-1 outputs
        const long long q2d = 2LL * h->D1;
        auto cut = [&](int j) { return j >= nsub ? static_cast<long long>(T) : (static_cast<long long>(T) * j / nsub) / q2d * q2d; };
        const long long t0 = cut(i), t1 = cut(i + 1);
        if (t1 <= t0) continue;
        const long long Ti = t1 - t0;
        cudaEvent_t pe = nullptr;
        // ---- stage 1: decimating FIR, one launch per group of slices (outputs k with D k <= last absolute input index)
        // stage-1 launch schedule: slice 0 alone (the loop stage starts as early as possible), then fir_group slices
        // per launch (bigger launches run closer to the HBM roofline)
        // (overlapped calls: the pipeline is already full, one launch for the whole call)
        const bool fir_here = h->overlap && !h->fir_group_forced ? (i == 0) : ((i == 0) || ((i - 1) % h->fir_group == 0));
        if (fir_here) {
            const long long tg1 = cut(h->overlap && !h->fir_group_forced ? nsub : (i == 0 ? 1 : std::min(i + h->fir_group, nsub)));
            const long long Tg = tg1 - t0;
            const float2* xg = x + t0;
            const long long Ng = h->n_in + Tg;
            const long long kg0 = h->n1;
            const long long kg1 = (Ng * h->L1 + h->D1 - 1) / h->D1;       // outputs i with floor(i M / L) <= N - 1
            pe = h->prof_begin(0, sp);
            int rc = stage1(h, xg, xstride, Tg, kg0, kg1);
            if (!rc && h->kind == QRL_DEMOD_SSB && kg1 > kg0) {
                // gr_demod_ssb's multiply_const_cc(_if_gain) sits between the resampler and the side-band filter: the gain is applied
                // to the samples as they pass (8 ksps), so after set_gain the filter's history keeps the old gain, like the reference's
                dim3 gs(static_cast<unsigned>((kg1 - kg0 + 255) / 256), h->C);
                scale2_ring_kernel<<<gs, 256, 0, sp>>>(static_cast<float2*>(h->r1.d), h->r1.mask, h->r1.stride, kg0, kg1, h->if_gain, 1.0f);
                h->launches++;
            }
            h->prof_end(pe);
            if (rc) return rc;
            dim3 g((h->H + 127) / 128, h->C);
            if (h->rot_fused) frontend_hist_kernel<<<g, 128, 0, sp>>>(h->d_rot, xg, xstride, Tg, h->n_in, h->d_hist[h->hist_cur], h->d_hist[h->hist_cur ^ 1], h->H);
            else hist_update_kernel<<<g, 128, 0, sp>>>(xg, xstride, Tg, h->d_hist[h->hist_cur], h->d_hist[h->hist_cur ^ 1], h->H);
            h->launches++;
            h->hist_cur ^= 1;
            h->n_in = Ng; h->n1 = kg1;
        }
        // ---- the stages behind it advance slice by slice
        const long long N = h->n_in_s + Ti;
        const long long k0 = h->n1_s;
        const long long k1 = (N * h->L1 + h->D1 - 1) / h->D1;
        h->n_in_s = N; h->n1_s = k1;
        h->cur_k1[i] = k1;
        const long long n_new = k1 - k0;
        h->port0_n += static_cast<long>(n_new);
        long long* nsoft_i = h->d_nsoft + static_cast<size_t>(i) * h->C;
        const int TB = 256;
        dim3 gtile(static_cast<unsigned>((std::max<long long>(n_new, 1) + TB - 1) / TB), h->C);
        const int groups = (h->C + 31) / 32;
        if (h->kind == QRL_DEMOD_DSSS) {
            CK(cudaEventRecord(h->ev_a[i], sp));
            CK(cudaStreamWaitEvent(h->s_loop, h->ev_a[i], 0));
            pe = h->prof_begin(3, h->s_loop);
            dsss_chain_kernel<<<h->C, 256, 0, h->s_loop>>>(h->dsp, h->d_ds, static_cast<const float2*>(h->r1.d), h->r1.mask, h->r1.stride, k1,
                h->d_ds_arms, h->d_taps2, h->d_ds_taps,
                static_cast<float2*>(h->ds_a.d), static_cast<float2*>(h->ds_c.d), h->ds_a.mask, h->ds_a.stride,
                static_cast<float2*>(h->ds_d.d), h->ds_d.mask, h->ds_d.stride,
                h->d_port0, h->port0_cap, h->ds_o_call0,
                h->d_port1, h->port1_cap, h->d_port1_cnt, static_cast<int>(h->port1_cap),
                static_cast<unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride, nsoft_i);
            h->launches++;
            h->prof_end(pe);
            CK(cudaEventRecord(h->ev_b[i], h->s_loop));
            CK(cudaStreamWaitEvent(h->s_fec, h->ev_b[i], 0));
            pe = h->prof_begin(4, h->s_fec);
            constexpr int CPB2 = 4;
            viterbi_k7_kernel<CPB2><<<(h->C + CPB2 - 1) / CPB2, 64 * CPB2, 0, h->s_fec>>>(h->d_vs, nsoft_i, h->C,
                static_cast<const unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride,
                h->d_port2, h->port2_cap, h->d_port2_cnt, static_cast<int>(h->port2_cap), 0);
            viterbi_k7_kernel<CPB2><<<(h->C + CPB2 - 1) / CPB2, 64 * CPB2, 0, h->s_fec>>>(h->d_vs2, nsoft_i, h->C,
                static_cast<const unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride,
                h->d_port3, h->port2_cap, h->d_port3_cnt, static_cast<int>(h->port2_cap), 1);
            h->launches += 2;
            h->prof_end(pe);
            continue;
        }
        if (h->kind == QRL_DEMOD_SSB) {
            if (n_new > 0) {
                pe = h->prof_begin(1, sp);
                fir_ccc_ring_kernel<<<gtile, TB, sizeof(float) * 2 * h->ntaps2, sp>>>(
                    static_cast<const float2*>(h->r1.d), h->r1.mask, h->r1.stride,
                    static_cast<float2*>(h->r2.d), h->r2.mask, h->r2.stride,
                    h->d_taps2, h->ntaps2, 1.0f, k0, k1, h->d_port0, h->port0_cap, k_call0);
                h->launches++;
                h->prof_end(pe);
            }
            CK(cudaEventRecord(h->ev_a[i], sp));
            CK(cudaStreamWaitEvent(h->s_loop, h->ev_a[i], 0));
            pe = h->prof_begin(3, h->s_loop);
            ssb_audio_kernel<<<h->C, 128, 0, h->s_loop>>>(h->ssbp, h->d_ssb,
                static_cast<const float2*>(h->r2.d), h->r2.mask, h->r2.stride, k1,
                static_cast<float2*>(h->rclip.d), h->rclip.mask, h->rclip.stride,
                static_cast<float*>(h->rstr.d), h->rstr.mask, h->rstr.stride,
                h->d_audio_taps, h->d_port1f, 2 * h->port1_cap, h->d_port1_cnt, static_cast<int>(2 * h->port1_cap));
            h->launches++;
            h->prof_end(pe);
            continue;
        }
        if (h->kind == QRL_DEMOD_AM) {
            if (n_new > 0) {
                pe = h->prof_begin(1, sp);
                fir_ccc_ring_kernel<<<gtile, TB, sizeof(float) * 2 * h->ntaps2, sp>>>(
                    static_cast<const float2*>(h->r1.d), h->r1.mask, h->r1.stride,
                    static_cast<float2*>(h->r2.d), h->r2.mask, h->r2.stride,
                    h->d_taps2, h->ntaps2, 1.0f, k0, k1, h->d_port0, h->port0_cap, k_call0);
                h->launches++;
                h->prof_end(pe);
            }
            CK(cudaEventRecord(h->ev_a[i], sp));
            CK(cudaStreamWaitEvent(h->s_loop, h->ev_a[i], 0));
            pe = h->prof_begin(3, h->s_loop);
            nbfm_audio_kernel<<<h->C, 128, 0, h->s_loop>>>(h->nbp, h->d_nb,
                static_cast<const float2*>(h->r2.d), h->r2.mask, h->r2.stride, k1, h->d_env,
                static_cast<float2*>(h->rg.d), h->rg.mask, h->rg.stride,
                static_cast<float*>(h->rd.d), h->rd.mask, h->rd.stride,
                static_cast<float*>(h->rr.d), h->rr.mask, h->rr.stride,
                h->d_arm_taps, h->d_audio_taps, h->d_port1f, 2 * h->port1_cap, h->d_port1_cnt, static_cast<int>(2 * h->port1_cap));
            h->launches++;
            h->prof_end(pe);
            continue;
        }
        if (h->kind == QRL_DEMOD_NBFM || h->kind == QRL_DEMOD_WBFM) {
            if (n_new > 0) {
                pe = h->prof_begin(1, sp);
                { int rc = launch_fir_ccf(h, sp, static_cast<const float2*>(h->r1.d), h->r1.mask, h->r1.stride,
                                          static_cast<float2*>(h->r2.d), h->r2.mask, h->r2.stride,
                                          h->d_taps2, h->ntaps2, k0, k1, h->d_port0, h->port0_cap, k_call0, 0); if (rc) return rc; }
                h->prof_end(pe);
            }
            CK(cudaEventRecord(h->ev_a[i], sp));
            CK(cudaStreamWaitEvent(h->s_loop, h->ev_a[i], 0));
            pe = h->prof_begin(3, h->s_loop);
            const size_t fat = h->nbfm_split ? 120 * 1024 : 0;       // one CTA per SM, and never next to a de-emphasis CTA
            if (h->nbfm_split) {
                static bool f_attr[16] = { false };
                if (!f_attr[h->device & 15]) {
                    CK(cudaFuncSetAttribute(nbfm_audio_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 120 * 1024));
                    CK(cudaFuncSetAttribute(nbfm_deemph_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 120 * 1024));
                    f_attr[h->device & 15] = true;
                }
            }
            nbfm_audio_kernel<<<h->C, 128, fat, h->s_loop>>>(h->nbp, h->d_nb,
                static_cast<const float2*>(h->r2.d), h->r2.mask, h->r2.stride, k1, h->d_env,
                static_cast<float2*>(h->rg.d), h->rg.mask, h->rg.stride,
                static_cast<float*>(h->rd.d), h->rd.mask, h->rd.stride,
                static_cast<float*>(h->rr.d), h->rr.mask, h->rr.stride,
                h->d_arm_taps, h->d_audio_taps, h->d_port1f, 2 * h->port1_cap, h->d_port1_cnt, static_cast<int>(2 * h->port1_cap),
                h->nbfm_split ? static_cast<float*>(h->raud.d) : nullptr, h->raud.mask, h->raud.stride, h->nbfm_split ? nsoft_i : nullptr,
                static_cast<float*>(h->rq.d), h->rq.mask, h->rq.stride, h->ctc, h->d_cenv);
            h->launches++;
            h->prof_end(pe);
            if (h->nbfm_split) {
                CK(cudaEventRecord(h->ev_b[i], h->s_loop));
                CK(cudaStreamWaitEvent(h->s_loop2, h->ev_b[i], 0));
                pe = h->prof_begin(5, h->s_loop2);
                nbfm_deemph_kernel<<<h->C, 128, fat, h->s_loop2>>>(h->nbp.b0, h->nbp.b1, h->nbp.a1, h->nbp.out_gain, h->d_nb2,
                    static_cast<const float*>(h->raud.d), h->raud.mask, h->raud.stride, nsoft_i,
                    h->d_port1f, 2 * h->port1_cap, h->d_port1_cnt, static_cast<int>(2 * h->port1_cap));
                h->launches++;
                h->prof_end(pe);
            }
            continue;
        }
        if (h->kind == QRL_DEMOD_2FSK || h->kind == QRL_DEMOD_BPSK) {
            const bool bpsk = h->kind == QRL_DEMOD_BPSK;
            // ---- FLL (sequential, per sample) on the loop stream: r1 -> rf
            CK(cudaEventRecord(h->ev_a[i], sp));
            CK(cudaStreamWaitEvent(h->s_loop, h->ev_a[i], 0));
            pe = h->prof_begin(1, h->s_loop);
            if (!h->gmsk) {
                fll_kernel<32><<<groups, 32, 0, h->s_loop>>>(h->fllp, h->d_fll, h->d_fll_hist, h->C, h->d_fll_taps,
                    static_cast<const float2*>(h->r1.d), h->r1.mask, h->r1.stride, k1,
                    static_cast<float2*>(h->rf.d), h->rf.mask, h->rf.stride);
                h->launches++;
            }
            h->prof_end(pe);
            const Ring& fin = h->gmsk ? h->r1 : h->rf;             // GMSK: no FLL in front of the channel filter
            if (n_new > 0) {
                // ---- channel filter / RRC on the FLL output -> port 0 (+ ring: channel-major for 2FSK, interleaved for BPSK)
                pe = h->prof_begin(2, h->s_loop);
                { int rc = launch_fir_ccf(h, h->s_loop, static_cast<const float2*>(fin.d), fin.mask, fin.stride,
                                          static_cast<float2*>(h->r2.d), h->r2.mask, h->r2.stride,
                                          h->d_taps2, h->ntaps2, k0, k1, h->d_port0, h->port0_cap, k_call0, bpsk ? 1 : 0); if (rc) return rc; }
                if (!bpsk && h->flag) {
                    { int rc = launch_qdemod_fir(h, h->s_loop, static_cast<const float2*>(h->r2.d), h->r2.mask, h->r2.stride,
                                                 static_cast<float*>(h->r4.d), h->r4.mask, h->r4.stride,
                                                 h->d_taps3, h->ntaps3, h->qd_gain, k0, k1); if (rc) return rc; }
                } else if (!bpsk) {
                    fsk_bank_kernel<2><<<gtile, TB, sizeof(float) * 4 * h->nt_bank, h->s_loop>>>(
                        static_cast<const float2*>(h->r2.d), h->r2.mask, h->r2.stride, h->d_bank_taps, h->nt_bank, k0, k1,
                        static_cast<float*>(h->rbank.d), h->rbank.mask, h->rbank.stride);
                    fir_fff_ring_kernel<<<gtile, TB, sizeof(float) * h->nt_symf, h->s_loop>>>(
                        static_cast<const float*>(h->rbank.d), h->rbank.mask, h->rbank.stride,
                        static_cast<float*>(h->r4.d), h->r4.mask, h->r4.stride, h->d_symf_taps, h->nt_symf, k0, k1);
                    h->launches += 2;
                }
                h->prof_end(pe);
            }
            pe = h->prof_begin(3, h->s_loop);
            if (bpsk) {
                {   // agc2_cc (Costas bypassed): r2 -> r3
                    constexpr int CH = 128, NST = 2;
                    const size_t smem = sizeof(float2) * (NST * CH + AC_NHB * (CH + 1)) * 32;      // every hand-off block + its padding row
                    auto kern = agc_costas_kernel<CH, NST, 0, 0>;
                    static bool a_attr[16] = { false };    // per device: function attributes belong to the device's context
                    if (!a_attr[h->device & 15]) { CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); a_attr[h->device & 15] = true; }
                    kern<<<groups, 96, smem, h->s_loop>>>(h->acp, h->d_ac, h->C,
                        static_cast<const float2*>(h->r2.d), h->r2.mask, h->r2.stride, k1,
                        static_cast<float2*>(h->r3.d), h->r3.mask, h->r3.stride);
                    h->launches++;
                }
                constexpr int CH = 128, NST = 3, NEPI = 1;
                const int maxs = static_cast<int>((CH + 1) / (h->ssp.min_period) + 3);
                const size_t smem = sizeof(float) * (NST * CH * 64 + SYMSYNC_TAB_FLOATS + 2 * maxs * 64) + sizeof(int) * 64;
                auto kern = symsync_kernel<2, SL_BPSK, EPI_BPSK, CH, NST, NEPI, LOOP_CRMM>;
                static bool b_attr[16] = { false };    // per device: function attributes belong to the device's context
                if (!b_attr[h->device & 15]) { CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); b_attr[h->device & 15] = true; }
                kern<<<groups, 64 + 32 * NEPI, smem, h->s_loop>>>(
                    h->ssp, h->d_ss, h->C, static_cast<const float*>(h->r3.d), h->r3.mask, h->r3.stride, k1,
                    h->d_port1, h->port1_cap, h->d_port1_cnt, static_cast<int>(h->port1_cap),
                    static_cast<unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride, maxs, nsoft_i, nullptr, 0, 0, nullptr);
                h->launches++;
            } else {
                constexpr int CH = 256, NST = 3, NEPI = 2;
                const int maxs = static_cast<int>((CH + 1) / (h->ssp.min_period - fabsf(h->ssp.alpha)) + 3);
                const size_t smem = sizeof(float) * (NST * CH * 32 + SYMSYNC_TAB_FLOATS + 2 * maxs * 32) + sizeof(int) * 64;
                auto kern = symsync_kernel<1, SL_BPSK, EPI_REAL1, CH, NST, NEPI>;
                static bool f_attr[16] = { false };    // per device: function attributes belong to the device's context
                if (!f_attr[h->device & 15]) { CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); f_attr[h->device & 15] = true; }
                kern<<<groups, 64 + 32 * NEPI, smem, h->s_loop>>>(
                    h->ssp, h->d_ss, h->C, static_cast<const float*>(h->r4.d), h->r4.mask, h->r4.stride, k1,
                    h->d_port1, h->port1_cap, h->d_port1_cnt, static_cast<int>(h->port1_cap),
                    static_cast<unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride, maxs, nsoft_i, nullptr, 0, 0, nullptr);
                h->launches++;
            }
            h->prof_end(pe);
            CK(cudaEventRecord(h->ev_b[i], h->s_loop));
            // ---- two decoders on the same soft stream, the second behind delay(1)
            CK(cudaStreamWaitEvent(h->s_fec, h->ev_b[i], 0));
            pe = h->prof_begin(4, h->s_fec);
            constexpr int CPB2 = 4;
            viterbi_k7_kernel<CPB2><<<(h->C + CPB2 - 1) / CPB2, 64 * CPB2, 0, h->s_fec>>>(h->d_vs, nsoft_i, h->C,
                static_cast<const unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride,
                h->d_port2, h->port2_cap, h->d_port2_cnt, static_cast<int>(h->port2_cap), 0);
            viterbi_k7_kernel<CPB2><<<(h->C + CPB2 - 1) / CPB2, 64 * CPB2, 0, h->s_fec>>>(h->d_vs2, nsoft_i, h->C,
                static_cast<const unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride,
                h->d_port3, h->port2_cap, h->d_port3_cnt, static_cast<int>(h->port2_cap), 1);
            h->launches += 2;
            h->prof_end(pe);
            continue;
        }
        if (h->kind == QRL_DEMOD_4FSK) {
            if (n_new > 0) {
                // ---- stage 2: channel filter -> ring + port 0
                pe = h->prof_begin(1, sp);
                { int rc = launch_fir_ccf(h, sp, static_cast<const float2*>(h->r1.d), h->r1.mask, h->r1.stride,
                                          static_cast<float2*>(h->r2.d), h->r2.mask, h->r2.stride,
                                          h->d_taps2, h->ntaps2, k0, k1, h->d_port0, h->port0_cap, k_call0, 0); if (rc) return rc; }
                h->prof_end(pe);
                // ---- stage 3: quadrature demod + RRC   |   band-pass bank + discriminator + symbol filter
                // overlapped calls: this slice overwrites ring slots the previous call's symbol sync (slices i, i+1) read
                if (h->overlap && h->prev_nsub > 0) {
                    // the slots [k0, k1) overwrite the samples cap older; the previous call's symbol sync of slice q has
                    // consumed everything up to prev_k1[q] - lookahead
                    const long long must = k1 - (static_cast<long long>(h->r4.mask) + 1) + 64;
                    int q = -1;
                    for (int j = 0; j < h->prev_nsub; j++) if (h->prev_k1[j] - 64 < must) q = j;      // not yet safe after slice j alone
                    if (q >= 0) CK(cudaStreamWaitEvent(sp, h->ev_c[std::min(q + 1, h->prev_nsub - 1)], 0));
                }
                pe = h->prof_begin(2, sp);
                if (h->flag) {
                    { int rc = launch_qdemod_fir(h, sp, static_cast<const float2*>(h->r2.d), h->r2.mask, h->r2.stride,
                                                 static_cast<float*>(h->r4.d), h->r4.mask, h->r4.stride,
                                                 h->d_taps3, h->ntaps3, h->qd_gain, k0, k1); if (rc) return rc; }
                    if (h->dmr) {      // gr_demod_dmr.cpp:103: the symbol filter output is port 3
                        ring_to_port_f32_kernel<<<dim3(static_cast<unsigned>((k1 - k0 + 31) / 32), groups), dim3(32, 8), 0, sp>>>(
                            static_cast<const float*>(h->r4.d), h->r4.mask, h->r4.stride, h->C, k0, k1,
                            h->d_port3f, h->port0_cap, k0 - k_call0);
                        h->launches++;
                    }
                } else {
                    fsk_bank_kernel<4><<<gtile, TB, sizeof(float) * 8 * h->nt_bank, sp>>>(
                        static_cast<const float2*>(h->r2.d), h->r2.mask, h->r2.stride, h->d_bank_taps, h->nt_bank, k0, k1,
                        static_cast<float*>(h->rbank.d), h->rbank.mask, h->rbank.stride);
                    h->launches++;
                    { int rc = launch_fir_ccf(h, sp, static_cast<const float2*>(h->rbank.d), h->rbank.mask, h->rbank.stride,
                                              static_cast<float2*>(h->r3.d), h->r3.mask, h->r3.stride,
                                              h->d_symf_taps, h->nt_symf, k0, k1, nullptr, 0, 0, 1); if (rc) return rc; }
                }
                h->prof_end(pe);
            }
            CK(cudaEventRecord(h->ev_a[i], sp));
            // ---- stage 4: symbol sync (+ phase mod + soft bits) on the loop stream
            CK(cudaStreamWaitEvent(h->s_loop, h->ev_a[i], 0));
            bool ext_recorded = false;
            if (!h->flag) {
                pe = h->prof_begin(3, h->s_loop);
                constexpr int CH = 128, NST = 3, NEPI = 2;
                const int maxs = static_cast<int>((CH + 1) / (h->ssp.min_period - fabsf(h->ssp.alpha)) + 3);
                const size_t smem = sizeof(float) * (NST * CH * 64 + SYMSYNC_TAB_FLOATS + 2 * maxs * 64) + sizeof(int) * 64;
                auto kern = symsync_kernel<2, SL_RECT4, EPI_CPLX, CH, NST, NEPI>;
                static bool sc_attr[16] = { false };    // per device: function attributes belong to the device's context
                if (!sc_attr[h->device & 15]) { CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); sc_attr[h->device & 15] = true; }
                kern<<<groups, 64 + 32 * NEPI, smem, h->s_loop>>>(
                    h->ssp, h->d_ss, h->C, static_cast<const float*>(h->r3.d), h->r3.mask, h->r3.stride, k1,
                    h->d_port1, h->port1_cap, h->d_port1_cnt, static_cast<int>(h->port1_cap),
                    static_cast<unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride, maxs, nsoft_i, nullptr, 0, 0, nullptr);
                h->launches++;
                h->prof_end(pe);
            } else {
                pe = h->prof_begin(3, h->s_loop);
                // real symbols: lean recurrence + external epilogue (symbols leave the SM by TMA bulk store; the phase
                // modulator / soft-bit stores run on the wide partition behind it, same stream)
                auto run_ext = [&](auto ch_tag, auto nst_tag) -> int {
                constexpr int CH = decltype(ch_tag)::value, NST = decltype(nst_tag)::value;
                const int maxs = static_cast<int>((CH + 1) / (h->ssp.min_period - fabsf(h->ssp.alpha)) + 3);
                const size_t smem_base = sizeof(float) * (NST * CH * 32 + SYMSYNC_TAB_FLOATS + 2 * (maxs + 2) * 32) + sizeof(int) * 64;
                const size_t smem_rep = smem_base + 129 * 512;          // + replicated (conflict-free) interpolator bank
                const bool rep = smem_rep <= 220 * 1024 && !h->dmr;
                const size_t smem = rep ? smem_rep : smem_base;
                // gr_demod_dmr: TED_MUELLER_AND_MULLER instead of the modified detector -> generic recurrence, variant 3
                auto kern = h->dmr ? symsync_kernel<1, SL_RECT4, EPI_EXT_4FSK_FM, CH, NST, 1, LOOP_SYMSYNC, 3>
                          : rep ? symsync_kernel<1, SL_RECT4, EPI_EXT_4FSK_FM, CH, NST, 1, LOOP_SYMSYNC, 2>
                                : symsync_kernel<1, SL_RECT4, EPI_EXT_4FSK_FM, CH, NST, 1, LOOP_SYMSYNC, 1>;
                static bool ss_attr[3][16] = { { false } };   // per (CH, NST) instantiation of this lambda, per variant, per device
                const int vi = h->dmr ? 2 : (rep ? 1 : 0);
                if (!ss_attr[vi][h->device & 15]) {
                    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024));
                    ss_attr[vi][h->device & 15] = true;
                }
                // overlapped calls: the previous call's Viterbi of slice i still reads d_nsoft[i], its epilogue scratch region i
                if (h->overlap) CK(cudaStreamWaitEvent(h->s_loop, h->ev_v[i], 0));
                // every slice of a call gets its own scratch region and header (the epilogue of slice i overlaps symsync i+1)
                if (i == 0) h->ss_chunk_off = 0;
                const int chunk_bound = static_cast<int>(std::min<long long>(h->ss_chunk_cap - h->ss_chunk_off, n_new / symsync_stride(CH, h->ssp.lookahead) + 3));
                float* scratch_i = h->d_ss_scratch + static_cast<size_t>(h->ss_chunk_off) * (maxs + 2) * 32;
                int* hdr_i = h->d_ss_hdr + static_cast<size_t>(i) * groups * 128;
                h->ss_chunk_off += chunk_bound;
                kern<<<groups, 96, smem, h->s_loop>>>(
                    h->ssp, h->d_ss, h->C, static_cast<const float*>(h->r4.d), h->r4.mask, h->r4.stride, k1,
                    h->d_port1, h->port1_cap, h->d_port1_cnt, static_cast<int>(h->port1_cap),
                    static_cast<unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride, maxs, nsoft_i,
                    scratch_i, chunk_bound, static_cast<int>(h->ss_chunk_cap), hdr_i);
                h->prof_end(pe);
                cudaStream_t se = h->s_epi ? h->s_epi : h->s_loop;
                if (se != h->s_loop || h->overlap) CK(cudaEventRecord(h->ev_c[i], h->s_loop));
                if (se != h->s_loop) CK(cudaStreamWaitEvent(se, h->ev_c[i], 0));
                pe = h->prof_begin(5, se);
                auto epi = h->dmr ? symsync_ext_epilogue_kernel<1> : symsync_ext_epilogue_kernel<0>;
                if (chunk_bound > 0)
                    epi<<<dim3(chunk_bound, groups), dim3(32, 8), 0, se>>>(
                        h->ssp, h->C, scratch_i, static_cast<int>(h->ss_chunk_cap), maxs, hdr_i,
                        h->d_port1, h->port1_cap, static_cast<int>(h->port1_cap),
                        static_cast<unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride,
                        h->m17 ? h->d_port2 : nullptr, h->port2_cap, static_cast<int>(h->port2_cap), h->d_port2_cnt, h->d_port1_cnt);
                h->launches++;
                h->prof_end(pe);
                CK(cudaEventRecord(h->ev_b[i], se));
                return QRL_OK;
                };
                const int rc_ext = h->ss_ch == 512 ? run_ext(std::integral_constant<int, 512>{}, std::integral_constant<int, 2>{})
                                                   : run_ext(std::integral_constant<int, 256>{}, std::integral_constant<int, 3>{});
                if (rc_ext) return rc_ext;
                ext_recorded = true;
            }
            if (!ext_recorded) CK(cudaEventRecord(h->ev_b[i], h->s_loop));
        } else {   // QRL_DEMOD_QPSK
            const float2* shaping_in = static_cast<const float2*>(h->r1.d);
            unsigned shaping_mask = h->r1.mask; long long shaping_stride = h->r1.stride;
            if (h->d_fll) {     // sps > 4: fll_band_edge_cc between resampler and shaping filter (sequential, on the loop stream)
                CK(cudaEventRecord(h->ev_a[i], sp));
                CK(cudaStreamWaitEvent(h->s_loop, h->ev_a[i], 0));
                fll_kernel<32><<<groups, 32, 0, h->s_loop>>>(h->fllp, h->d_fll, h->d_fll_hist, h->C, h->d_fll_taps,
                    static_cast<const float2*>(h->r1.d), h->r1.mask, h->r1.stride, k1,
                    static_cast<float2*>(h->rf.d), h->rf.mask, h->rf.stride);
                h->launches++;
                CK(cudaEventRecord(h->ev_c[i], h->s_loop));
                CK(cudaStreamWaitEvent(sp, h->ev_c[i], 0));
                shaping_in = static_cast<const float2*>(h->rf.d); shaping_mask = h->rf.mask; shaping_stride = h->rf.stride;
            }
            if (n_new > 0) {
                // ---- stage 2: RRC shaping filter -> interleaved ring + port 0
                pe = h->prof_begin(1, sp);
                { int rc = launch_fir_ccf(h, sp, shaping_in, shaping_mask, shaping_stride,
                                          static_cast<float2*>(h->r2.d), h->r2.mask, h->r2.stride,
                                          h->d_taps2, h->ntaps2, k0, k1, h->d_port0, h->port0_cap, k_call0, 1); if (rc) return rc; }
                h->prof_end(pe);
            }
            CK(cudaEventRecord(h->ev_a[i], sp));
            // ---- stage 3: agc2 + costas "PLL" per sample on the loop stream
            CK(cudaStreamWaitEvent(h->s_loop, h->ev_a[i], 0));
            {
                pe = h->prof_begin(2, h->s_loop);
                auto run_ac = [&](auto ch_tag) -> int {
                    constexpr int CH = decltype(ch_tag)::value, NST = 2;      // input stages (2) + hand-off blocks (3): 164 KB at CH = 128
                    const size_t smem = sizeof(float2) * (NST * CH + AC_NHB * (CH + 1)) * 32;      // every hand-off block + its padding row
                    auto kern = (h->acp.order == 4 && h->acp.use_snr) ? agc_costas_kernel<CH, NST, 4, 1> : agc_costas_kernel<CH, NST>;
                    static bool ac_attr[16] = { false };    // per CH instantiation, per device: function attributes belong to the device's context
                    if (!ac_attr[h->device & 15]) {
                        CK(cudaFuncSetAttribute(agc_costas_kernel<CH, NST, 4, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
                        CK(cudaFuncSetAttribute(agc_costas_kernel<CH, NST>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
                        ac_attr[h->device & 15] = true;
                    }
                    kern<<<groups, 96, smem, h->s_loop>>>(h->acp, h->d_ac, h->C,
                        static_cast<const float2*>(h->r2.d), h->r2.mask, h->r2.stride, k1,
                        static_cast<float2*>(h->r3.d), h->r3.mask, h->r3.stride);
                    return QRL_OK;
                };
                // many channels: 32-row windows (41 KB of shared memory, five CTAs per SM) instead of 128-row ones (164 KB)
                const int rc_ac = h->many ? run_ac(std::integral_constant<int, 32>{}) : run_ac(std::integral_constant<int, 128>{});
                if (rc_ac) return rc_ac;
                h->launches++;
                h->prof_end(pe);
            }
            CK(cudaEventRecord(h->ev_c[i], h->s_loop));
            // ---- stage 4: symbol sync + second Costas + diff phasor + soft bits on the second loop stream
            CK(cudaStreamWaitEvent(h->s_loop2, h->ev_c[i], 0));
            {
                pe = h->prof_begin(3, h->s_loop2);
                // lean: the prefetching complex recurrence (symbol-sync variant 2, replicated tap bank) with the epilogue split into a
                // Costas warp and a feed-forward warp over a 3-deep symbol ring (NEPI = 2); else the generic recurrence, one epilogue warp
                auto run_sq = [&](auto ch_tag, auto nst_tag, auto lean_tag) -> int {
                    constexpr int CH = decltype(ch_tag)::value, NST = decltype(nst_tag)::value;
                    constexpr bool LEAN = decltype(lean_tag)::value;
                    constexpr int NEPI = LEAN ? 2 : 1, NB = LEAN ? 3 : 2;
                    const int maxs = static_cast<int>((CH + 1) / (h->ssp.min_period - fabsf(h->ssp.alpha)) + 3);
                    const size_t smem = sizeof(float) * (NST * CH * 64 + SYMSYNC_TAB_FLOATS + NB * maxs * 64) + sizeof(int) * 32 * (NB == 2 ? 2 : 4) +
                                        (LEAN ? 129 * 512 : 0);
                    auto kern = symsync_kernel<2, SL_DQPSK, EPI_QPSK, CH, NST, NEPI, LOOP_SYMSYNC, LEAN ? 2 : 0>;
                    static bool sq_attr[16] = { false };    // per (CH, NST, LEAN) instantiation, per device
                    if (!sq_attr[h->device & 15]) {
                        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024));
                        sq_attr[h->device & 15] = true;
                    }
                    if (smem > 224 * 1024) { set_err(h, "QPSK symbol sync: window does not fit shared memory"); return QRL_EINVAL; }
                    kern<<<groups, 64 + 32 * NEPI, smem, h->s_loop2>>>(
                        h->ssp, h->d_ss, h->C, static_cast<const float*>(h->r3.d), h->r3.mask, h->r3.stride, k1,
                        h->d_port1, h->port1_cap, h->d_port1_cnt, static_cast<int>(h->port1_cap),
                        static_cast<unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride, maxs, nsoft_i, nullptr, 0, 0, nullptr);
                    return QRL_OK;
                };
                // many channels: 64-row windows, two stages (~55 KB, four CTAs per SM) instead of 128-row ones
                const bool small_win = h->many && symsync_stride(64, h->ssp.lookahead) >= 32;
                static const bool lean_env = [] { const char* e = getenv("QRL_QPSK_LEAN_SS"); return !(e && e[0] == '0'); }();
                // the lean recurrence needs the in-lock window proof (kernel: lean_ok && window_sure) -- true for every QPSK instance of
                // gr_demod_base.cpp; the kernel itself falls back to the generic loop when it does not hold
                const int rc_sq = small_win ? run_sq(std::integral_constant<int, 64>{}, std::integral_constant<int, 2>{}, std::false_type{})
                                : lean_env  ? run_sq(std::integral_constant<int, 128>{}, std::integral_constant<int, 2>{}, std::true_type{})
                                            : run_sq(std::integral_constant<int, 128>{}, std::integral_constant<int, 3>{}, std::false_type{});
                if (rc_sq) return rc_sq;
                h->launches++;
                h->prof_end(pe);
            }
            CK(cudaEventRecord(h->ev_b[i], h->s_loop2));
        }
        // ---- stage 5: Viterbi + descrambler on the FEC stream
        CK(cudaStreamWaitEvent(h->s_fec, h->ev_b[i], 0));
        if (h->m17) {                    // gr_demod_m17 has no FEC: the epilogue wrote the hard bits of port 2 (s_fec joins it at the end)
            if (h->overlap) CK(cudaEventRecord(h->ev_v[i], h->s_fec));
            continue;
        }
        pe = h->prof_begin(4, h->s_fec);
        constexpr int CPB = 4;    // 4 channels (8 warps) per CTA
        viterbi_k7_kernel<CPB><<<(h->C + CPB - 1) / CPB, 64 * CPB, 0, h->s_fec>>>(h->d_vs, nsoft_i, h->C,
            static_cast<const unsigned char*>(h->r5.d), h->r5.mask, h->r5.stride,
            h->d_port2, h->port2_cap, h->d_port2_cnt, static_cast<int>(h->port2_cap), 0);
        h->launches++;
        h->prof_end(pe);
        if (h->overlap) CK(cudaEventRecord(h->ev_v[i], h->s_fec));
    }
    if (h->kind == QRL_DEMOD_DSSS) {          // port 0 holds 5200 sps items (13 / 50 of the stage-1 items counted in the loop)
        const long long o_end = (h->n1_s * 13 + 49) / 50;
        h->port0_n = static_cast<long>(o_end - h->ds_o_call0);
        h->ds_o_call0 = o_end;
    }
    if (h->rssi_on && h->port0_n > 0) {
        // port 0 of this call is complete on the parallel stream: append to the |x|^2 ring, evaluate the latest RSSI value
        rssi_kernel<<<h->C, 256, 0, sp>>>(h->d_port0, h->port0_cap, static_cast<int>(std::min<long>(h->port0_n, h->port0_cap)),
                                          h->rssi_n, h->d_rssi_ring, h->d_rssi_y, h->d_rssi_db);
        h->launches++;
        h->rssi_n += std::min<long>(h->port0_n, h->port0_cap);
    }
    for (int i = 0; i < nsub; i++) h->prev_k1[i] = h->cur_k1[i];
    h->prev_nsub = nsub;
    h->prev_T = T;
    if (h->overlap) {
        // the caller's stream only waits for the parallel stages (the input has been consumed); the loop / FEC tail runs
        // on under the next call and is joined by qrl_rx_join / qrl_rx_sync / qrl_rx_read_port
        CK(cudaEventRecord(h->ev_tail[h->call_parity][0], h->s_loop));
        CK(cudaEventRecord(h->ev_tail[h->call_parity][1], h->s_fec));
        CK(cudaEventRecord(h->ev_tail[h->call_parity][2], h->s_epi ? h->s_epi : h->s_loop));
        if (h->s_par) { CK(cudaEventRecord(h->ev_par_done, h->s_par)); CK(cudaStreamWaitEvent(h->stream, h->ev_par_done, 0)); }
        CK(cudaGetLastError());
        return QRL_OK;
    }
    CK(cudaEventRecord(h->ev_loop_done, h->s_loop));
    CK(cudaEventRecord(h->ev_loop2_done, h->s_loop2));
    CK(cudaStreamWaitEvent(h->stream, h->ev_loop2_done, 0));
    CK(cudaEventRecord(h->ev_fec_done, h->s_fec));
    if (h->s_par) { CK(cudaEventRecord(h->ev_par_done, h->s_par)); CK(cudaStreamWaitEvent(h->stream, h->ev_par_done, 0)); }
    CK(cudaStreamWaitEvent(h->stream, h->ev_loop_done, 0));
    CK(cudaStreamWaitEvent(h->stream, h->ev_fec_done, 0));
    CK(cudaGetLastError());
    return QRL_OK;
}

int qrl_rx_join(qrl_rx* h)
{
    if (!h) return QRL_EINVAL;
    if (!h->overlap) return QRL_OK;
    for (int j = 0; j < 3; j++) CK(cudaStreamWaitEvent(h->stream, h->ev_tail[h->call_parity][j], 0));
    return QRL_OK;
}

int qrl_rx_profile(qrl_rx* h, int enable)
{
    if (!h) return QRL_EINVAL;
    CK(cudaStreamSynchronize(h->stream));
    h->prof = enable != 0;
    h->prof_used = 0;
    for (int i = 0; i < 8; i++) { h->prof_ms[i] = 0; h->prof_n[i] = 0; }
    return QRL_OK;
}

int qrl_rx_profile_read(qrl_rx* h, int stage, double* ms_total, long* n_launches)
{
    if (!h || stage < 0 || stage >= 8) return QRL_EINVAL;
    CK(cudaStreamSynchronize(h->stream));
    if (h->overlap) { int rc = rx_join_host(h); if (rc) return rc; }
    for (size_t i = 0; i < h->prof_used; i++) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, h->prof_recs[i].a, h->prof_recs[i].b) == cudaSuccess) {
            h->prof_ms[h->prof_recs[i].stage] += ms; h->prof_n[h->prof_recs[i].stage]++;
        }
    }
    h->prof_used = 0;
    if (ms_total) *ms_total = h->prof_ms[stage];
    if (n_launches) *n_launches = h->prof_n[stage];
    return QRL_OK;
}

int qrl_rx_sync(qrl_rx* h)
{
    if (!h) return QRL_EINVAL;
    CK(cudaStreamSynchronize(h->stream));
    if (h->overlap) return rx_join_host(h);
    return QRL_OK;
}

int qrl_rx_rssi(qrl_rx* h, float level, float* rssi_db_host)
{
    if (!h || !rssi_db_host) return QRL_EINVAL;
    if (!h->rssi_on || !h->d_rssi_db) { set_err(h, "qrl_rx_rssi: enable QRL_PARAM_RSSI first"); return QRL_EINVAL; }
    CK(cudaStreamSynchronize(h->stream));
    if (h->s_par) CK(cudaStreamSynchronize(h->s_par));
    CK(cudaMemcpy(rssi_db_host, h->d_rssi_db, sizeof(float) * h->C, cudaMemcpyDeviceToHost));
    for (int c = 0; c < h->C; c++) rssi_db_host[c] = (h->rssi_n > 0 ? rssi_db_host[c] : -180.0f) + level;      // add_const_ff(level)
    return QRL_OK;
}

int qrl_rx_num_ports(const qrl_rx* h) { return h ? h->nports : QRL_EINVAL; }
int qrl_rx_port_itemsize(const qrl_rx* h, int port)
{
    if (!h || port < 0 || port >= h->nports) return QRL_EINVAL;
    if (port == 0) return 8;
    if (port == 1) return (h->kind == QRL_DEMOD_NBFM || h->kind == QRL_DEMOD_SSB || h->kind == QRL_DEMOD_AM || h->kind == QRL_DEMOD_WBFM) ? 4 : 8;
    if (port == 3 && h->dmr) return 4;
    return 1;
}

int qrl_rx_port_device(qrl_rx* h, int port, void** data, long* cap, int** counts)
{
    if (!h || port < 0 || port >= h->nports) return QRL_EINVAL;
    if (port == 0) { *data = h->d_port0; *cap = h->port0_cap; *counts = nullptr; }
    else if (port == 1) {
        *data = h->d_port1; *counts = h->d_port1_cnt;
        *cap = (h->kind == QRL_DEMOD_NBFM || h->kind == QRL_DEMOD_SSB || h->kind == QRL_DEMOD_AM || h->kind == QRL_DEMOD_WBFM) ? 2 * h->port1_cap : h->port1_cap;      // float view of the same buffer
    }
    else if (port == 2) { *data = h->d_port2; *cap = h->port2_cap; *counts = h->d_port2_cnt; }
    else if (h->dmr) { *data = h->d_port3f; *cap = h->port0_cap; *counts = nullptr; }      // one float per port-0 sample
    else { *data = h->d_port3; *cap = h->port2_cap; *counts = h->d_port3_cnt; }
    return QRL_OK;
}

int qrl_rx_read_port(qrl_rx* h, int port, void* dst, long cap, int* counts, int dst_on_device)
{
    if (!h || port < 0 || port >= h->nports || !counts) return QRL_EINVAL;
    void* src; long scap; int* dcnt;
    int rc = qrl_rx_port_device(h, port, &src, &scap, &dcnt);
    if (rc) return rc;
    const int isz = qrl_rx_port_itemsize(h, port);
    long maxn = 0;
    if (h->overlap) { CK(cudaStreamSynchronize(h->stream)); rc = rx_join_host(h); if (rc) return rc; }
    if (dcnt) {
        CK(cudaMemcpyAsync(counts, dcnt, sizeof(int) * h->C, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        for (int c = 0; c < h->C; c++) { if (counts[c] > scap) counts[c] = static_cast<int>(scap); maxn = std::max<long>(maxn, counts[c]); }
    } else {
        for (int c = 0; c < h->C; c++) counts[c] = static_cast<int>(h->port0_n);
        maxn = h->port0_n;
    }
    if (dst && maxn > 0) {
        const long w = std::min(maxn, cap);
        CK(cudaMemcpy2DAsync(dst, static_cast<size_t>(cap) * isz, src, static_cast<size_t>(scap) * isz, static_cast<size_t>(w) * isz, h->C,
                             dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return QRL_OK;
}

long qrl_rx_launch_count(const qrl_rx* h) { return h ? h->launches : 0; }
int qrl_rx_sm_partition(const qrl_rx* h, int* loop_sms, int* parallel_sms)
{
    if (!h) return QRL_EINVAL;
    if (loop_sms) *loop_sms = h->sm_loop;
    if (parallel_sms) *parallel_sms = h->sm_par;
    return QRL_OK;
}

// ---------------------------------------------------------------------------------------------- TX
// gr_zero_idle_bursts (gr_zero_idle_bursts.cpp:47-86) as host-side bookkeeping: the "zero_samples" tags waiting per channel and the count
// still running at the end of the last call; a call turns them into {channel, first item, end item} ranges that one kernel clears
// (a tag loads the counter, a later one overrides what is left of it, one output is cleared per count).  Shared by gr_mod_dmr (delay
// 62) and the MMDVM modulators (delay 0).
struct ZeroIdle {
    std::vector<std::map<long long, unsigned long long>> tags;      // per channel: start item -> count (first registered wins)
    std::vector<unsigned long long> counter;                       // per channel: count still running at the end of the last call
    long long* d_ranges = nullptr; size_t ranges_cap = 0;
    void init(int C) { tags.assign(C, {}); counter.assign(C, 0); }
    // tag for item `start` (already corrected for the block's delay); `produced` = items the block has put out so far
    void add(int channel, int C, long long start, unsigned long long val, long long produced)
    {
        if (start < produced) {                                                  // late: clear what is left of the count
            const unsigned long long late = static_cast<unsigned long long>(produced - start);
            if (late >= val) return;
            val -= late; start = produced;
        }
        for (int c = (channel < 0 ? 0 : channel); c < (channel < 0 ? C : channel + 1); c++) tags[c].emplace(start, val);
    }
    // ranges of the items [m0, m1) this call produces, as {c, a0 - base, a1 - base} triples
    void collect(int C, long long m0, long long m1, long long base, std::vector<long long>& ranges)
    {
        for (int c = 0; c < C; c++) {
            auto& tg = tags[c];
            tg.erase(tg.begin(), tg.lower_bound(m0));
            unsigned long long cnt = counter[c];
            if (cnt == 0 && (tg.empty() || tg.begin()->first >= m1)) continue;
            long long cur = m0;
            auto it = tg.begin();
            while (true) {
                const long long next = (it != tg.end() && it->first < m1) ? it->first : m1;
                const long long z_end = cnt >= static_cast<unsigned long long>(next - cur) ? next : cur + static_cast<long long>(cnt);
                if (z_end > cur) { ranges.push_back(c); ranges.push_back(cur - base); ranges.push_back(z_end - base); }
                cnt -= static_cast<unsigned long long>(z_end - cur);
                if (next == m1) break;
                cnt = it->second; cur = next; it = tg.erase(it);
            }
            counter[c] = cnt;
        }
    }
    // upload the triples (growing the device buffer if needed); returns a CUDA error code
    cudaError_t upload(const std::vector<long long>& ranges, cudaStream_t stream)
    {
        if (ranges.size() > ranges_cap) {
            cudaError_t e = cudaStreamSynchronize(stream); if (e != cudaSuccess) return e;
            if (d_ranges) { e = cudaFree(d_ranges); if (e != cudaSuccess) return e; d_ranges = nullptr; }
            ranges_cap = 2 * ranges.size() + 48;
            e = cudaMalloc(&d_ranges, sizeof(long long) * ranges_cap); if (e != cudaSuccess) return e;
        }
        return cudaMemcpyAsync(d_ranges, ranges.data(), sizeof(long long) * ranges.size(), cudaMemcpyHostToDevice, stream);
    }
    void release() { if (d_ranges) cudaFree(d_ranges); d_ranges = nullptr; }
};

struct qrl_tx : HandleBase {
    int kind = 0, sps = 0, samp_rate = 0, filter_width = 0, flag = 0, C = 0;
    long max_items = 0;
    int L1 = 1, nt1 = 0;            // first interpolation (RRC): L1 arms of nt1 taps
    int L2 = 1, nt2 = 0;            // second interpolation (x20 low-pass), 4FSK only
    float* d_arms1 = nullptr; float* d_arms2 = nullptr;
    float fm_sens = 0, amplif = 0, bb_gain = 1.0f, pulse_scale = 0.66666666f;
    int repeat_only = 0;
    bool m17 = false; int M2 = 1;  // gr_mod_m17: 4 symbols per byte, IF low-pass at 24 ksps, x L2 / M2 rational interpolator
    // gr_mod_dsss: chips (complex ring d_sym) -> x25 (ring d_if) -> x50 / 13 (ring d_rc, arms in d_cfilt) -> x50 (d_out)
    bool dsss_tx = false;
    // gr_mod_am: audio ring d_ra -> 8 ksps complex ring d_if -> x sps (ring d_rc at the output rate) -> output filter (taps d_cfilt) -> d_out
    bool am_tx = false; float am_dc = 0.0f;
    // gr_mod_nbfm::set_ctcss: multiply_const_ff gain and the CTCSS tone source (fxpt_nco phase / increment, advanced per sample with the tone on)
    float audio_gain = 0.99f; bool tone_on = false; unsigned tone_phase = 0, tone_inc = 0;
    // gr_mod_dmr: the m17 path with gr_zero_idle_bursts in place of the IF low-pass (a delay of history - 1 items + "zero_samples" tags)
    bool dmr_tx = false; long long zi_delay_items = 0; unsigned zi_tag_delay = 0;
    ZeroIdle zi;                                                      // gr_mod_dmr: gr_zero_idle_bursts(62)
    TxBitState* d_bits = nullptr;
    unsigned char* d_in = nullptr;
    float* d_sym = nullptr; unsigned sym_mask = 0; long long sym_stride = 0;    // float (4FSK) / float2 (QPSK)
    float2* d_if = nullptr; unsigned if_mask = 0; long long if_stride = 0;
    float2* d_out = nullptr; long long out_stride = 0; long n_out_last = 0;
    long long n_sym = 0;           // symbols produced so far (absolute)
    // analog modulators (NBFM / SSB)
    TxAnalogState* d_an = nullptr;
    float* d_ra = nullptr; unsigned ra_mask = 0; long long ra_stride = 0;          // audio ring
    float* d_rb = nullptr;                                                         // filtered audio ring (same geometry)
    float2* d_rc = nullptr; unsigned rc_mask = 0; long long rc_stride = 0;         // SSB clip ring / NBFM IF-filter ring
    float2* d_rs2 = nullptr;                                                       // SSB stretcher ring (same geometry as rc)
    float* d_lpf = nullptr; int nt_lpf = 0; float* d_cfilt = nullptr; int nt_cfilt = 0;
    double pe_b0 = 0, pe_b1 = 0, pe_a1 = 0;
    long long n_audio = 0, n_mid = 0;        // audio samples consumed / mid-rate items produced (host mirror of the device counters)
    float* d_audio_in = nullptr;
    // 4FSK: the three stages (bit chain, pulse shaping + FM scan, x20 interpolator) run slice by slice on three streams
    static constexpr int kTxSub = 8;
    cudaStream_t s_bits = nullptr, s_shape = nullptr;
    cudaEvent_t ev_start = nullptr, ev_bits[kTxSub] = { nullptr }, ev_shape[kTxSub] = { nullptr }, ev_shape_done = nullptr, ev_out_done = nullptr;
    // optional per-stage device timing (qrl_tx_profile): 0 = bit chain, 1 = pulse shaping / FM scan, 2 = final interpolator
    bool prof = false;
    struct ProfRec { int stage; cudaEvent_t a, b; };
    std::vector<ProfRec> prof_recs; size_t prof_used = 0;
    double prof_ms[4] = { 0 }; long prof_n[4] = { 0 };
    cudaStream_t prof_stream = nullptr;
    cudaEvent_t prof_begin(int stage, cudaStream_t on)
    {
        prof_stream = on;
        if (!prof) return nullptr;
        if (prof_used == prof_recs.size()) {
            ProfRec r{ stage, nullptr, nullptr };
            cudaEventCreate(&r.a); cudaEventCreate(&r.b);
            prof_recs.push_back(r);
        }
        ProfRec& r = prof_recs[prof_used];
        r.stage = stage;
        cudaEventRecord(r.a, prof_stream);
        return r.b;
    }
    void prof_end(cudaEvent_t b) { if (b) { cudaEventRecord(b, prof_stream); prof_used++; } }
};

static std::vector<float> make_arms(const std::vector<float>& taps, int L, int nt)
{
    std::vector<float> a(static_cast<size_t>(L) * nt, 0.0f);
    for (int p = 0; p < L; p++)
        for (int k = 0; k < nt; k++) { const size_t j = p + static_cast<size_t>(k) * L; if (j < taps.size()) a[p * nt + k] = taps[j]; }
    return a;
}

int qrl_tx_create(int kind, int sps, int samp_rate, int carrier_freq, int filter_width, int flag,
                  int n_channels, long max_items, int device, qrl_tx** out)
{
    (void)carrier_freq;
    if (!out || n_channels <= 0 || max_items <= 0) { set_err(nullptr, "qrl_tx_create: bad argument"); return QRL_EINVAL; }
    *out = nullptr;
    if (qrl_device_count() <= device) { set_err(nullptr, "qrl_tx_create: no CUDA device (this library has no CPU fallback)"); return QRL_ENODEV; }
    qrl_tx* h = new qrl_tx();
    h->kind = kind; h->sps = sps; h->samp_rate = samp_rate; h->filter_width = filter_width; h->flag = flag;
    h->C = n_channels; h->max_items = max_items; h->device = device;
    auto fail = [&](int rc) { std::string e = h->err; qrl_tx_destroy(h); g_err = e; return rc; };
    if (cudaSetDevice(device) != cudaSuccess) { set_err(h, "cudaSetDevice failed"); return fail(QRL_ECUDA); }
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { set_err(h, "stream create failed"); return fail(QRL_ECUDA); }
    h->own_stream = true;
    int rc = upload_tables(h);
    if (rc) return fail(rc);
    std::vector<float> t1, t2;
    if (kind == QRL_MOD_4FSK) {
        // gr_mod_4fsk.cpp:55-92
        int sym_sps = sps, nfilts = sym_sps * 10, second_interp = 20;
        if (sps == 2) { sym_sps = 5; second_interp = 2; nfilts = 256; }
        int spacing = 2; h->amplif = 0.8f;
        if (flag) { h->amplif = 0.9f; spacing = 1; }
        h->repeat_only = flag ? 0 : 1;
        t1 = root_raised_cosine(sym_sps, sym_sps, 1, 0.2, nfilts);
        h->L1 = sym_sps; h->nt1 = (static_cast<int>(t1.size()) + sym_sps - 1) / sym_sps;
        h->fm_sens = static_cast<float>((spacing * kPi) / sym_sps);
        t2 = low_pass(second_interp, samp_rate, filter_width, filter_width, WIN_HAMMING);
        h->L2 = second_interp; h->nt2 = (static_cast<int>(t2.size()) + second_interp - 1) / second_interp;
        if (h->L2 == 20 && h->nt2 <= 35) h->nt2 = 35;      // register-tiled instance <20, 35>
    } else if (kind == QRL_MOD_QPSK) {
        // gr_mod_qpsk.cpp:58-75
        int nfilts = sps > 120 ? 11 : (sps > 10 ? 13 : 15);
        t1 = root_raised_cosine(sps, sps, 1, 0.35, nfilts * sps);
        h->L1 = sps; h->nt1 = (static_cast<int>(t1.size()) + sps - 1) / sps;
        if (h->L1 == 4 && h->nt1 <= 16) h->nt1 = 16;      // register-tiled instance <4, 16>
        h->amplif = 0.6f;
    } else if (kind == QRL_MOD_NBFM) {
        // gr_mod_nbfm.cpp:35-63 (sps = final interpolation, 20)
        double a[2], b[2];
        preemph_taps(8000, 50e-6, -1.0, a, b);
        h->pe_b0 = b[0]; h->pe_b1 = b[1]; h->pe_a1 = a[1];
        std::vector<float> lp = low_pass_2(1, 8000, 3500, 200, 35, WIN_BLACKMAN_HARRIS);
        h->nt_lpf = static_cast<int>(lp.size());
        if ((rc = upload_floats(h, &h->d_lpf, lp))) return fail(rc);
        t1 = low_pass_2(25, 50000 * 4, filter_width, 3500, 60, WIN_BLACKMAN_HARRIS);          // 25/4 resampler arms
        h->L1 = 25; h->nt1 = (static_cast<int>(t1.size()) + 24) / 25;
        h->fm_sens = static_cast<float>(4 * kPi * filter_width / 50000.0f);
        std::vector<float> ifl = low_pass_2(1, 50000, filter_width, 3500, 60, WIN_BLACKMAN_HARRIS);
        h->nt_cfilt = static_cast<int>(ifl.size());
        if ((rc = upload_floats(h, &h->d_cfilt, ifl))) return fail(rc);
        t2 = low_pass_2(sps, samp_rate, filter_width, 3500, 60, WIN_BLACKMAN_HARRIS);
        h->L2 = sps; h->nt2 = (static_cast<int>(t2.size()) + sps - 1) / sps;
        h->amplif = 0.8f;
    } else if (kind == QRL_MOD_SSB) {
        // gr_mod_ssb.cpp:40-58 (sps = final interpolation, 125; flag = sb)
        std::vector<float> bp = band_pass_2(1, 8000, 300, filter_width, 200, 90, WIN_BLACKMAN_HARRIS);
        h->nt_lpf = static_cast<int>(bp.size());
        if ((rc = upload_floats(h, &h->d_lpf, bp))) return fail(rc);
        std::vector<float> sb = flag ? complex_band_pass_2(1, 8000, -filter_width, -200, 200, 90, WIN_BLACKMAN_HARRIS)
                                     : complex_band_pass_2(1, 8000, 200, filter_width, 200, 90, WIN_BLACKMAN_HARRIS);
        h->nt_cfilt = static_cast<int>(sb.size() / 2);
        if ((rc = upload_floats(h, &h->d_cfilt, sb))) return fail(rc);
        t2 = low_pass_2(sps, samp_rate, filter_width, filter_width, 90, WIN_BLACKMAN_HARRIS);
        h->L2 = sps; h->nt2 = (static_cast<int>(t2.size()) + sps - 1) / sps;
        h->L1 = 1; h->nt1 = 1; t1 = { 1.0f };
        h->amplif = 0.9f;
    } else if (kind == QRL_MOD_BPSK) {
        // gr_mod_bpsk.cpp:44-56
        t1 = root_raised_cosine(sps, sps, 1, 0.35, 11 * sps);
        h->L1 = sps; h->nt1 = (static_cast<int>(t1.size()) + sps - 1) / sps;
        h->amplif = 0.6f;
    } else if (kind == QRL_MOD_AM) {
        // gr_mod_am.cpp:25-72: agc2_ff -> rail -> x0.95 -> band_pass_2(1, 8000, 300, 3000, 200, 60, Hamming) -> + 0.5 cos(0) -> float_to_complex ->
        // rational_resampler_ccf(sps, 1, low_pass(sps, fs, fw, fw)) -> x0.5 -> bb gain -> fft_filter_ccc(complex_band_pass_2(1, fs, -fw, fw, 1200,
        // 120, BH)).  The band is symmetric, so the complex taps are the low-pass prototype times e^{j0}: imaginary parts exactly 0 and the
        // filter is the real-tap ring FIR (same accumulation, see oracle fircc_work with hi = 0).
        h->am_tx = true; h->amplif = 0.5f;
        const std::vector<float> bp = band_pass_2(1, 8000, 300, 3000, 200, 60, WIN_HAMMING);
        h->nt_lpf = static_cast<int>(bp.size());
        if ((rc = upload_floats(h, &h->d_lpf, bp))) return fail(rc);
        t1 = { 1.0f }; h->L1 = 1; h->nt1 = 1;
        t2 = low_pass(sps, samp_rate, filter_width, filter_width, WIN_HAMMING);
        h->L2 = sps; h->nt2 = (static_cast<int>(t2.size()) + sps - 1) / sps;
        const std::vector<float> cb = complex_band_pass_2(1, samp_rate, -filter_width, filter_width, 1200, 120, WIN_BLACKMAN_HARRIS);
        std::vector<float> of(cb.size() / 2);
        for (size_t i = 0; i < of.size(); i++) {
            if (cb[2 * i + 1] != 0.0f) { set_err(h, "make_gr_mod_am: output filter taps are not real"); return fail(QRL_EINVAL); }
            of[i] = cb[2 * i];
        }
        h->nt_cfilt = static_cast<int>(of.size());
        if ((rc = upload_floats(h, &h->d_cfilt, of))) return fail(rc);
        if (static_cast<size_t>(h->L2) * h->nt2 * sizeof(float) > 40 * 1024 || h->nt_cfilt > 8192) { set_err(h, "make_gr_mod_am: unsupported sps / filter_width"); return fail(QRL_EINVAL); }
        { const std::vector<float> st_ = fxpt_sine_table(); const unsigned uc = 0x40000000u; const int ci = uc >> 22;
          const float c0 = st_[2 * ci] * static_cast<float>(uc >> 1) + st_[2 * ci + 1];
          h->am_dc = static_cast<float>(static_cast<double>(c0) * 0.5); }
    } else if (kind == QRL_MOD_DSSS) {
        // gr_mod_dsss.cpp:27-93: scrambler -> cc_encoder -> Barker-13 spreading -> {-1, +1} -> rational_resampler_ccf(sps, 1, RRC(sps, sps, 1,
        // 0.35, 11 sps)) -> x0.65 -> bb gain -> rational_resampler_ccf(50, 13, low_pass(50, 5200 * 50, fw, 5 fw)) ->
        // rational_resampler_ccf(50, 1, low_pass(50, fs, fw, 5 fw)); one input byte = 208 chips = 10^6 output samples (sps = 25)
        h->dsss_tx = true; h->amplif = 0.65f;
        t1 = root_raised_cosine(sps, sps, 1, 0.35, 11 * sps);
        h->L1 = sps; h->nt1 = (static_cast<int>(t1.size()) + sps - 1) / sps;
        const std::vector<float> tif = low_pass(50.0, 5200.0 * 50, filter_width, filter_width * 5, WIN_HAMMING);
        h->nt_cfilt = (static_cast<int>(tif.size()) + 49) / 50;
        if ((rc = upload_floats(h, &h->d_cfilt, make_arms(tif, 50, h->nt_cfilt)))) return fail(rc);
        t2 = low_pass(50, samp_rate, filter_width, filter_width * 5, WIN_HAMMING);
        h->L2 = 50; h->nt2 = (static_cast<int>(t2.size()) + 49) / 50;
        if (static_cast<size_t>(50) * std::max(h->nt2, h->nt_cfilt) * sizeof(float) > 40 * 1024 || static_cast<size_t>(h->L1) * h->nt1 * sizeof(float) > 40 * 1024) {
            set_err(h, "make_gr_mod_dsss: filter_width too small for the shared-memory arm tables"); return fail(QRL_EINVAL);
        }
    } else if (kind == QRL_MOD_GMSK) {
        // gr_mod_gmsk.cpp:30-100: the 2FSK (fm) modulator path with a Gaussian pulse (BT 0.3), sensitivity (pi/2)/sps and a
        // x5 (x1 for the 10k mode) final interpolation; instances gr_mod_base.cpp:160-162
        int nfilts = 35, second_interp = 5;
        if (sps == 10) { sps = 50; second_interp = 1; nfilts = 55; }
        if (sps == 50) nfilts = 55;
        if (sps == 100) nfilts = 35;
        if ((nfilts % 2) == 0) nfilts += 1;
        kind = QRL_MOD_2FSK; h->kind = QRL_MOD_2FSK; h->sps = sps; flag = 1; h->flag = 1;
        h->amplif = 0.9f; h->repeat_only = 0; h->pulse_scale = 1.0f;
        t1 = gaussian(sps, sps, 0.3, nfilts);
        h->L1 = sps; h->nt1 = (static_cast<int>(t1.size()) + sps - 1) / sps;
        h->fm_sens = static_cast<float>((kPi / 2) / sps);
        t2 = low_pass(second_interp, samp_rate, filter_width, filter_width, WIN_HAMMING);
        h->L2 = second_interp; h->nt2 = (static_cast<int>(t2.size()) + second_interp - 1) / second_interp;
    } else if (kind == QRL_MOD_M17) {
        // gr_mod_m17.cpp:30-95: pulse shaping x5 (RRC 0.5, 250 + 1 taps) -> x0.66666666 -> frequency modulator (pi / 5) -> low-pass at
        // 24 ksps -> x0.9 -> bb gain -> rational_resampler_ccf(sps = 125, 3)
        h->m17 = true; h->amplif = 0.9f; h->repeat_only = 0;
        t1 = root_raised_cosine(5, 5, 1, 0.5, 250);
        h->L1 = 5; h->nt1 = (static_cast<int>(t1.size()) + 4) / 5;
        h->fm_sens = static_cast<float>(kPi / 5);
        std::vector<float> ifl = low_pass(1, 24000, filter_width, filter_width, WIN_BLACKMAN_HARRIS);
        h->nt_cfilt = static_cast<int>(ifl.size());
        if ((rc = upload_floats(h, &h->d_cfilt, ifl))) return fail(rc);
        t2 = low_pass(sps, 3.0 * samp_rate, 12000, 12000, WIN_BLACKMAN_HARRIS);
        h->L2 = sps; h->M2 = 3; h->nt2 = (static_cast<int>(t2.size()) + sps - 1) / sps;
        if (sps <= 3 || static_cast<size_t>(h->L2) * h->nt2 * sizeof(float) > 40 * 1024) { set_err(h, "make_gr_mod_m17: unsupported sps"); return fail(QRL_EINVAL); }
    } else if (kind == QRL_MOD_DMR) {
        // gr_mod_dmr.cpp:27-93: pulse shaping x5 (RRC(5, 24000, 4800, 0.2, 125 taps)) -> x0.66666666 -> frequency modulator
        // (pi * 4800 * 0.85 / 24000) -> gr_zero_idle_bursts(62) -> x0.9 -> bb gain -> rational_resampler_ccf(sps, 3, low_pass_2(sps, 3 fs,
        // fw, 2000, 60, BH)); the fft_filter_ccf of :72-73 is never connected
        h->m17 = true; h->dmr_tx = true; h->amplif = 0.9f; h->repeat_only = 0;
        const float if_samp_rate = 24000, symbol_rate = if_samp_rate / 5.0f;
        t1 = root_raised_cosine(5, if_samp_rate, symbol_rate, 0.2, 25 * 5);
        h->L1 = 5; h->nt1 = (static_cast<int>(t1.size()) + 4) / 5;
        h->zi_tag_delay = static_cast<unsigned>((t1.size() - 1) / 2);                        // gr_mod_dmr.cpp:58
        h->zi_delay_items = h->zi_tag_delay > 0 ? 2 * 720 - 1 : 0;                             // gr_zero_idle_bursts.cpp:35-38, bursttimer.h:30
        h->fm_sens = static_cast<float>((kPi * symbol_rate * 0.85) / if_samp_rate);
        t2 = low_pass_2(sps, 3.0 * samp_rate, filter_width, 2000, 60, WIN_BLACKMAN_HARRIS);
        h->L2 = sps; h->M2 = 3; h->nt2 = (static_cast<int>(t2.size()) + sps - 1) / sps;
        if (sps <= 3 || static_cast<size_t>(h->L2) * h->nt2 * sizeof(float) > 40 * 1024) { set_err(h, "make_gr_mod_dmr: unsupported sps"); return fail(QRL_EINVAL); }
        h->zi.init(h->C);
    } else if (kind == QRL_MOD_2FSK) {
        // gr_mod_2fsk.cpp:43-76
        int nfilts = 25 * sps, spacing = 2; h->amplif = 0.8f;
        if (flag) { spacing = 1; h->amplif = 0.9f; }
        if (sps == 5) nfilts = nfilts * 5;
        if ((nfilts % 2) == 0) nfilts += 1;
        h->repeat_only = flag ? 0 : 1;
        h->pulse_scale = 1.0f;
        t1 = root_raised_cosine(sps, sps, 1, 0.2, nfilts);
        h->L1 = sps; h->nt1 = (static_cast<int>(t1.size()) + sps - 1) / sps;
        h->fm_sens = static_cast<float>((spacing * kPi / 2) / sps);
        t2 = low_pass(10, samp_rate, filter_width, filter_width, WIN_HAMMING);
        h->L2 = 10; h->nt2 = (static_cast<int>(t2.size()) + 9) / 10;
    } else { set_err(h, "qrl_tx_create: mod kind " + std::to_string(kind) + " not built"); return fail(QRL_EINVAL); }
    if ((rc = upload_floats(h, &h->d_arms1, make_arms(t1, h->L1, h->nt1)))) return fail(rc);
    if (!t2.empty() && (rc = upload_floats(h, &h->d_arms2, make_arms(t2, h->L2, h->nt2)))) return fail(rc);
    if ((rc = dev_alloc(h, &h->d_bits, h->C))) return fail(rc);
    if ((rc = dev_alloc(h, &h->d_in, static_cast<size_t>(h->max_items) * h->C))) return fail(rc);
    const bool one_per_bit = kind == QRL_MOD_BPSK || kind == QRL_MOD_2FSK;
    const bool analog = kind == QRL_MOD_NBFM || kind == QRL_MOD_SSB;
    long long max_sym = (one_per_bit ? 16LL : 8LL) * max_items;
    if (kind == QRL_MOD_NBFM) max_sym = max_items * 25 / 4 + 8;        // 50 ksps items per call
    if (kind == QRL_MOD_SSB) max_sym = max_items + 8;                  // 8 ksps complex items per call
    if (h->am_tx) {
        unsigned cap = pow2_at_least(max_items + h->nt_lpf + 64); h->ra_mask = cap - 1; h->ra_stride = cap;
        if ((rc = dev_alloc(h, &h->d_ra, static_cast<size_t>(cap) * h->C))) return fail(rc);
        unsigned cap2 = pow2_at_least(static_cast<long long>(max_items) * h->L2 + h->nt_cfilt + 64); h->rc_mask = cap2 - 1; h->rc_stride = cap2;
        if ((rc = dev_alloc(h, &h->d_rc, static_cast<size_t>(cap2) * h->C))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_rs2, static_cast<size_t>(cap2) * h->C))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_an, h->C))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_audio_in, static_cast<size_t>(max_items) * h->C))) return fail(rc);
        std::vector<TxAnalogState> an(h->C);
        for (auto& a : an) { std::memset(&a, 0, sizeof a); a.agc = 1.0f; }               // agc2_ff::make(1e-2, 1e-4, 1, 1): initial gain 1
        if (cudaMemcpy(h->d_an, an.data(), sizeof(TxAnalogState) * h->C, cudaMemcpyHostToDevice) != cudaSuccess) { set_err(h, "state upload failed"); return fail(QRL_ECUDA); }
    }
    if (h->dsss_tx) {
        max_sym = 16LL * 13 * max_items;                               // chips per call
        unsigned cap1 = pow2_at_least(max_sym * h->L1 + h->nt_cfilt + 128); h->if_mask = cap1 - 1; h->if_stride = cap1;
        if ((rc = dev_alloc(h, &h->d_if, static_cast<size_t>(cap1) * h->C))) return fail(rc);
        const long long n20 = (max_sym * h->L1 * 50 + 12) / 13 + 8;
        unsigned cap2 = pow2_at_least(n20 + h->nt2 + 512); h->rc_mask = cap2 - 1; h->rc_stride = cap2;
        if ((rc = dev_alloc(h, &h->d_rc, static_cast<size_t>(cap2) * h->C))) return fail(rc);
    }
    if (h->m17) {                                                      // IF ring behind the 24 ksps low-pass: 20 samples per byte
        unsigned cap2 = pow2_at_least(max_sym * h->L1 + 512 + h->nt2); h->rc_mask = cap2 - 1; h->rc_stride = cap2;
        if ((rc = dev_alloc(h, &h->d_rc, static_cast<size_t>(cap2) * h->C))) return fail(rc);
    }
    if (analog) {
        unsigned cap = pow2_at_least(max_items + 512); h->ra_mask = cap - 1; h->ra_stride = cap;
        if ((rc = dev_alloc(h, &h->d_ra, static_cast<size_t>(cap) * h->C))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_rb, static_cast<size_t>(cap) * h->C))) return fail(rc);
        unsigned cap2 = pow2_at_least(max_sym + 512); h->rc_mask = cap2 - 1; h->rc_stride = cap2;
        if ((rc = dev_alloc(h, &h->d_rc, static_cast<size_t>(cap2) * h->C))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_rs2, static_cast<size_t>(cap2) * h->C))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_an, h->C))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_audio_in, static_cast<size_t>(max_items) * h->C))) return fail(rc);
    }
    const bool qpsk = kind == QRL_MOD_QPSK || kind == QRL_MOD_BPSK || h->dsss_tx;      // complex symbols (QPSK / BPSK: single interpolation stage)
    { unsigned cap = pow2_at_least(max_sym + 64); h->sym_mask = cap - 1; h->sym_stride = cap;
      if ((rc = dev_alloc(h, &h->d_sym, static_cast<size_t>(cap) * h->C * (qpsk ? 2 : 1)))) return fail(rc); }
    if (!qpsk) {
        unsigned cap = pow2_at_least(max_sym * (analog ? 1 : h->L1) + 128 + h->zi_delay_items); h->if_mask = cap - 1; h->if_stride = cap;
        if ((rc = dev_alloc(h, &h->d_if, static_cast<size_t>(cap) * h->C))) return fail(rc);
    }
    h->out_stride = analog ? max_sym * h->L2 : max_sym * h->L1 * (qpsk ? 1 : h->L2);
    if (h->m17) h->out_stride = (4LL * max_items * h->L1 * h->L2 + h->M2 - 1) / h->M2 + 8;
    if (h->dsss_tx) h->out_stride = ((max_sym * h->L1 * 50 + 12) / 13 + 1) * 50;
    if (h->am_tx) h->out_stride = static_cast<long long>(max_items) * h->L2;
    if ((rc = dev_alloc(h, &h->d_out, static_cast<size_t>(h->out_stride) * h->C, false))) return fail(rc);
    std::vector<TxBitState> st(h->C);
    for (auto& x : st) { x.scr_reg = 0x7F; x.enc_state = 0; x.diff_prev = 0; x.phase_q = 0; }
    if (cudaMemcpy(h->d_bits, st.data(), sizeof(TxBitState) * h->C, cudaMemcpyHostToDevice) != cudaSuccess) { set_err(h, "state upload failed"); return fail(QRL_ECUDA); }
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) { set_err(h, "create sync failed"); return fail(QRL_ECUDA); }
    *out = h;
    return QRL_OK;
}
int qrl_tx_destroy(qrl_tx* h)
{
    if (!h) return QRL_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->s_bits) { cudaStreamSynchronize(h->s_bits); cudaStreamDestroy(h->s_bits); }
    if (h->s_shape) { cudaStreamSynchronize(h->s_shape); cudaStreamDestroy(h->s_shape); }
    for (cudaEvent_t e : { h->ev_start, h->ev_shape_done, h->ev_out_done }) if (e) cudaEventDestroy(e);
    for (int i = 0; i < qrl_tx::kTxSub; i++) { if (h->ev_bits[i]) cudaEventDestroy(h->ev_bits[i]); if (h->ev_shape[i]) cudaEventDestroy(h->ev_shape[i]); }
    for (auto& r : h->prof_recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (void* p : h->allocs) cudaFree(p);
    h->zi.release();
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return QRL_OK;
}
int qrl_tx_set_stream(qrl_tx* h, void* s)
{
    if (!h) return QRL_EINVAL;
    CK(cudaStreamSynchronize(h->stream));
    if (h->own_stream && h->stream) { cudaStreamDestroy(h->stream); h->own_stream = false; }
    if (s) h->stream = static_cast<cudaStream_t>(s);
    else { CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); h->own_stream = true; }
    return QRL_OK;
}
int qrl_tx_set_param(qrl_tx* h, int, int key, double value)
{
    if (!h) return QRL_EINVAL;
    if (key == QRL_PARAM_BB_GAIN) { h->bb_gain = static_cast<float>(value); return QRL_OK; }   // gr_mod_4fsk::set_bb_gain
    if (key == QRL_PARAM_FILTER_WIDTH && h->kind == QRL_MOD_NBFM) {
        // gr_mod_nbfm::set_filter_width (gr_mod_nbfm.cpp:78-93): new taps for the 25/4 resampler, the 50 ksps filter and the final
        // interpolator, new sensitivity.  The rings keep the stream's true history, which the longer filters read from their next output on.
        const int fw = static_cast<int>(value);
        if (fw <= 0) { set_err(h, "qrl_tx_set_param: filter width must be positive"); return QRL_EINVAL; }
        const float if_samp_rate = 50000;
        const std::vector<float> t1 = low_pass_2(25, if_samp_rate * 4, fw, fw, 60, WIN_BLACKMAN_HARRIS);
        const std::vector<float> tc = low_pass_2(1, if_samp_rate, fw, 1200, 60, WIN_BLACKMAN_HARRIS);
        const std::vector<float> t2 = low_pass_2(h->L2, h->samp_rate, fw, fw, 60, WIN_BLACKMAN_HARRIS);
        const int nt1 = (static_cast<int>(t1.size()) + 24) / 25, nt2 = (static_cast<int>(t2.size()) + h->L2 - 1) / h->L2;
        if (nt1 > 256 || static_cast<int>(tc.size()) > 400 || nt2 > 400 || static_cast<size_t>(h->L2) * nt2 * sizeof(float) > 40 * 1024) {
            set_err(h, "qrl_tx_set_param: filter width too small for the rings' history"); return QRL_EINVAL;
        }
        CK(cudaSetDevice(h->device));
        CK(cudaStreamSynchronize(h->stream));
        float *a1 = nullptr, *cf = nullptr, *a2 = nullptr;
        int rc;
        if ((rc = upload_floats(h, &a1, make_arms(t1, 25, nt1)))) return rc;
        if ((rc = upload_floats(h, &cf, tc))) return rc;
        if ((rc = upload_floats(h, &a2, make_arms(t2, h->L2, nt2)))) return rc;
        h->d_arms1 = a1; h->nt1 = nt1; h->d_cfilt = cf; h->nt_cfilt = static_cast<int>(tc.size()); h->d_arms2 = a2; h->nt2 = nt2;
        h->fm_sens = static_cast<float>(4 * kPi * fw / if_samp_rate);
        h->filter_width = fw;
        return QRL_OK;
    }
    if (key == QRL_PARAM_CTCSS && h->kind == QRL_MOD_NBFM) {
        // gr_mod_nbfm::set_ctcss (gr_mod_nbfm.cpp:101-139)
        std::vector<float> lp;
        if (value == 0) { h->audio_gain = 0.98f; h->tone_on = false; lp = low_pass_2(1, 8000, 3500, 200, 35, WIN_BLACKMAN_HARRIS); }
        else {
            h->audio_gain = 0.85f; h->tone_on = true;
            lp = band_pass_2(1, 8000, 300, 3500, 200, 35, WIN_BLACKMAN_HARRIS);
            float x = static_cast<float>(2 * kPi * static_cast<double>(static_cast<float>(value)) / 8000.0);      // fxpt::float_to_fixed
            const int d = static_cast<int>(std::floor(x / static_cast<float>(2.0 * kPi) + 0.5));
            x -= d * static_cast<float>(2.0 * kPi);
            h->tone_inc = static_cast<unsigned>(static_cast<int>(static_cast<float>(x) * 2147483648.0f / static_cast<float>(kPi)));
        }
        if (static_cast<int>(lp.size()) > 400) { set_err(h, "qrl_tx_set_param: audio filter too long"); return QRL_EINVAL; }
        CK(cudaSetDevice(h->device));
        CK(cudaStreamSynchronize(h->stream));
        float* p = nullptr;
        int rc = upload_floats(h, &p, lp);
        if (rc) return rc;
        h->d_lpf = p; h->nt_lpf = static_cast<int>(lp.size());
        return QRL_OK;
    }
    if (key == QRL_PARAM_FILTER_WIDTH && (h->kind == QRL_MOD_SSB || h->am_tx)) {
        // gr_mod_ssb::set_filter_width (gr_mod_ssb.cpp:85-100) / gr_mod_am::set_filter_width (gr_mod_am.cpp:75-85)
        const int fw = static_cast<int>(value);
        if (fw <= 0) { set_err(h, "qrl_tx_set_param: filter width must be positive"); return QRL_EINVAL; }
        std::vector<float> t2, cf;
        if (h->am_tx) {
            t2 = low_pass(h->L2, h->samp_rate, fw, fw, WIN_HAMMING);
            const std::vector<float> cb = complex_band_pass_2(1, h->samp_rate, -fw, fw, 1200, 120, WIN_BLACKMAN_HARRIS);
            cf.resize(cb.size() / 2);
            for (size_t i = 0; i < cf.size(); i++) cf[i] = cb[2 * i];
        } else {
            t2 = low_pass_2(h->L2, h->samp_rate, fw, fw, 90, WIN_BLACKMAN_HARRIS);
            cf = h->flag ? complex_band_pass_2(1, 8000, -fw, -300, 250, 90, WIN_BLACKMAN_HARRIS) : complex_band_pass_2(1, 8000, 300, fw, 250, 90, WIN_BLACKMAN_HARRIS);
        }
        const int nt2 = (static_cast<int>(t2.size()) + h->L2 - 1) / h->L2;
        const int ntc = static_cast<int>(h->am_tx ? cf.size() : cf.size() / 2);
        if (nt2 > 60 || static_cast<size_t>(h->L2) * nt2 * sizeof(float) > 40 * 1024 || ntc > (h->am_tx ? 8192 : 500)) {
            set_err(h, "qrl_tx_set_param: filter width too small for the rings' history"); return QRL_EINVAL;
        }
        CK(cudaSetDevice(h->device));
        CK(cudaStreamSynchronize(h->stream));
        float *a2 = nullptr, *c2 = nullptr;
        int rc;
        if ((rc = upload_floats(h, &a2, make_arms(t2, h->L2, nt2)))) return rc;
        if ((rc = upload_floats(h, &c2, cf))) return rc;
        h->d_arms2 = a2; h->nt2 = nt2; h->d_cfilt = c2; h->nt_cfilt = ntc;
        h->filter_width = fw;
        return QRL_OK;
    }
    set_err(h, "qrl_tx_set_param: unsupported key");
    return QRL_EINVAL;
}
int qrl_tx_work(qrl_tx* h, const void* in, long n, long stride, int on_device)
{
    if (!h || !in || n < 0) return QRL_EINVAL;
    if (n > h->max_items) { set_err(h, "qrl_tx_work: n exceeds max_items given at create"); return QRL_ERANGE; }
    h->n_out_last = 0;
    if (n == 0) return QRL_OK;
    CK(cudaSetDevice(h->device));
    if (on_device) { int rc = check_device_ptr(h, in, "qrl_tx_work"); if (rc) return rc; }
    if (h->am_tx) {
        // `in` = [C][n] float audio at 8 ksps
        const float* au = static_cast<const float*>(in);
        long long astride = stride;
        if (!on_device) {
            CK(cudaMemcpy2DAsync(h->d_audio_in, sizeof(float) * h->max_items, in, sizeof(float) * stride, sizeof(float) * n, h->C,
                                 cudaMemcpyHostToDevice, h->stream));
            au = h->d_audio_in; astride = h->max_items;
        }
        const long long a0 = h->n_audio, a1 = h->n_audio + n;
        tx_am_front_kernel<<<h->C, 128, 0, h->stream>>>(h->d_an, au, n, astride, 1e-2f, 1e-4f, 1.0f, 1.0f,
            h->d_ra, h->ra_mask, h->ra_stride, h->d_lpf, h->nt_lpf, h->am_dc, h->d_if, h->if_mask, h->if_stride);
        const long long o0 = a0 * h->L2, o1 = a1 * h->L2;
        resamp_ring_to_ring_ccf_kernel<<<dim3(static_cast<unsigned>((o1 - o0 + 255) / 256), h->C), 256, sizeof(float) * h->L2 * h->nt2, h->stream>>>(
            h->d_if, h->if_mask, h->if_stride, h->d_arms2, h->L2, 1, h->nt2, o0, o1, h->amplif, h->bb_gain, 1, h->d_rc, h->rc_mask, h->rc_stride);
        h->launches += 2;
        { int rc = launch_fir_ccf_c(h, h->C, h->stream, h->d_rc, h->rc_mask, h->rc_stride, h->d_rs2, h->rc_mask, h->rc_stride, h->d_cfilt, h->nt_cfilt, o0, o1,
                                    h->d_out, h->out_stride, o0, 0); if (rc) return rc; }
        h->n_audio = a1;
        h->n_out_last = static_cast<long>(o1 - o0);
        CK(cudaGetLastError());
        return QRL_OK;
    }
    if (h->kind == QRL_MOD_NBFM || h->kind == QRL_MOD_SSB) {
        // `in` = [C][n] float audio at 8 ksps
        const float* au = static_cast<const float*>(in);
        long long astride = stride;
        if (!on_device) {
            CK(cudaMemcpy2DAsync(h->d_audio_in, sizeof(float) * h->max_items, in, sizeof(float) * stride, sizeof(float) * n, h->C,
                                 cudaMemcpyHostToDevice, h->stream));
            au = h->d_audio_in; astride = h->max_items;
        }
        const int TB = 256;
        if (h->kind == QRL_MOD_NBFM) {
            tx_nbfm_front_kernel<<<h->C, 128, 0, h->stream>>>(h->d_an, au, n, astride, h->d_ra, h->ra_mask, h->ra_stride,
                h->d_rb, h->ra_mask, h->ra_stride, h->d_lpf, h->nt_lpf, h->pe_b0, h->pe_b1, h->pe_a1, h->d_arms1, h->nt1,
                h->d_sym, h->sym_mask, h->sym_stride, h->audio_gain, h->tone_on ? 1 : 0, h->tone_phase, h->tone_inc);
            if (h->tone_on) h->tone_phase += h->tone_inc * static_cast<unsigned>(n);
            const long long r0 = h->n_mid, r1 = ((h->n_audio + n) * 25 + 3) / 4;
            static const float one = 1.0f; (void)one;
            // frequency modulator (Q32 scan) on the 50 ksps stream: "RRC" stage degenerated to a pass-through arm {1}
            tx_shape_fm_kernel<1024, 2><<<h->C, 1024, 0, h->stream>>>(h->d_bits, h->d_sym, h->sym_mask, h->sym_stride, r0, r1 - r0,
                1, 1, h->d_arms1, 1, 1.0f, h->fm_sens, 1.0f, 1.0f, h->d_if, h->if_mask, h->if_stride);
            dim3 g(static_cast<unsigned>((r1 - r0 + TB - 1) / TB), h->C);
            if (r1 > r0) {
                fir_ccf_ring_kernel<<<g, TB, sizeof(float) * h->nt_cfilt, h->stream>>>(h->d_if, h->if_mask, h->if_stride,
                    h->d_rc, h->rc_mask, h->rc_stride, h->d_cfilt, h->nt_cfilt, r0, r1, nullptr, 0, 0, 0);
                scale2_ring_kernel<<<g, TB, 0, h->stream>>>(h->d_rc, h->rc_mask, h->rc_stride, r0, r1, h->amplif, h->bb_gain);
                int MT = std::max(1, 4096 / h->L2);
                const size_t smem = sizeof(float) * ((h->L2 * h->nt2 + 1) & ~1) + sizeof(float2) * (MT + h->nt2);
                dim3 gi(static_cast<unsigned>((r1 - r0 + MT - 1) / MT), h->C);
                interp_fir_ccf_generic_kernel<<<gi, 256, smem, h->stream>>>(h->d_rc, h->rc_mask, h->rc_stride, r0, r1, h->d_arms2, h->L2, h->nt2, MT,
                                                                            1.0f, 1.0f, 0, h->d_out, h->out_stride, r0 * h->L2);
            }
            h->launches += 5;
            h->n_out_last = static_cast<long>((r1 - r0) * h->L2);
            h->n_mid = r1;
        } else {
            tx_ssb_front_kernel<<<h->C, 128, 0, h->stream>>>(h->d_an, au, n, astride, h->d_ra, h->ra_mask, h->ra_stride,
                h->d_rc, h->rc_mask, h->rc_stride, h->d_lpf, h->nt_lpf, 0.95f, static_cast<float>(1 / (std::sqrt(0.5) / 2)),
                h->d_rs2, h->rc_mask, h->rc_stride);
            const long long s0 = h->n_mid, s1 = std::max<long long>(s0, h->n_audio + n - 2);
            if (s1 > s0) {
                dim3 g(static_cast<unsigned>((s1 - s0 + TB - 1) / TB), h->C);
                fir_ccc_ring_kernel<<<g, TB, sizeof(float) * 2 * h->nt_cfilt, h->stream>>>(h->d_rs2, h->rc_mask, h->rc_stride,
                    h->d_if, h->if_mask, h->if_stride, h->d_cfilt, h->nt_cfilt, 1.0f, s0, s1, nullptr, 0, 0);
                scale2_ring_kernel<<<g, TB, 0, h->stream>>>(h->d_if, h->if_mask, h->if_stride, s0, s1, h->amplif, h->bb_gain);
                int MT = std::max(1, 4096 / h->L2);
                const size_t smem = sizeof(float) * ((h->L2 * h->nt2 + 1) & ~1) + sizeof(float2) * (MT + h->nt2);
                dim3 gi(static_cast<unsigned>((s1 - s0 + MT - 1) / MT), h->C);
                interp_fir_ccf_generic_kernel<<<gi, 256, smem, h->stream>>>(h->d_if, h->if_mask, h->if_stride, s0, s1, h->d_arms2, h->L2, h->nt2, MT,
                                                                            1.0f, 1.0f, 0, h->d_out, h->out_stride, s0 * h->L2);
            }
            h->launches += 4;
            h->n_out_last = static_cast<long>((s1 - s0) * h->L2);
            h->n_mid = s1;
        }
        h->n_audio += n;
        CK(cudaGetLastError());
        return QRL_OK;
    }
    const unsigned char* b = static_cast<const unsigned char*>(in);
    long long bstride = stride;
    if (!on_device) {
        CK(cudaMemcpy2DAsync(h->d_in, h->max_items, in, stride, n, h->C, cudaMemcpyHostToDevice, h->stream));
        b = h->d_in; bstride = h->max_items;
    }
    const bool cplx = h->kind == QRL_MOD_QPSK || h->kind == QRL_MOD_BPSK;
    const bool one_per_bit = h->kind == QRL_MOD_BPSK || h->kind == QRL_MOD_2FSK;
    if (h->dsss_tx) {
        const long long sym0 = h->n_sym, nsym = 16LL * 13 * n;                         // chips
        tx_bits_kernel<TXM_DSSS><<<dim3((h->C + 31) / 32), 32, 0, h->stream>>>(h->d_bits, h->C, b, n, bstride, h->d_sym, h->sym_mask, h->sym_stride, sym0);
        // x sps pulse shaping + the two gains -> 5200 sps ring
        const long long a0 = sym0 * h->L1, a1 = (sym0 + nsym) * h->L1;
        resamp_ring_to_ring_ccf_kernel<<<dim3(static_cast<unsigned>((a1 - a0 + 255) / 256), h->C), 256, sizeof(float) * h->L1 * h->nt1, h->stream>>>(
            reinterpret_cast<const float2*>(h->d_sym), h->sym_mask, h->sym_stride, h->d_arms1, h->L1, 1, h->nt1, a0, a1,
            h->amplif, h->bb_gain, 1, h->d_if, h->if_mask, h->if_stride);
        // x50 / 13 -> 20 ksps ring: outputs i with floor(13 i / 50) < a1
        const long long o0 = (a0 * 50 + 12) / 13, o1 = (a1 * 50 + 12) / 13;
        resamp_ring_to_ring_ccf_kernel<<<dim3(static_cast<unsigned>((o1 - o0 + 255) / 256), h->C), 256, sizeof(float) * 50 * h->nt_cfilt, h->stream>>>(
            h->d_if, h->if_mask, h->if_stride, h->d_cfilt, 50, 13, h->nt_cfilt, o0, o1, 1.0f, 1.0f, 0, h->d_rc, h->rc_mask, h->rc_stride);
        // x50 -> output
        if ((o1 - o0) * 50 > h->out_stride) { set_err(h, "qrl_tx_work: output buffer too small"); return QRL_ERANGE; }
        {
            const int L = 50, NT = h->nt2, MT = std::max(1, 4096 / L);
            const size_t smem = sizeof(float) * ((L * NT + 1) & ~1) + sizeof(float2) * (MT + NT);
            dim3 g(static_cast<unsigned>((o1 - o0 + MT - 1) / MT), h->C);
            interp_fir_ccf_generic_kernel<<<g, 256, smem, h->stream>>>(h->d_rc, h->rc_mask, h->rc_stride, o0, o1, h->d_arms2, L, NT, MT, 1.0f, 1.0f, 0,
                                                                       h->d_out, h->out_stride, o0 * L);
        }
        h->launches += 4;
        h->n_out_last = static_cast<long>((o1 - o0) * 50);
        h->n_sym += nsym;
        CK(cudaGetLastError());
        return QRL_OK;
    }
    const long long sym0 = h->n_sym, nsym = (h->m17 ? 4LL : (one_per_bit ? 16LL : 8LL)) * n;
    // 4FSK: bit chain / pulse shaping + FM scan / x20 interpolator are pipelined slice by slice on three streams (the
    // first two are one-CTA-per-channel recurrences that leave most SMs idle; the interpolator fills them)
    bool pipelined = h->kind == QRL_MOD_4FSK && h->L2 == 20 && h->nt2 == 35 && n >= 8 * qrl_tx::kTxSub;
    if (pipelined && !h->s_bits) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        bool ok = cudaStreamCreateWithPriority(&h->s_bits, cudaStreamNonBlocking, hi) == cudaSuccess &&
                  cudaStreamCreateWithPriority(&h->s_shape, cudaStreamNonBlocking, hi) == cudaSuccess;
        auto mk = [&](cudaEvent_t* e) { ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess; };
        mk(&h->ev_start); mk(&h->ev_shape_done); mk(&h->ev_out_done);
        for (int i = 0; i < qrl_tx::kTxSub; i++) { mk(&h->ev_bits[i]); mk(&h->ev_shape[i]); }
        if (!ok) { set_err(h, "qrl_tx_work: stream/event creation failed"); return QRL_ECUDA; }
    }
    if (pipelined) {
        constexpr int S = qrl_tx::kTxSub;
        CK(cudaEventRecord(h->ev_start, h->stream));
        CK(cudaStreamWaitEvent(h->s_bits, h->ev_start, 0));
        CK(cudaStreamWaitEvent(h->s_bits, h->ev_shape_done, 0));      // previous call: symbol ring consumed
        CK(cudaStreamWaitEvent(h->s_shape, h->ev_out_done, 0));       // previous call: IF ring consumed
        const long long out_base = sym0 * h->L1 * h->L2;
        for (int j = 0; j < S; j++) {
            const long b0 = n * j / S, b1 = n * (j + 1) / S;
            if (b1 <= b0) continue;
            const long long symA = sym0 + 8LL * b0, nsym_j = 8LL * (b1 - b0);
            cudaEvent_t pe = h->prof_begin(0, h->s_bits);
            tx_bits_kernel<TXM_4FSK><<<dim3((h->C + 31) / 32), 32, 0, h->s_bits>>>(h->d_bits, h->C, b + b0, b1 - b0, bstride,
                                                                                 h->d_sym, h->sym_mask, h->sym_stride, symA);
            h->prof_end(pe);
            CK(cudaEventRecord(h->ev_bits[j], h->s_bits));
            CK(cudaStreamWaitEvent(h->s_shape, h->ev_bits[j], 0));
            pe = h->prof_begin(1, h->s_shape);
            tx_shape_fm_kernel<1024, 2><<<h->C, 1024, 0, h->s_shape>>>(h->d_bits, h->d_sym, h->sym_mask, h->sym_stride, symA, nsym_j,
                h->L1, h->nt1, h->d_arms1, h->repeat_only, h->pulse_scale, h->fm_sens, h->amplif, h->bb_gain,
                h->d_if, h->if_mask, h->if_stride);
            h->prof_end(pe);
            CK(cudaEventRecord(h->ev_shape[j], h->s_shape));
            CK(cudaStreamWaitEvent(h->stream, h->ev_shape[j], 0));
            constexpr int L = 20, NT = 35, R = 8, G = 16;
            const long long m0 = symA * h->L1, m1 = (symA + nsym_j) * h->L1;
            dim3 g(static_cast<unsigned>((m1 - m0 + R * G - 1) / (R * G)), h->C);
            pe = h->prof_begin(2, h->stream);
            interp_fir_ccf_rt_kernel<L, NT, R, G><<<g, L * G, 0, h->stream>>>(
                h->d_if, h->if_mask, h->if_stride, m0, m1, h->d_arms2, 1.0f, 1.0f, 0, h->d_out, h->out_stride, out_base);
            h->prof_end(pe);
            h->launches += 3;
        }
        CK(cudaEventRecord(h->ev_shape_done, h->s_shape));
        CK(cudaEventRecord(h->ev_out_done, h->stream));
        h->n_out_last = static_cast<long>(nsym * h->L1 * h->L2);
        h->n_sym += nsym;
        CK(cudaGetLastError());
        return QRL_OK;
    }
    {
        dim3 g((h->C + 31) / 32);
        if (h->m17) tx_bits_kernel<TXM_M17><<<g, 32, 0, h->stream>>>(h->d_bits, h->C, b, n, bstride, h->d_sym, h->sym_mask, h->sym_stride, sym0);
        else if (h->kind == QRL_MOD_QPSK) tx_bits_kernel<TXM_QPSK><<<g, 32, 0, h->stream>>>(h->d_bits, h->C, b, n, bstride, h->d_sym, h->sym_mask, h->sym_stride, sym0);
        else if (h->kind == QRL_MOD_BPSK) tx_bits_kernel<TXM_BPSK><<<g, 32, 0, h->stream>>>(h->d_bits, h->C, b, n, bstride, h->d_sym, h->sym_mask, h->sym_stride, sym0);
        else if (h->kind == QRL_MOD_2FSK) tx_bits_kernel<TXM_2FSK><<<g, 32, 0, h->stream>>>(h->d_bits, h->C, b, n, bstride, h->d_sym, h->sym_mask, h->sym_stride, sym0);
        else tx_bits_kernel<TXM_4FSK><<<g, 32, 0, h->stream>>>(h->d_bits, h->C, b, n, bstride, h->d_sym, h->sym_mask, h->sym_stride, sym0);
        h->launches++;
    }
    auto generic_interp = [&](const float2* in, unsigned mask, long long stride_, long long m0, long long m1, const float* arms, int L, int NT,
                              float g1, float g2, int apply) {
        int MT = std::max(1, 4096 / L);
        const size_t smem = sizeof(float) * ((L * NT + 1) & ~1) + sizeof(float2) * (MT + NT);
        dim3 g(static_cast<unsigned>((m1 - m0 + MT - 1) / MT), h->C);
        interp_fir_ccf_generic_kernel<<<g, 256, smem, h->stream>>>(in, mask, stride_, m0, m1, arms, L, NT, MT, g1, g2, apply,
                                                                   h->d_out, h->out_stride, m0 * L);
        h->launches++;
    };
    if (h->m17) {
        // pulse shaping + FM scan (gains of 1: x0.9 and the bb gain sit behind the IF filter here), IF low-pass, gains, x125 / 3
        tx_shape_fm_kernel<1024, 2><<<h->C, 1024, 0, h->stream>>>(h->d_bits, h->d_sym, h->sym_mask, h->sym_stride, sym0, nsym,
            h->L1, h->nt1, h->d_arms1, 0, h->pulse_scale, h->fm_sens, 1.0f, 1.0f, h->d_if, h->if_mask, h->if_stride);
        const long long m0 = sym0 * h->L1, m1 = (sym0 + nsym) * h->L1;
        const int TB = 256;
        dim3 g(static_cast<unsigned>((m1 - m0 + TB - 1) / TB), h->C);
        if (h->dmr_tx) {
            tx_delay_ring_kernel<<<g, TB, 0, h->stream>>>(h->d_if, h->if_mask, h->if_stride, h->d_rc, h->rc_mask, h->rc_stride, m0, m1,
                                                          h->zi_delay_items);
            // the "zero_samples" counters of this call as item ranges (gr_zero_idle_bursts.cpp:61-79: a tag loads the counter, a later
            // one overrides what is left of it, one output is cleared per count)
            std::vector<long long> ranges;
            h->zi.collect(h->C, m0, m1, 0, ranges);
            if (!ranges.empty()) {
                CK(h->zi.upload(ranges, h->stream));
                tx_zero_ranges_kernel<<<static_cast<unsigned>(ranges.size() / 3), 256, 0, h->stream>>>(h->d_rc, h->rc_mask, h->rc_stride, h->zi.d_ranges);
                h->launches++;
            }
        } else {
        fir_ccf_ring_kernel<<<g, TB, sizeof(float) * h->nt_cfilt, h->stream>>>(h->d_if, h->if_mask, h->if_stride,
            h->d_rc, h->rc_mask, h->rc_stride, h->d_cfilt, h->nt_cfilt, m0, m1, nullptr, 0, 0, 0);
        }
        scale2_ring_kernel<<<g, TB, 0, h->stream>>>(h->d_rc, h->rc_mask, h->rc_stride, m0, m1, h->amplif, h->bb_gain);
        const long long o0 = (m0 * h->L2 + h->M2 - 1) / h->M2, o1 = (m1 * h->L2 + h->M2 - 1) / h->M2;   // outputs i with floor(i M / L) < m1
        if (o1 - o0 > h->out_stride) { set_err(h, "qrl_tx_work: output buffer too small"); return QRL_ERANGE; }
        dim3 go(static_cast<unsigned>((o1 - o0 + 255) / 256), h->C);
        resamp_ring_ccf_generic_kernel<<<go, 256, sizeof(float) * h->L2 * h->nt2, h->stream>>>(h->d_rc, h->rc_mask, h->rc_stride,
            h->d_arms2, h->L2, h->M2, h->nt2, o0, o1, h->d_out, h->out_stride);
        h->launches += 4;
        h->n_out_last = static_cast<long>(o1 - o0);
    } else if (cplx) {
        if (h->L1 == 4 && h->nt1 == 16) {
            constexpr int L = 4, NT = 16, MB = 8, MLEN = 64;
            dim3 g(static_cast<unsigned>((nsym + MB * MLEN - 1) / (MB * MLEN)), h->C);
            interp_fir_ccf_kernel<L, NT, MB, MLEN><<<g, L * MB, 0, h->stream>>>(
                reinterpret_cast<const float2*>(h->d_sym), h->sym_mask, h->sym_stride, sym0, sym0 + nsym,
                h->d_arms1, h->amplif, h->bb_gain, 1, h->d_out, h->out_stride, sym0 * L);
            h->launches++;
        } else {
            generic_interp(reinterpret_cast<const float2*>(h->d_sym), h->sym_mask, h->sym_stride, sym0, sym0 + nsym,
                           h->d_arms1, h->L1, h->nt1, h->amplif, h->bb_gain, 1);
        }
        h->n_out_last = static_cast<long>(nsym * h->L1);
    } else {
        tx_shape_fm_kernel<1024, 2><<<h->C, 1024, 0, h->stream>>>(h->d_bits, h->d_sym, h->sym_mask, h->sym_stride, sym0, nsym,
            h->L1, h->nt1, h->d_arms1, h->repeat_only, h->pulse_scale, h->fm_sens, h->amplif, h->bb_gain,
            h->d_if, h->if_mask, h->if_stride);
        h->launches++;
        const long long m0 = sym0 * h->L1, m1 = (sym0 + nsym) * h->L1;
        if (h->L2 == 20 && h->nt2 == 35) {
            constexpr int L = 20, NT = 35, R = 8, G = 16;
            dim3 g(static_cast<unsigned>((m1 - m0 + R * G - 1) / (R * G)), h->C);
            interp_fir_ccf_rt_kernel<L, NT, R, G><<<g, L * G, 0, h->stream>>>(
                h->d_if, h->if_mask, h->if_stride, m0, m1, h->d_arms2, 1.0f, 1.0f, 0, h->d_out, h->out_stride, m0 * L);
            h->launches++;
        } else {
            generic_interp(h->d_if, h->if_mask, h->if_stride, m0, m1, h->d_arms2, h->L2, h->nt2, 1.0f, 1.0f, 0);
        }
        h->n_out_last = static_cast<long>((m1 - m0) * h->L2);
    }
    h->n_sym += nsym;
    CK(cudaGetLastError());
    return QRL_OK;
}
int qrl_tx_zero_samples(qrl_tx* h, int channel, long long byte_offset, long n_samples)
{
    if (!h || channel < -1 || channel >= h->C || byte_offset < 0 || n_samples < 0) return QRL_EINVAL;
    if (!h->dmr_tx) { set_err(h, "qrl_tx_zero_samples: only gr_mod_dmr has a zero-idle stage"); return QRL_EINVAL; }
    // the tag rides through packed_to_unpacked (x8), pack_k_bits(2) (/2) and the x5 pulse shaper: item 20 * byte_offset at the block
    const long long item = byte_offset * 4 * h->L1;
    if (item < static_cast<long long>(h->zi_tag_delay)) return QRL_OK;          // gr_zero_idle_bursts.cpp:63 can never match
    h->zi.add(channel, h->C, item - static_cast<long long>(h->zi_tag_delay), static_cast<unsigned long long>(n_samples), h->n_sym * h->L1);
    return QRL_OK;
}
int qrl_tx_sync(qrl_tx* h)
{
    if (!h) return QRL_EINVAL;
    CK(cudaStreamSynchronize(h->stream));
    return QRL_OK;
}
int qrl_tx_profile(qrl_tx* h, int enable)
{
    if (!h) return QRL_EINVAL;
    CK(cudaStreamSynchronize(h->stream));
    h->prof = enable != 0;
    h->prof_used = 0;
    for (int i = 0; i < 4; i++) { h->prof_ms[i] = 0; h->prof_n[i] = 0; }
    return QRL_OK;
}
int qrl_tx_profile_read(qrl_tx* h, int stage, double* ms_total, long* n_launches)
{
    if (!h || stage < 0 || stage >= 4) return QRL_EINVAL;
    CK(cudaStreamSynchronize(h->stream));
    if (h->s_bits) CK(cudaStreamSynchronize(h->s_bits));
    if (h->s_shape) CK(cudaStreamSynchronize(h->s_shape));
    for (size_t i = 0; i < h->prof_used; i++) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, h->prof_recs[i].a, h->prof_recs[i].b) == cudaSuccess) { h->prof_ms[h->prof_recs[i].stage] += ms; h->prof_n[h->prof_recs[i].stage]++; }
    }
    h->prof_used = 0;
    if (ms_total) *ms_total = h->prof_ms[stage];
    if (n_launches) *n_launches = h->prof_n[stage];
    return QRL_OK;
}
int qrl_tx_read(qrl_tx* h, float* dst, long cap, long* n_out, int dst_on_device)
{
    if (!h || !n_out) return QRL_EINVAL;
    *n_out = h->n_out_last;
    if (dst && h->n_out_last > 0) {
        const long w = std::min(cap, h->n_out_last);
        CK(cudaMemcpy2DAsync(dst, static_cast<size_t>(cap) * 8, h->d_out, static_cast<size_t>(h->out_stride) * 8, static_cast<size_t>(w) * 8, h->C,
                             dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return QRL_OK;
}
int qrl_tx_out_device(qrl_tx* h, float** data, long* stride, long* n_out)
{
    if (!h) return QRL_EINVAL;
    if (data) *data = reinterpret_cast<float*>(h->d_out);
    if (stride) *stride = static_cast<long>(h->out_stride);
    if (n_out) *n_out = h->n_out_last;
    return QRL_OK;
}
long qrl_tx_launch_count(const qrl_tx* h) { return h ? h->launches : 0; }

// ---------------------------------------------------------------------------------------------- front end (device rate >= 2 Msps)
struct qrl_frontend : HandleBase {
    int samp_rate = 0, D = 1, C = 0, ntaps = 0, H = 0, hist_cur = 0;
    long max_in = 0;
    float* d_taps = nullptr;
    float2* d_hist[2] = { nullptr, nullptr };
    float2* d_in = nullptr; float2* d_out = nullptr; long long out_stride = 0; long n_out_last = 0;
    long long n_in = 0, n1 = 0;
    std::vector<RotState> rot; RotState* d_rot = nullptr; bool rot_active = false;
};

int qrl_frontend_destroy(qrl_frontend* h)
{
    if (!h) return QRL_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (void* p : h->allocs) cudaFree(p);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return QRL_OK;
}
int qrl_frontend_create(int samp_rate, int n_channels, long max_in, int device, qrl_frontend** out)
{
    if (!out || n_channels <= 0 || max_in <= 0 || samp_rate < 2000000 || samp_rate % 1000000) { set_err(nullptr, "qrl_frontend_create: bad argument (samp_rate must be a multiple of 1e6, >= 2e6)"); return QRL_EINVAL; }
    *out = nullptr;
    if (qrl_device_count() <= device) { set_err(nullptr, "qrl_frontend_create: no CUDA device (this library has no CPU fallback)"); return QRL_ENODEV; }
    qrl_frontend* h = new qrl_frontend();
    h->samp_rate = samp_rate; h->D = samp_rate / 1000000; h->C = n_channels; h->max_in = max_in; h->device = device;
    auto fail = [&](int rc) { std::string e = h->err; qrl_frontend_destroy(h); g_err = e; return rc; };
    if (cudaSetDevice(device) != cudaSuccess) { set_err(h, "cudaSetDevice failed"); return fail(QRL_ECUDA); }
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { set_err(h, "stream create failed"); return fail(QRL_ECUDA); }
    h->own_stream = true;
    int rc = upload_tables(h);
    if (rc) return fail(rc);
    // gr_demod_base.cpp:1329-1333: low_pass(1, samp_rate, 480000, 100000, BLACKMAN_HARRIS) in rational_resampler_ccf(1, samp_rate / 1e6)
    std::vector<float> taps = low_pass(1, samp_rate, 480000, 100000, WIN_BLACKMAN_HARRIS);
    h->ntaps = static_cast<int>(taps.size());
    h->H = h->ntaps + h->D;
    if ((rc = upload_floats(h, &h->d_taps, taps))) return fail(rc);
    if ((rc = dev_alloc(h, &h->d_hist[0], static_cast<size_t>(h->H) * h->C))) return fail(rc);
    if ((rc = dev_alloc(h, &h->d_hist[1], static_cast<size_t>(h->H) * h->C))) return fail(rc);
    h->out_stride = max_in / h->D + 2;
    if ((rc = dev_alloc(h, &h->d_out, static_cast<size_t>(h->out_stride) * h->C, false))) return fail(rc);
    if ((rc = dev_alloc(h, &h->d_rot, h->C))) return fail(rc);
    h->rot.assign(h->C, RotState{ 0u, 0u, 0 });
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) { set_err(h, "create sync failed"); return fail(QRL_ECUDA); }
    *out = h;
    return QRL_OK;
}
int qrl_frontend_set_stream(qrl_frontend* h, void* s)
{
    if (!h) return QRL_EINVAL;
    CK(cudaStreamSynchronize(h->stream));
    if (h->own_stream && h->stream) { cudaStreamDestroy(h->stream); h->own_stream = false; }
    if (s) h->stream = static_cast<cudaStream_t>(s);
    else { CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); h->own_stream = true; }
    return QRL_OK;
}
int qrl_frontend_set_carrier_offset(qrl_frontend* h, int channel, double offset_hz)
{
    // gr_demod_base::set_carrier_offset (:1220-1225): rotator phase increment 2 pi (-offset) / samp_rate at the DEVICE rate
    if (!h || channel >= h->C) return QRL_EINVAL;
    const unsigned inc = static_cast<unsigned>(static_cast<int>(static_cast<long long>(std::rint(-offset_hz / h->samp_rate * 4294967296.0))));
    for (int c = 0; c < h->C; c++) {
        if (channel >= 0 && c != channel) continue;
        RotState& r = h->rot[c];
        r.base = r.base + r.inc * static_cast<unsigned>(h->n_in - r.n_base);
        r.n_base = h->n_in;
        r.inc = inc;
    }
    h->rot_active = false;
    for (auto& r : h->rot) if (r.inc != 0 || r.base != 0) h->rot_active = true;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->d_rot, h->rot.data(), sizeof(RotState) * h->C, cudaMemcpyHostToDevice));
    return QRL_OK;
}
int qrl_frontend_work(qrl_frontend* h, const float* iq, long T, long stride, int on_device, long* n_out)
{
    if (!h || !iq || T < 0) return QRL_EINVAL;
    if (T > h->max_in) { set_err(h, "qrl_frontend_work: T exceeds max_in given at create"); return QRL_ERANGE; }
    h->n_out_last = 0;
    if (n_out) *n_out = 0;
    if (T == 0) return QRL_OK;
    CK(cudaSetDevice(h->device));
    const float2* x = reinterpret_cast<const float2*>(iq);
    long long xstride = stride;
    if (!on_device) {
        if (!h->d_in) { int rc = dev_alloc(h, &h->d_in, static_cast<size_t>(h->max_in) * h->C, false); if (rc) return rc; }
        CK(cudaMemcpy2DAsync(h->d_in, sizeof(float2) * h->max_in, iq, sizeof(float2) * stride, sizeof(float2) * T, h->C, cudaMemcpyHostToDevice, h->stream));
        x = h->d_in; xstride = h->max_in;
    }
    const long long N = h->n_in + T;
    const long long k0 = h->n1, k1 = (N + h->D - 1) / h->D;              // outputs k with D k <= N - 1
    const RotState* rs = h->rot_active ? h->d_rot : nullptr;
    if (k1 > k0) {
        const size_t smem = sizeof(float) * ((h->ntaps + 1) & ~1) + sizeof(float2) * (127 * h->D + h->ntaps);
        static bool attr[16] = { false };
        if (!attr[h->device & 15]) { CK(cudaFuncSetAttribute(frontend_fir_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024)); attr[h->device & 15] = true; }
        if (smem > 160 * 1024) { set_err(h, "qrl_frontend_work: device rate too high for this kernel"); return QRL_EINVAL; }
        dim3 g(static_cast<unsigned>((k1 - k0 + 127) / 128), h->C);
        frontend_fir_kernel<<<g, 128, smem, h->stream>>>(rs, x, xstride, T, h->n_in, h->d_hist[h->hist_cur], h->H, h->d_taps, h->ntaps, h->D,
                                                          h->d_out, h->out_stride, k0, k1);
        h->launches++;
    }
    dim3 gh((h->H + 127) / 128, h->C);
    frontend_hist_kernel<<<gh, 128, 0, h->stream>>>(rs, x, xstride, T, h->n_in, h->d_hist[h->hist_cur], h->d_hist[h->hist_cur ^ 1], h->H);
    h->launches++;
    h->hist_cur ^= 1;
    h->n_in = N; h->n1 = k1;
    h->n_out_last = static_cast<long>(k1 - k0);
    if (n_out) *n_out = h->n_out_last;
    CK(cudaGetLastError());
    return QRL_OK;
}
int qrl_frontend_out_device(qrl_frontend* h, float** data, long* stride, long* n_out)
{
    if (!h) return QRL_EINVAL;
    if (data) *data = reinterpret_cast<float*>(h->d_out);
    if (stride) *stride = static_cast<long>(h->out_stride);
    if (n_out) *n_out = h->n_out_last;
    return QRL_OK;
}
int qrl_frontend_read(qrl_frontend* h, float* dst, long cap)
{
    if (!h || !dst) return QRL_EINVAL;
    const long w = std::min(cap, h->n_out_last);
    if (w > 0) CK(cudaMemcpy2DAsync(dst, static_cast<size_t>(cap) * 8, h->d_out, static_cast<size_t>(h->out_stride) * 8, static_cast<size_t>(w) * 8, h->C, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return QRL_OK;
}
long qrl_frontend_launch_count(const qrl_frontend* h) { return h ? h->launches : 0; }

// ---------------------------------------------------------------------------------------------- TX front end (1 Msps -> device rate)
namespace {
constexpr int TXF_R = 8;                // outputs per thread and pass of txfront_interp_kernel
constexpr int TXF_SMEM_MAX = 96 * 1024; // >= the 58 KB the kernel needs at 56 Msps
}
struct qrl_txfront : HandleBase {
    int samp_rate = 0, N = 1, C = 0, fmt = QRL_TXFRONT_FC32, ntaps = 0, NTP = 0, H = 0, G = 1, P = 1, hist_cur = 0;
    float scale = 32767.0f;
    long max_in = 0;
    size_t smem = 0;
    float* d_taps = nullptr;                // [NTP][N] chain order
    float2* d_hist[2] = { nullptr, nullptr };
    float2* d_in = nullptr; void* d_out = nullptr; long long out_stride = 0; long n_out_last = 0;
    long long n_in = 0;
    std::vector<RotState> rot; RotState* d_rot = nullptr; bool rot_active = false;
    size_t item_bytes() const { return fmt == QRL_TXFRONT_SC16 ? sizeof(short2) : sizeof(float2); }
};

int qrl_txfront_destroy(qrl_txfront* h)
{
    if (!h) return QRL_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (void* p : h->allocs) cudaFree(p);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return QRL_OK;
}
int qrl_txfront_create(int samp_rate, int n_channels, long max_in, int out_format, float sc16_scale, int device, qrl_txfront** out)
{
    if (!out || n_channels <= 0 || max_in <= 0 || (out_format != QRL_TXFRONT_FC32 && out_format != QRL_TXFRONT_SC16)) {
        set_err(nullptr, "qrl_txfront_create: bad argument"); return QRL_EINVAL;
    }
    if (samp_rate != 1000000 && (samp_rate < 2000000 || samp_rate > 56000000 || samp_rate % 1000000)) {
        set_err(nullptr, "qrl_txfront_create: samp_rate " + std::to_string(samp_rate) + " is not supported (1e6, or a multiple of 1e6 in [2e6, 56e6])");
        return QRL_EINVAL;
    }
    *out = nullptr;
    if (qrl_device_count() <= device) { set_err(nullptr, "qrl_txfront_create: no CUDA device (this library has no CPU fallback)"); return QRL_ENODEV; }
    qrl_txfront* h = new qrl_txfront();
    h->samp_rate = samp_rate; h->N = samp_rate / 1000000; h->C = n_channels; h->max_in = max_in; h->device = device;
    h->fmt = out_format; h->scale = sc16_scale;
    auto fail = [&](int rc) { std::string e = h->err; qrl_txfront_destroy(h); g_err = e; return rc; };
    if (cudaSetDevice(device) != cudaSuccess) { set_err(h, "cudaSetDevice failed"); return fail(QRL_ECUDA); }
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { set_err(h, "stream create failed"); return fail(QRL_ECUDA); }
    h->own_stream = true;
    int rc = upload_tables(h);
    if (rc) return fail(rc);
    if (h->N > 1) {
        // gr_mod_base.cpp:211-258: rational_resampler_ccf(N, 1, low_pass(N, samp_rate, 480000, 20000, BLACKMAN_HARRIS))
        const std::vector<float> taps = low_pass(h->N, samp_rate, 480000, 20000, WIN_BLACKMAN_HARRIS);
        const int N = h->N;
        h->ntaps = static_cast<int>(taps.size());
        const int nt = (h->ntaps + N - 1) / N;
        h->NTP = (nt + TXF_R - 1) / TXF_R * TXF_R;
        h->H = h->NTP - 1;
        std::vector<float> chain(static_cast<size_t>(h->NTP) * N, 0.0f);    // row i = step i of the chain: arm tap k = NTP - 1 - i
        for (int i = 0; i < h->NTP; i++)
            for (int p = 0; p < N; p++) {
                const long j = p + static_cast<long>(h->NTP - 1 - i) * N;
                if (j < h->ntaps) chain[static_cast<size_t>(i) * N + p] = taps[j];
            }
        if ((rc = upload_floats(h, &h->d_taps, chain))) return fail(rc);
        h->G = 256 / N;
        h->P = std::max(1, 1024 / (h->G * TXF_R));
        h->smem = sizeof(float) * ((h->NTP * N + 1) & ~1) + sizeof(float2) * (h->G * TXF_R * h->P + h->NTP - 1);
        if (h->smem > static_cast<size_t>(TXF_SMEM_MAX)) { set_err(h, "qrl_txfront_create: filter too long for the kernel's shared memory"); return fail(QRL_EINVAL); }
        if (cudaFuncSetAttribute(txfront_interp_kernel<TXF_R, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TXF_SMEM_MAX) != cudaSuccess ||
            cudaFuncSetAttribute(txfront_interp_kernel<TXF_R, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TXF_SMEM_MAX) != cudaSuccess) {
            set_err(h, "qrl_txfront_create: cudaFuncSetAttribute failed"); return fail(QRL_ECUDA);
        }
        if ((rc = dev_alloc(h, &h->d_hist[0], static_cast<size_t>(h->H) * h->C))) return fail(rc);
        if ((rc = dev_alloc(h, &h->d_hist[1], static_cast<size_t>(h->H) * h->C))) return fail(rc);
    }
    h->out_stride = static_cast<long long>(max_in) * h->N;
    {
        unsigned char* o = nullptr;
        if ((rc = dev_alloc(h, &o, h->item_bytes() * static_cast<size_t>(h->out_stride) * h->C, false))) return fail(rc);
        h->d_out = o;
    }
    if ((rc = dev_alloc(h, &h->d_rot, h->C))) return fail(rc);
    h->rot.assign(h->C, RotState{ 0u, 0u, 0 });
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) { set_err(h, "create sync failed"); return fail(QRL_ECUDA); }
    *out = h;
    return QRL_OK;
}
int qrl_txfront_set_stream(qrl_txfront* h, void* s)
{
    if (!h) return QRL_EINVAL;
    CK(cudaStreamSynchronize(h->stream));
    if (h->own_stream && h->stream) { cudaStreamDestroy(h->stream); h->own_stream = false; }
    if (s) h->stream = static_cast<cudaStream_t>(s);
    else { CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); h->own_stream = true; }
    return QRL_OK;
}
int qrl_txfront_set_carrier_offset(qrl_txfront* h, int channel, double offset_hz)
{
    // gr_mod_base::set_carrier_offset (:799-805): rotator phase increment 2 pi offset / 1e6, at 1 Msps in front of the resampler
    if (!h || channel < -1 || channel >= h->C) return QRL_EINVAL;
    const unsigned inc = static_cast<unsigned>(static_cast<int>(static_cast<long long>(std::rint(offset_hz / 1e6 * 4294967296.0))));
    for (int c = 0; c < h->C; c++) {
        if (channel >= 0 && c != channel) continue;
        RotState& r = h->rot[c];
        r.base = r.base + r.inc * static_cast<unsigned>(h->n_in - r.n_base);
        r.n_base = h->n_in;
        r.inc = inc;
    }
    h->rot_active = false;
    for (auto& r : h->rot) if (r.inc != 0 || r.base != 0) h->rot_active = true;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->d_rot, h->rot.data(), sizeof(RotState) * h->C, cudaMemcpyHostToDevice));
    return QRL_OK;
}
int qrl_txfront_work(qrl_txfront* h, const float* iq, long n, long stride, int on_device, long* n_out)
{
    if (!h || !iq || n < 0 || stride < n) return QRL_EINVAL;
    if (n > h->max_in) { set_err(h, "qrl_txfront_work: n exceeds max_in given at create"); return QRL_ERANGE; }
    h->n_out_last = 0;
    if (n_out) *n_out = 0;
    if (n == 0) return QRL_OK;
    CK(cudaSetDevice(h->device));
    if (on_device) { int rc = check_device_ptr(h, iq, "qrl_txfront_work"); if (rc) return rc; }
    const float2* x = reinterpret_cast<const float2*>(iq);
    long long xstride = stride;
    if (!on_device) {
        if (!h->d_in) { int rc = dev_alloc(h, &h->d_in, static_cast<size_t>(h->max_in) * h->C, false); if (rc) return rc; }
        CK(cudaMemcpy2DAsync(h->d_in, sizeof(float2) * h->max_in, iq, sizeof(float2) * stride, sizeof(float2) * n, h->C, cudaMemcpyHostToDevice, h->stream));
        x = h->d_in; xstride = h->max_in;
    }
    const RotState* rs = h->rot_active ? h->d_rot : nullptr;
    const bool sc16 = h->fmt == QRL_TXFRONT_SC16;
    if (h->N == 1) {
        dim3 g(static_cast<unsigned>(std::min<long>((n + 255) / 256, 4096)), h->C);
        if (sc16) txfront_rot_kernel<true><<<g, 256, 0, h->stream>>>(rs, x, xstride, n, h->n_in, h->d_out, h->out_stride, h->scale);
        else txfront_rot_kernel<false><<<g, 256, 0, h->stream>>>(rs, x, xstride, n, h->n_in, h->d_out, h->out_stride, h->scale);
        h->launches++;
    } else {
        const int TM = h->G * TXF_R * h->P;
        dim3 g(static_cast<unsigned>((n + TM - 1) / TM), h->C);
        const unsigned nthr = static_cast<unsigned>(h->N * h->G);
        if (sc16)
            txfront_interp_kernel<TXF_R, true><<<g, nthr, h->smem, h->stream>>>(rs, x, xstride, n, h->n_in, h->d_hist[h->hist_cur], h->d_taps, h->N, h->NTP,
                                                                              h->G, h->P, h->d_out, h->out_stride, h->scale);
        else
            txfront_interp_kernel<TXF_R, false><<<g, nthr, h->smem, h->stream>>>(rs, x, xstride, n, h->n_in, h->d_hist[h->hist_cur], h->d_taps, h->N, h->NTP,
                                                                               h->G, h->P, h->d_out, h->out_stride, h->scale);
        dim3 gh((h->H + 127) / 128, h->C);
        frontend_hist_kernel<<<gh, 128, 0, h->stream>>>(rs, x, xstride, n, h->n_in, h->d_hist[h->hist_cur], h->d_hist[h->hist_cur ^ 1], h->H);
        h->launches += 2;
        h->hist_cur ^= 1;
    }
    h->n_in += n;
    h->n_out_last = static_cast<long>(n * h->N);
    if (n_out) *n_out = h->n_out_last;
    CK(cudaGetLastError());
    return QRL_OK;
}
int qrl_txfront_out_device(qrl_txfront* h, void** data, long* stride, long* n_out)
{
    if (!h) return QRL_EINVAL;
    if (data) *data = h->d_out;
    if (stride) *stride = static_cast<long>(h->out_stride);
    if (n_out) *n_out = h->n_out_last;
    return QRL_OK;
}
int qrl_txfront_read(qrl_txfront* h, void* dst, long cap)
{
    if (!h || !dst || cap < 0) return QRL_EINVAL;
    const long w = std::min(cap, h->n_out_last);
    const size_t isz = h->item_bytes();
    if (w > 0) CK(cudaMemcpy2DAsync(dst, static_cast<size_t>(cap) * isz, h->d_out, static_cast<size_t>(h->out_stride) * isz, static_cast<size_t>(w) * isz, h->C, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return QRL_OK;
}
long qrl_txfront_launch_count(const qrl_txfront* h) { return h ? h->launches : 0; }

// ---------------------------------------------------------------------------------------------- design helpers
static int copy_out(const std::vector<float>& v, float* out, int cap, int per_item = 1)
{
    const int n = static_cast<int>(v.size()) / per_item;
    if (n > cap) return -n;
    if (out) std::memcpy(out, v.data(), v.size() * sizeof(float));
    return n;
}
int qrl_firdes_low_pass(double gain, double fs, double fc, double tw, int window, float* out, int cap)
{ return copy_out(low_pass(gain, fs, fc, tw, window), out, cap); }
int qrl_firdes_low_pass_2(double gain, double fs, double fc, double tw, double att, int window, float* out, int cap)
{ return copy_out(low_pass_2(gain, fs, fc, tw, att, window), out, cap); }
int qrl_firdes_band_pass(double gain, double fs, double lo, double hi, double tw, int window, float* out, int cap)
{ return copy_out(band_pass(gain, fs, lo, hi, tw, window), out, cap); }
int qrl_firdes_complex_band_pass(double gain, double fs, double lo, double hi, double tw, int window, float* out, int cap)
{ return copy_out(complex_band_pass(gain, fs, lo, hi, tw, window), out, cap, 2); }
int qrl_firdes_root_raised_cosine(double gain, double fs, double symrate, double alpha, int ntaps, float* out, int cap)
{ return copy_out(root_raised_cosine(gain, fs, symrate, alpha, ntaps), out, cap); }
int qrl_firdes_gaussian(double gain, double spb, double bt, int ntaps, float* out, int cap)
{ return copy_out(gaussian(gain, spb, bt, ntaps), out, cap); }
int qrl_design_table(const char* name, float* out, int cap)
{
    std::string n(name ? name : "");
    if (n == "atan") return copy_out(atan_table(), out, cap);
    if (n == "tanh") return copy_out(tanh_table(), out, cap);
    if (n == "mmse") return copy_out(mmse_table(), out, cap);
    if (n == "fxpt_sine") return copy_out(fxpt_sine_table(), out, cap);
    return QRL_EINVAL;
}
int qrl_design_deemph(int fs, double tau, double* a2, double* b2) { deemph_taps(fs, tau, a2, b2); return QRL_OK; }

int qrl_fir_decim_ccf_device(const float* taps, int ntaps, int D, const float* x_dev, long T, long x_stride,
                             float* y_dev, long y_stride, int C, void* cuda_stream)
{
    if (!taps || ntaps < 1 || ntaps > 65536 || D < 1 || !x_dev || !y_dev || T < 0 || C < 1) { set_err(nullptr, "qrl_fir_decim_ccf_device: bad argument"); return QRL_EINVAL; }
    if (qrl_device_count() < 1) { set_err(nullptr, "qrl_fir_decim_ccf_device: no CUDA device (this library has no CPU fallback)"); return QRL_ENODEV; }
    const long long nout = (static_cast<long long>(T) + D - 1) / D;
    if (nout == 0) return QRL_OK;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    float* d_taps = nullptr;
    HandleBase* h = nullptr;
    CK(cudaMalloc(&d_taps, sizeof(float) * ntaps));
    cudaError_t e = cudaMemcpyAsync(d_taps, taps, sizeof(float) * ntaps, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        dim3 g(static_cast<unsigned>(std::min<long long>((nout + 7) / 8, 148LL * 16)), static_cast<unsigned>(C));
        fir_decim_generic_kernel<<<g, 256, 0, st>>>(d_taps, ntaps, D, reinterpret_cast<const float2*>(x_dev), T, x_stride,
                                                    reinterpret_cast<float2*>(y_dev), y_stride, nout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);          // the tap buffer is released below
    cudaFree(d_taps);
    if (e != cudaSuccess) { set_err(nullptr, std::string("qrl_fir_decim_ccf_device: ") + cudaGetErrorString(e)); return QRL_ECUDA; }
    return QRL_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------- MMDVM channel chains
// gr_demod_mmdvm_multi2.cpp:56-126 behind the channelizer (qrl_pfb): per channel rational_resampler_ccf(24, 25) -> low-pass -> RSSI tags ->
// quadrature_demod_cf -> x level -> float_to_short; gr_mod_mmdvm_multi2.cpp:47-126 in front of the synthesizer: short_to_float -> x level ->
// frequency_modulator_fc -> low-pass -> x0.8 -> rational_resampler_ccf(25, 24) [-> synthesizer -> x 1 / num_channels -> x bb_gain].
struct qrl_mmdvm_rx : HandleBase {
    int C = 0, n_rows = 0, nt_arm = 0, nt2 = 0;
    long max_in = 0;
    int* d_rows = nullptr; float* d_arms = nullptr; float* d_taps2 = nullptr;
    float2 *d_r25 = nullptr, *d_r24 = nullptr, *d_rf = nullptr, *d_in = nullptr;
    unsigned m25 = 0, m24 = 0; long long s25 = 0, s24 = 0;
    short* d_out = nullptr; long long out_stride = 0; long n_out_last = 0;
    float* d_rssi = nullptr; long long rssi_stride = 0; int n_rssi_last = 0; long long rssi_b0_last = 0;
    long long n_in = 0, n24 = 0, n_blocks = 0;
    float qd_gain = 0, level = 1.0f, cal = 0.0f;
    int L = 24, M = 25; bool single = false;       // single: gr_demod_mmdvm (250 ksps in, x12 / 125, RSSI in front of the filter, 10 kHz discriminator)
};
struct qrl_mmdvm_tx : HandleBase {
    int C = 0, n_rows = 0, num_channels = 0, nt_arm = 0, nt2 = 0;
    long max_in = 0;
    int* d_rows = nullptr; float* d_arms = nullptr; float* d_taps2 = nullptr; float* d_one = nullptr;
    TxBitState* d_bits = nullptr;
    short* d_in = nullptr;
    float* d_sym = nullptr; unsigned sym_mask = 0; long long sym_stride = 0;
    float2 *d_if = nullptr, *d_rf = nullptr; unsigned if_mask = 0; long long if_stride = 0;
    float2* d_lin = nullptr; long long lin_stride = 0;
    float2* d_out = nullptr; long long out_stride = 0; long n_out_last = 0;
    long long n_in = 0, n25 = 0;
    float fm_sens = 0, level = 1.0f, bb_gain = 1.0f;
    int L = 25, M = 24; bool single = false;       // single: gr_mod_mmdvm (x125 / 12 to 250 ksps, bb_gain in front of the resampler)
    ZeroIdle zi;                                   // gr_zero_idle_bursts(0): behind the FM modulator (single) / behind the resampler (multi2)
};

template <class H> static int mmdvm_destroy(H* h)
{
    if (!h) return QRL_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (void* p : h->allocs) cudaFree(p);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return QRL_OK;
}
template <class H> static int mmdvm_set_stream(H* h, void* s)
{
    if (!h) return QRL_EINVAL;
    CK(cudaStreamSynchronize(h->stream));
    if (h->own_stream && h->stream) { cudaStreamDestroy(h->stream); h->own_stream = false; }
    if (s) h->stream = static_cast<cudaStream_t>(s);
    else { CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); h->own_stream = true; }
    return QRL_OK;
}
static int mmdvm_rows(HandleBase* h, int** d_rows, const int* rows, int C, int n_rows)
{
    std::vector<int> r(C);
    for (int c = 0; c < C; c++) {
        r[c] = rows ? rows[c] : c;
        if (r[c] < 0 || r[c] >= n_rows) { set_err(h, "mmdvm: row index outside the slab"); return QRL_EINVAL; }
    }
    int rc = dev_alloc(h, d_rows, static_cast<size_t>(C), false);
    if (rc) return rc;
    if (cudaMemcpy(*d_rows, r.data(), sizeof(int) * C, cudaMemcpyHostToDevice) != cudaSuccess) { set_err(h, "mmdvm: row upload failed"); return QRL_ECUDA; }
    return QRL_OK;
}

extern "C" {

int qrl_mmdvm_rx_destroy(qrl_mmdvm_rx* h) { return mmdvm_destroy(h); }
int qrl_mmdvm_rx_set_stream(qrl_mmdvm_rx* h, void* s) { return mmdvm_set_stream(h, s); }
int qrl_mmdvm_rx_create(int variant, int n_channels, const int* rows, int n_rows, int filter_width, long max_in, int device, qrl_mmdvm_rx** out)
{
    if (!out || variant < 0 || variant > 1 || n_channels <= 0 || n_rows < n_channels || max_in <= 0 || filter_width <= 0) { set_err(nullptr, "qrl_mmdvm_rx_create: bad argument"); return QRL_EINVAL; }
    *out = nullptr;
    if (qrl_device_count() <= device) { set_err(nullptr, "qrl_mmdvm_rx_create: no CUDA device (this library has no CPU fallback)"); return QRL_ENODEV; }
    qrl_mmdvm_rx* h = new qrl_mmdvm_rx();
    h->C = n_channels; h->n_rows = n_rows; h->max_in = max_in; h->device = device;
    auto fail = [&](int rc) { std::string e = h->err; qrl_mmdvm_rx_destroy(h); g_err = e; return rc; };
    if (cudaSetDevice(device) != cudaSuccess) { set_err(h, "cudaSetDevice failed"); return fail(QRL_ECUDA); }
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { set_err(h, "stream create failed"); return fail(QRL_ECUDA); }
    h->own_stream = true;
    int rc = upload_tables(h);
    if (rc) return fail(rc);
    if ((rc = mmdvm_rows(h, &h->d_rows, rows, h->C, n_rows))) return fail(rc);
    // gr_demod_mmdvm_multi2.cpp:58-62,66,71,76 | gr_demod_mmdvm.cpp:43-52
    h->single = variant == 1;
    h->L = h->single ? 12 : 24; h->M = h->single ? 125 : 25;
    const std::vector<float> ti = h->single ? low_pass_2(12, 12 * 250000.0, filter_width, 2000, 60, WIN_BLACKMAN_HARRIS)
                                            : low_pass_2(1, 600000.0, filter_width, 2000, 60, WIN_BLACKMAN_HARRIS);
    const std::vector<float> tf = low_pass_2(1, 24000.0, filter_width, 2000, 60, WIN_BLACKMAN_HARRIS);
    h->nt_arm = (static_cast<int>(ti.size()) + h->L - 1) / h->L; h->nt2 = static_cast<int>(tf.size());
    if (static_cast<size_t>(h->L) * h->nt_arm * sizeof(float) > 40 * 1024 || h->nt2 > kMaxTapsSmem) { set_err(h, "qrl_mmdvm_rx_create: filter_width too small"); return fail(QRL_EINVAL); }
    if ((rc = upload_floats(h, &h->d_arms, make_arms(ti, h->L, h->nt_arm)))) return fail(rc);
    if ((rc = upload_floats(h, &h->d_taps2, tf))) return fail(rc);
    h->qd_gain = static_cast<float>(24000.0f / (2 * kPi * (h->single ? 10000.0f : 12500.0f)));
    const unsigned c25 = pow2_at_least(max_in + h->nt_arm + 64), c24 = pow2_at_least(max_in + h->nt2 + 400);
    h->m25 = c25 - 1; h->s25 = c25; h->m24 = c24 - 1; h->s24 = c24;
    if ((rc = dev_alloc(h, &h->d_r25, static_cast<size_t>(c25) * h->C))) return fail(rc);
    if ((rc = dev_alloc(h, &h->d_r24, static_cast<size_t>(c24) * h->C))) return fail(rc);
    if ((rc = dev_alloc(h, &h->d_rf, static_cast<size_t>(c24) * h->C))) return fail(rc);
    h->out_stride = max_in * h->L / h->M + 2;
    if ((rc = dev_alloc(h, &h->d_out, static_cast<size_t>(h->out_stride) * h->C, false))) return fail(rc);
    h->rssi_stride = h->out_stride / 300 + 2;
    if ((rc = dev_alloc(h, &h->d_rssi, static_cast<size_t>(h->rssi_stride) * h->C, false))) return fail(rc);
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) { set_err(h, "create sync failed"); return fail(QRL_ECUDA); }
    *out = h;
    return QRL_OK;
}
int qrl_mmdvm_rx_calibrate_rssi(qrl_mmdvm_rx* h, float level) { if (!h) return QRL_EINVAL; h->cal = level; return QRL_OK; }   // rssi_tag_block::calibrate_rssi
int qrl_mmdvm_rx_work(qrl_mmdvm_rx* h, const float* iq, long n, long stride, int on_device, long* n_out)
{
    if (!h || !iq || n < 0) return QRL_EINVAL;
    if (n > h->max_in) { set_err(h, "qrl_mmdvm_rx_work: n exceeds max_in given at create"); return QRL_ERANGE; }
    h->n_out_last = 0; h->n_rssi_last = 0;
    if (n_out) *n_out = 0;
    if (n == 0) return QRL_OK;
    CK(cudaSetDevice(h->device));
    const float2* x = reinterpret_cast<const float2*>(iq);
    long long xstride = stride;
    if (on_device) { int rc = check_device_ptr(h, iq, "qrl_mmdvm_rx_work"); if (rc) return rc; }
    else {
        if (!h->d_in) { int rc = dev_alloc(h, &h->d_in, static_cast<size_t>(h->max_in) * h->n_rows, false); if (rc) return rc; }
        CK(cudaMemcpy2DAsync(h->d_in, sizeof(float2) * h->max_in, iq, sizeof(float2) * stride, sizeof(float2) * n, h->n_rows, cudaMemcpyHostToDevice, h->stream));
        x = h->d_in; xstride = h->max_in;
    }
    const int TB = 256;
    mmdvm_gather_kernel<<<dim3(static_cast<unsigned>(std::min<long long>((n + TB - 1) / TB, 4096)), h->C), TB, 0, h->stream>>>(
        x, xstride, h->d_rows, n, h->d_r25, h->m25, h->s25, h->n_in);
    const long long N = h->n_in + n;
    const long long o0 = h->n24, o1 = (N * h->L + h->M - 1) / h->M;    // outputs o whose newest input floor(M o / L) has arrived
    h->launches++;
    if (o1 > o0) {
        dim3 g(static_cast<unsigned>((o1 - o0 + TB - 1) / TB), h->C);
        if (!h->single && h->nt_arm == 35) {       // the reference's filter width (5000 Hz: 819 taps): tiled instance
            const int span_cap = 256 * 25 / 24 + 35 + 4;
            const size_t smem = sizeof(float) * ((24 * 35 + 1) & ~1) + sizeof(float2) * span_cap;
            resamp_ring_to_ring_tiled_kernel<35><<<g, 256, smem, h->stream>>>(h->d_r25, h->m25, h->s25, h->d_arms, 24, 25, o0, o1, h->d_r24, h->m24, h->s24, span_cap);
        } else {
            resamp_ring_to_ring_ccf_kernel<<<g, TB, sizeof(float) * h->L * h->nt_arm, h->stream>>>(h->d_r25, h->m25, h->s25, h->d_arms, h->L, h->M, h->nt_arm, o0, o1,
                                                                                                    1.0f, 1.0f, 0, h->d_r24, h->m24, h->s24);
        }
        { int rc = launch_fir_ccf_c(h, h->C, h->stream, h->d_r24, h->m24, h->s24, h->d_rf, h->m24, h->s24, h->d_taps2, h->nt2, o0, o1, nullptr, 0, 0, 0); if (rc) return rc; h->launches--; }
        mmdvm_demod_short_kernel<<<g, TB, 0, h->stream>>>(h->d_rf, h->m24, h->s24, o0, o1, h->qd_gain, h->level, h->d_out, h->out_stride);
        h->launches += 3;
        const long long b1 = o1 / 300;                                   // complete 300-item blocks so far
        if (b1 > h->n_blocks) {
            const int nb = static_cast<int>(b1 - h->n_blocks);
            // gr_demod_mmdvm tags the resampler's output, gr_demod_mmdvm_multi2 the channel filter's
            mmdvm_rssi_kernel<<<dim3((nb + 63) / 64, h->C), 64, 0, h->stream>>>(h->single ? h->d_r24 : h->d_rf, h->m24, h->s24, h->n_blocks, nb, h->cal, h->d_rssi, h->rssi_stride);
            h->launches++;
            h->n_rssi_last = nb; h->rssi_b0_last = h->n_blocks; h->n_blocks = b1;
        }
    }
    h->n_in = N; h->n24 = o1;
    h->n_out_last = static_cast<long>(o1 - o0);
    if (n_out) *n_out = h->n_out_last;
    CK(cudaGetLastError());
    return QRL_OK;
}
int qrl_mmdvm_rx_out_device(qrl_mmdvm_rx* h, short** data, long* stride, long* n_out, float** rssi_db, long* rssi_stride, int* n_rssi, long long* first_rssi_item)
{
    if (!h) return QRL_EINVAL;
    if (data) *data = h->d_out;
    if (stride) *stride = static_cast<long>(h->out_stride);
    if (n_out) *n_out = h->n_out_last;
    if (rssi_db) *rssi_db = h->d_rssi;
    if (rssi_stride) *rssi_stride = static_cast<long>(h->rssi_stride);
    if (n_rssi) *n_rssi = h->n_rssi_last;
    if (first_rssi_item) *first_rssi_item = h->rssi_b0_last * 300 + 299;
    return QRL_OK;
}
int qrl_mmdvm_rx_read(qrl_mmdvm_rx* h, short* dst, long dst_stride, float* rssi_db, long rssi_cap, int* n_rssi, long long* first_rssi_item)
{
    if (!h || !dst) return QRL_EINVAL;
    CK(cudaSetDevice(h->device));
    if (h->n_out_last > 0)
        CK(cudaMemcpy2DAsync(dst, sizeof(short) * dst_stride, h->d_out, sizeof(short) * h->out_stride, sizeof(short) * h->n_out_last, h->C, cudaMemcpyDeviceToHost, h->stream));
    const int nr = static_cast<int>(std::min<long>(h->n_rssi_last, rssi_cap));
    if (rssi_db && nr > 0)
        CK(cudaMemcpy2DAsync(rssi_db, sizeof(float) * rssi_cap, h->d_rssi, sizeof(float) * h->rssi_stride, sizeof(float) * nr, h->C, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (n_rssi) *n_rssi = nr;
    if (first_rssi_item) *first_rssi_item = h->rssi_b0_last * 300 + 299;
    return QRL_OK;
}
long qrl_mmdvm_rx_launch_count(qrl_mmdvm_rx* h) { return h ? h->launches : 0; }

int qrl_mmdvm_tx_destroy(qrl_mmdvm_tx* h) { if (h) { cudaSetDevice(h->device); if (h->stream) cudaStreamSynchronize(h->stream); h->zi.release(); } return mmdvm_destroy(h); }
int qrl_mmdvm_tx_set_stream(qrl_mmdvm_tx* h, void* s) { return mmdvm_set_stream(h, s); }
int qrl_mmdvm_tx_create(int variant, int n_channels, const int* rows, int n_rows, int filter_width, long max_in, int device, qrl_mmdvm_tx** out)
{
    if (!out || variant < 0 || variant > 1 || n_channels <= 0 || n_rows < n_channels || max_in <= 0 || filter_width <= 0) { set_err(nullptr, "qrl_mmdvm_tx_create: bad argument"); return QRL_EINVAL; }
    *out = nullptr;
    if (qrl_device_count() <= device) { set_err(nullptr, "qrl_mmdvm_tx_create: no CUDA device (this library has no CPU fallback)"); return QRL_ENODEV; }
    qrl_mmdvm_tx* h = new qrl_mmdvm_tx();
    h->C = n_channels; h->n_rows = n_rows; h->num_channels = n_channels; h->max_in = max_in; h->device = device;
    h->zi.init(h->C);
    auto fail = [&](int rc) { std::string e = h->err; qrl_mmdvm_tx_destroy(h); g_err = e; return rc; };
    if (cudaSetDevice(device) != cudaSuccess) { set_err(h, "cudaSetDevice failed"); return fail(QRL_ECUDA); }
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { set_err(h, "stream create failed"); return fail(QRL_ECUDA); }
    h->own_stream = true;
    int rc = upload_tables(h);
    if (rc) return fail(rc);
    if ((rc = mmdvm_rows(h, &h->d_rows, rows, h->C, n_rows))) return fail(rc);
    // gr_mod_mmdvm_multi2.cpp:47-50,64,72,80 | gr_mod_mmdvm.cpp:36-45
    h->single = variant == 1;
    h->L = h->single ? 125 : 25; h->M = h->single ? 12 : 24;
    const std::vector<float> ti = h->single ? low_pass_2(125, 125 * 24000.0, filter_width, 2000, 60, WIN_BLACKMAN_HARRIS)
                                            : low_pass_2(25, 600000.0, filter_width, 2000, 60, WIN_BLACKMAN_HARRIS);
    const std::vector<float> tf = low_pass_2(1, 24000.0, filter_width, 2000, 60, WIN_BLACKMAN_HARRIS);
    h->nt_arm = (static_cast<int>(ti.size()) + h->L - 1) / h->L; h->nt2 = static_cast<int>(tf.size());
    if (static_cast<size_t>(h->L) * h->nt_arm * sizeof(float) > 40 * 1024 || h->nt2 > kMaxTapsSmem) { set_err(h, "qrl_mmdvm_tx_create: filter_width too small"); return fail(QRL_EINVAL); }
    if ((rc = upload_floats(h, &h->d_arms, make_arms(ti, h->L, h->nt_arm)))) return fail(rc);
    if ((rc = upload_floats(h, &h->d_taps2, tf))) return fail(rc);
    if ((rc = upload_floats(h, &h->d_one, std::vector<float>{ 1.0f }))) return fail(rc);
    h->fm_sens = static_cast<float>(2 * kPi * 12500.0f / 24000.0f);
    if ((rc = dev_alloc(h, &h->d_bits, h->C))) return fail(rc);
    { std::vector<TxBitState> st(h->C); for (auto& x : st) { x.scr_reg = 0x7F; x.enc_state = 0; x.diff_prev = 0; x.phase_q = 0; }
      if (cudaMemcpy(h->d_bits, st.data(), sizeof(TxBitState) * h->C, cudaMemcpyHostToDevice) != cudaSuccess) { set_err(h, "state upload failed"); return fail(QRL_ECUDA); } }
    { const unsigned cap = pow2_at_least(max_in + 64); h->sym_mask = cap - 1; h->sym_stride = cap;
      if ((rc = dev_alloc(h, &h->d_sym, static_cast<size_t>(cap) * h->C))) return fail(rc); }
    { const unsigned cap = pow2_at_least(max_in + std::max(h->nt2, h->nt_arm) + 128); h->if_mask = cap - 1; h->if_stride = cap;
      if ((rc = dev_alloc(h, &h->d_if, static_cast<size_t>(cap) * h->C))) return fail(rc);
      if ((rc = dev_alloc(h, &h->d_rf, static_cast<size_t>(cap) * h->C))) return fail(rc); }
    h->lin_stride = max_in * h->L / h->M + 4; h->out_stride = h->lin_stride;
    if ((rc = dev_alloc(h, &h->d_lin, static_cast<size_t>(h->lin_stride) * h->C, false))) return fail(rc);
    if ((rc = dev_alloc(h, &h->d_out, static_cast<size_t>(h->out_stride) * h->n_rows))) return fail(rc);      // unused rows stay zero (null_source)
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) { set_err(h, "create sync failed"); return fail(QRL_ECUDA); }
    *out = h;
    return QRL_OK;
}
int qrl_mmdvm_tx_set_bb_gain(qrl_mmdvm_tx* h, float g) { if (!h) return QRL_EINVAL; h->bb_gain = g; return QRL_OK; }      // gr_mod_mmdvm_multi2::set_bb_gain
int qrl_mmdvm_tx_zero_samples(qrl_mmdvm_tx* h, int channel, long long item_offset, long n_samples)
{
    if (!h || channel < -1 || channel >= h->C || item_offset < 0 || n_samples < 0) return QRL_EINVAL;
    h->zi.add(channel, h->C, item_offset, static_cast<unsigned long long>(n_samples), h->single ? h->n_in : h->n25);
    return QRL_OK;
}
int qrl_mmdvm_tx_work(qrl_mmdvm_tx* h, const short* in, long n, long stride, int on_device, long* n_out)
{
    if (!h || !in || n < 0) return QRL_EINVAL;
    if (n > h->max_in) { set_err(h, "qrl_mmdvm_tx_work: n exceeds max_in given at create"); return QRL_ERANGE; }
    h->n_out_last = 0;
    if (n_out) *n_out = 0;
    if (n == 0) return QRL_OK;
    CK(cudaSetDevice(h->device));
    const short* s = in; long long sstride = stride;
    if (on_device) { int rc = check_device_ptr(h, in, "qrl_mmdvm_tx_work"); if (rc) return rc; }
    else {
        if (!h->d_in) { int rc = dev_alloc(h, &h->d_in, static_cast<size_t>(h->max_in) * h->C, false); if (rc) return rc; }
        CK(cudaMemcpy2DAsync(h->d_in, sizeof(short) * h->max_in, in, sizeof(short) * stride, sizeof(short) * n, h->C, cudaMemcpyHostToDevice, h->stream));
        s = h->d_in; sstride = h->max_in;
    }
    const int TB = 256;
    const long long a0 = h->n_in, a1 = h->n_in + n;
    mmdvm_short_float_kernel<<<dim3(static_cast<unsigned>(std::min<long long>((n + TB - 1) / TB, 4096)), h->C), TB, 0, h->stream>>>(
        s, sstride, n, h->level, h->d_sym, h->sym_mask, h->sym_stride, a0);
    // frequency_modulator_fc: the FM scan kernel with a one-tap "pulse" (x * 1.0 is exact), Q32 phase carried in the state
    tx_shape_fm_kernel<1024, 2><<<h->C, 1024, 0, h->stream>>>(h->d_bits, h->d_sym, h->sym_mask, h->sym_stride, a0, n,
        1, 1, h->d_one, 0, 1.0f, h->fm_sens, 1.0f, 1.0f, h->d_if, h->if_mask, h->if_stride);
    if (h->single) {
        // gr_mod_mmdvm.cpp:51-58: gr_zero_idle_bursts(0) between the FM modulator and the filter (items of the 24 ksps stream)
        std::vector<long long> ranges;
        h->zi.collect(h->C, a0, a1, 0, ranges);
        if (!ranges.empty()) {
            CK(h->zi.upload(ranges, h->stream));
            tx_zero_ranges_kernel<<<static_cast<unsigned>(ranges.size() / 3), 256, 0, h->stream>>>(h->d_if, h->if_mask, h->if_stride, h->zi.d_ranges);
            h->launches++;
        }
    }
    dim3 g(static_cast<unsigned>((n + TB - 1) / TB), h->C);
    { int rc = launch_fir_ccf_c(h, h->C, h->stream, h->d_if, h->if_mask, h->if_stride, h->d_rf, h->if_mask, h->if_stride, h->d_taps2, h->nt2, a0, a1, nullptr, 0, 0, 0); if (rc) return rc; h->launches--; }
    scale2_ring_kernel<<<g, TB, 0, h->stream>>>(h->d_rf, h->if_mask, h->if_stride, a0, a1, 0.8f, h->single ? h->bb_gain : 1.0f);   // gr_mod_mmdvm: bb_gain here
    const long long o0 = h->n25, o1 = (a1 * h->L + h->M - 1) / h->M;     // outputs i with floor(M i / L) < a1
    if (o1 - o0 > h->lin_stride) { set_err(h, "qrl_mmdvm_tx_work: output buffer too small"); return QRL_ERANGE; }
    if (o1 > o0) {
        dim3 go(static_cast<unsigned>((o1 - o0 + 255) / 256), h->C);
        resamp_ring_ccf_generic_kernel<<<go, 256, sizeof(float) * h->L * h->nt_arm, h->stream>>>(h->d_rf, h->if_mask, h->if_stride, h->d_arms, h->L, h->M, h->nt_arm, o0, o1,
                                                                                               h->d_lin, h->lin_stride);
        if (!h->single) {
            // gr_mod_mmdvm_multi2.cpp:88,108-117: gr_zero_idle_bursts(0) between the x25/24 resampler and the synthesizer (items of the
            // 25 ksps stream; the linear buffer holds items o0 .. o1 of this call)
            std::vector<long long> ranges;
            h->zi.collect(h->C, o0, o1, o0, ranges);
            if (!ranges.empty()) {
                CK(h->zi.upload(ranges, h->stream));
                tx_zero_ranges_kernel<<<static_cast<unsigned>(ranges.size() / 3), 256, 0, h->stream>>>(h->d_lin, 0xffffffffu, h->lin_stride, h->zi.d_ranges);
                h->launches++;
            }
        }
        mmdvm_scatter_kernel<<<dim3(static_cast<unsigned>(std::min<long long>((o1 - o0 + TB - 1) / TB, 4096)), h->C), TB, 0, h->stream>>>(
            h->d_lin, h->lin_stride, h->d_rows, o1 - o0, h->d_out, h->out_stride);
    }
    h->launches += 6;
    h->n_in = a1; h->n25 = o1;
    h->n_out_last = static_cast<long>(o1 - o0);
    if (n_out) *n_out = h->n_out_last;
    CK(cudaGetLastError());
    return QRL_OK;
}
int qrl_mmdvm_tx_out_device(qrl_mmdvm_tx* h, float** data, long* stride, long* n_out)
{
    if (!h) return QRL_EINVAL;
    if (data) *data = reinterpret_cast<float*>(h->d_out);
    if (stride) *stride = static_cast<long>(h->out_stride);
    if (n_out) *n_out = h->n_out_last;
    return QRL_OK;
}
int qrl_mmdvm_tx_read(qrl_mmdvm_tx* h, float* dst, long dst_stride)
{
    if (!h || !dst) return QRL_EINVAL;
    CK(cudaSetDevice(h->device));
    if (h->n_out_last > 0)
        CK(cudaMemcpy2DAsync(dst, sizeof(float2) * dst_stride, h->d_out, sizeof(float2) * h->out_stride, sizeof(float2) * h->n_out_last, h->n_rows, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return QRL_OK;
}
// behind the synthesizer (gr_mod_mmdvm_multi2.cpp:94-96,123-125): multiply_const_cc(1 / num_channels) -> multiply_const_cc(bb_gain), in place
int qrl_mmdvm_tx_finish(qrl_mmdvm_tx* h, float* wideband_dev, long n)
{
    if (!h || !wideband_dev || n < 0) return QRL_EINVAL;
    if (n == 0) return QRL_OK;
    CK(cudaSetDevice(h->device));
    int rc = check_device_ptr(h, wideband_dev, "qrl_mmdvm_tx_finish"); if (rc) return rc;
    scale2_linear_kernel<<<static_cast<unsigned>(std::min<long>((n + 255) / 256, 4096)), 256, 0, h->stream>>>(
        reinterpret_cast<float2*>(wideband_dev), n, 1.0f / static_cast<float>(h->num_channels), h->bb_gain);
    h->launches++;
    CK(cudaGetLastError());
    return QRL_OK;
}
int qrl_mmdvm_rx_sync(qrl_mmdvm_rx* h) { if (!h) return QRL_EINVAL; CK(cudaStreamSynchronize(h->stream)); return QRL_OK; }
int qrl_mmdvm_tx_sync(qrl_mmdvm_tx* h) { if (!h) return QRL_EINVAL; CK(cudaStreamSynchronize(h->stream)); return QRL_OK; }
long qrl_mmdvm_tx_launch_count(qrl_mmdvm_tx* h) { return h ? h->launches : 0; }

}  // extern "C"

#ifdef QRL_SS_PROF
// profiling build only (tools/ss_prof.py): read and clear the symbol-sync loop warp's cycle counters
extern "C" int qrl_debug_ss_prof(long long* out16)
{
    if (cudaMemcpyFromSymbol(out16, qrl::d_ss_prof, sizeof(long long) * 16) != cudaSuccess) return -1;
    long long z[16] = { 0 };
    return cudaMemcpyToSymbol(qrl::d_ss_prof, z, sizeof(z)) == cudaSuccess ? 0 : -1;
}
#endif
