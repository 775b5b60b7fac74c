// qrl_b200_gr.hpp -- header-only C++ host side above the C ABI (include/qrl_b200.h), mirroring the operator surface
// QRadioLink's gr_demod_base / gr_mod_base / gr_modem use for the hot path:
//
//   make_gr_demod_4fsk(sps, samp_rate, carrier_freq, filter_width, fm)      src/gr/gr_demod_4fsk.h:51-53
//   make_gr_demod_qpsk(sps, samp_rate, carrier_freq, filter_width)          src/gr/gr_demod_qpsk.h:48-50
//   make_gr_demod_nbfm(sps, samp_rate, carrier_freq, filter_width)          src/gr/gr_demod_nbfm.h:38-39
//   make_gr_demod_{bpsk,2fsk,ssb,am,gmsk}(...)                              src/gr/gr_demod_<mode>.h
//   make_gr_mod_4fsk / make_gr_mod_qpsk                                     src/gr/gr_mod_4fsk.h:46-48
//   gr_bit_sink / gr_audio_sink / gr_const_sink  get_data() semantics       src/gr/gr_bit_sink.cpp:45-84 ...
//
// The reference's toolchain (GNU Radio 3.10 + Qt5) is not available in this image, so these classes do not derive
// from gr::block; they keep its streaming contract instead: work(noutput-style chunk) with state carried across
// calls, one caller thread per object, constructor failure -> std::runtime_error (what RadioController::toggleRX
// catches, radiocontroller.cpp:1975-1984), work() never throws (returns WORK_DONE = -1 on a shim error).
// INTEGRATION.md shows the 30-line gr::block adapter that wraps exactly this class inside GNU Radio.
#pragma once
#include <algorithm>
#include <complex>
#include <cstdint>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "qrl_b200.h"

namespace qrl_gr {

using gr_complex = std::complex<float>;
static const int WORK_DONE = -1;

// ---- sink blocks: what gr_modem::demodulate()/demodulateAnalog() poll (caller deletes the returned vector).
// Like the reference's, they are crossed by two threads (the block thread calls work(), the radioop thread polls get_data()):
// every access to the buffer is under the mutex (gr_bit_sink.cpp:47,70; gr_audio_sink.cpp:51,74; gr_const_sink.cpp:51,80).
class gr_bit_sink {
public:
    int work(const unsigned char* in, int n)
    {
        if (n < 1) return n;
        std::lock_guard<std::mutex> guard(_mutex);
        if (_data.size() > 1048576) return n;                 // reader too slow: drop (gr_bit_sink.cpp:71-76)
        _data.insert(_data.end(), in, in + n);
        return n;
    }
    std::vector<unsigned char>* get_data()
    {
        std::lock_guard<std::mutex> guard(_mutex);
        if (_data.size() < 32) return nullptr;               // gr_bit_sink.cpp:49-52
        auto* d = new std::vector<unsigned char>(_data);
        _data.clear();
        return d;
    }
    void flush() { std::lock_guard<std::mutex> guard(_mutex); _data.clear(); }
private:
    std::vector<unsigned char> _data;
    std::mutex _mutex;
};

class gr_audio_sink {
public:
    int work(const float* in, int n)
    {
        if (n < 1) return n;
        std::lock_guard<std::mutex> guard(_mutex);
        if (_data.size() > 8000) { _data.clear(); return n; }  // gr_audio_sink.cpp:77-83
        _data.insert(_data.end(), in, in + n);
        return n;
    }
    std::vector<float>* get_data()
    {
        std::lock_guard<std::mutex> guard(_mutex);
        const size_t pkt = 640;                               // 40 ms packets, gr_audio_sink.cpp:53
        if (_data.size() < pkt) return nullptr;
        auto* d = new std::vector<float>(_data.begin(), _data.begin() + pkt);
        _data.erase(_data.begin(), _data.begin() + pkt);
        return d;
    }
    void flush() { std::lock_guard<std::mutex> guard(_mutex); _data.clear(); }
private:
    std::vector<float> _data;
    std::mutex _mutex;
};

class gr_const_sink {
public:
    int work(const gr_complex* in, int n)
    {
        if (n < 1) return n;
        std::lock_guard<std::mutex> guard(_mutex);            // (the reference tests the size before locking: benign there, not copied)
        if (_data.size() > 256) return n;                     // gr_const_sink.cpp:75-79
        _data.insert(_data.end(), in, in + n);
        return n;
    }
    std::vector<gr_complex>* get_data()
    {
        std::lock_guard<std::mutex> guard(_mutex);
        if (_data.size() < 32) return nullptr;
        auto* d = new std::vector<gr_complex>(_data);
        _data.clear();
        return d;
    }
    void flush() { std::lock_guard<std::mutex> guard(_mutex); _data.clear(); }
private:
    std::vector<gr_complex> _data;
    std::mutex _mutex;
};

class gr_sample_sink {      // src/gr/gr_sample_sink.cpp: time-domain display tap behind gr_demod_base::get_sample_data (gr_demod_base.cpp:988-1006)
public:
    int work(const gr_complex* in, int n)
    {
        std::lock_guard<std::mutex> guard(_mutex);
        if (n < 1 || !_enabled) return n;
        if (_data.size() > 524288) return n;                  // gr_sample_sink.cpp:77-82
        _data.insert(_data.end(), in, in + n);
        return n;
    }
    std::vector<gr_complex>* get_data()
    {
        std::lock_guard<std::mutex> guard(_mutex);
        if (_data.size() < 2) return nullptr;
        unsigned size = std::min(static_cast<unsigned>(_data.size()), _window_size);
        if (size % 2 != 0) size = size - 1;
        auto* d = new std::vector<gr_complex>(_data.begin(), _data.begin() + size);
        _data.erase(_data.begin(), _data.begin() + size);
        return d;
    }
    void set_sample_window(unsigned size) { std::lock_guard<std::mutex> guard(_mutex); if (size % 2 != 0) size = size + 1; _window_size = size; }
    void set_enabled(bool v) { std::lock_guard<std::mutex> guard(_mutex); _enabled = v; }
    void flush() { std::lock_guard<std::mutex> guard(_mutex); _data.clear(); }
private:
    std::vector<gr_complex> _data;
    unsigned _window_size = 8096;
    bool _enabled = false;
    std::mutex _mutex;
};

// ---- batched demodulator: n_channels instances of one reference hier block on one B200
class gr_demod_b200 {
public:
    gr_demod_b200(int kind, int sps, int samp_rate, int carrier_freq, int filter_width, int flag,
                  int n_channels, long max_samples, int device)
        : _C(n_channels)
    {
        const int rc = qrl_rx_create(kind, sps, samp_rate, carrier_freq, filter_width, flag, n_channels, max_samples, device, &_h);
        if (rc != QRL_OK) throw std::runtime_error(std::string("qrl_rx_create: ") + qrl_last_error(nullptr));
        _nports = qrl_rx_num_ports(_h);
        for (int p = 0; p < _nports; p++) {
            void* d; long cap; int* cnt;
            qrl_rx_port_device(_h, p, &d, &cap, &cnt);
            _cap.push_back(cap);
            _buf.emplace_back(static_cast<size_t>(cap) * qrl_rx_port_itemsize(_h, p) * _C);
        }
        _counts.resize(_C);
    }
    ~gr_demod_b200() { qrl_rx_destroy(_h); }
    gr_demod_b200(const gr_demod_b200&) = delete;
    gr_demod_b200& operator=(const gr_demod_b200&) = delete;

    int n_channels() const { return _C; }
    int n_ports() const { return _nports; }
    // runtime setters of the analog blocks (gr_demod_nbfm.h:47-49, gr_demod_ssb.h:47-51, gr_demod_am.h:47-50, gr_demod_wbfm.h:47-48); like the
    // reference's they return nothing: a block without the setter ignores it (the shim's QRL_EINVAL stays readable through last_error())
    void set_squelch(int db) { qrl_rx_set_param(_h, -1, QRL_PARAM_SQUELCH_DB, db); }
    void set_filter_width(int w) { qrl_rx_set_param(_h, -1, QRL_PARAM_FILTER_WIDTH, w); }
    void set_ctcss(float v) { qrl_rx_set_param(_h, -1, QRL_PARAM_CTCSS, v); }
    void set_agc_attack(float v) { qrl_rx_set_param(_h, -1, QRL_PARAM_AGC_ATTACK, v); }
    void set_agc_decay(float v) { qrl_rx_set_param(_h, -1, QRL_PARAM_AGC_DECAY, v); }
    void set_gain(float v) { qrl_rx_set_param(_h, -1, QRL_PARAM_GAIN, v); }
    void set_carrier_offset(double hz, int channel = -1) { qrl_rx_set_param(_h, channel, QRL_PARAM_CARRIER_OFFSET_HZ, hz); }

    // one chunk of the [channels][T] gr_complex stream (host memory); returns T or WORK_DONE on a shim error
    int work(const gr_complex* iq, int T, long stride)
    {
        _fetched_mask = 0;
        if (qrl_rx_work(_h, reinterpret_cast<const float*>(iq), T, stride, 0) != QRL_OK) return WORK_DONE;
        return T;
    }
    // items the last work() produced on `port` for `channel`: pointer into an internal host buffer + count
    template <class T>
    const T* port(int port, int channel, int* n_items)
    {
        if (!(_fetched_mask & (1u << port))) {
            if (qrl_rx_read_port(_h, port, _buf[port].data(), _cap[port], _counts.data(), 0) != QRL_OK) { *n_items = 0; return nullptr; }
            _fetched_counts[port] = _counts;
            _fetched_mask |= 1u << port;
        }
        *n_items = _fetched_counts[port][channel];
        return reinterpret_cast<const T*>(_buf[port].data()) + static_cast<size_t>(channel) * _cap[port];
    }
    const char* last_error() const { return qrl_last_error(_h); }
    qrl_rx* handle() { return _h; }

private:
    qrl_rx* _h = nullptr;
    int _C = 0, _nports = 0;
    unsigned _fetched_mask = 0;
    std::vector<long> _cap;
    std::vector<std::vector<unsigned char>> _buf;
    std::vector<int> _counts;
    std::vector<int> _fetched_counts[4];
};
using gr_demod_b200_sptr = std::shared_ptr<gr_demod_b200>;

inline gr_demod_b200_sptr make_gr_demod_4fsk(int sps, int samp_rate, int carrier_freq, int filter_width, bool fm,
                                             int n_channels = 1, long max_samples = 1 << 20, int device = 0)
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_4FSK, sps, samp_rate, carrier_freq, filter_width, fm ? 1 : 0, n_channels, max_samples, device); }
inline gr_demod_b200_sptr make_gr_demod_qpsk(int sps, int samp_rate, int carrier_freq, int filter_width,
                                             int n_channels = 1, long max_samples = 1 << 20, int device = 0)
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_QPSK, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_samples, device); }
inline gr_demod_b200_sptr make_gr_demod_nbfm(int sps, int samp_rate, int carrier_freq, int filter_width,
                                             int n_channels = 1, long max_samples = 1 << 20, int device = 0)
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_NBFM, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_samples, device); }

inline gr_demod_b200_sptr make_gr_demod_bpsk(int sps, int samp_rate, int carrier_freq, int filter_width,
                                             int n_channels = 1, long max_samples = 1 << 20, int device = 0)
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_BPSK, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_samples, device); }
inline gr_demod_b200_sptr make_gr_demod_2fsk(int sps, int samp_rate, int carrier_freq, int filter_width, bool fm,
                                             int n_channels = 1, long max_samples = 1 << 20, int device = 0)
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_2FSK, sps, samp_rate, carrier_freq, filter_width, fm ? 1 : 0, n_channels, max_samples, device); }

inline gr_demod_b200_sptr make_gr_demod_ssb(int sps, int samp_rate, int carrier_freq, int filter_width, int sb,
                                            int n_channels = 1, long max_samples = 1 << 20, int device = 0)      // src/gr/gr_demod_ssb.h
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_SSB, sps, samp_rate, carrier_freq, filter_width, sb, n_channels, max_samples, device); }
inline gr_demod_b200_sptr make_gr_demod_am(int sps, int samp_rate, int carrier_freq, int filter_width,
                                           int n_channels = 1, long max_samples = 1 << 20, int device = 0)       // src/gr/gr_demod_am.h
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_AM, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_samples, device); }
inline gr_demod_b200_sptr make_gr_demod_gmsk(int sps, int samp_rate, int carrier_freq, int filter_width,
                                             int n_channels = 1, long max_samples = 1 << 20, int device = 0)     // src/gr/gr_demod_gmsk.h
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_GMSK, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_samples, device); }

inline gr_demod_b200_sptr make_gr_demod_wbfm(int sps, int samp_rate, int carrier_freq, int filter_width,
                                             int n_channels = 1, long max_samples = 1 << 20, int device = 0)     // src/gr/gr_demod_wbfm.h
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_WBFM, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_samples, device); }

inline gr_demod_b200_sptr make_gr_demod_m17(int sps = 125, int samp_rate = 1000000, int carrier_freq = 1700, int filter_width = 9000,
                                            int n_channels = 1, long max_samples = 1 << 20, int device = 0)      // src/gr/gr_demod_m17.h:41-42
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_M17, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_samples, device); }

inline gr_demod_b200_sptr make_gr_demod_dsss(int sps = 25, int samp_rate = 1000000, int carrier_freq = 1700, int filter_width = 150,
                                             int n_channels = 1, long max_samples = 1 << 20, int device = 0)     // instance gr_demod_base.cpp:218
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_DSSS, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_samples, device); }
inline gr_demod_b200_sptr make_gr_demod_dmr(int sps = 5, int samp_rate = 1000000,
                                            int n_channels = 1, long max_samples = 1 << 20, int device = 0)      // src/gr/gr_demod_dmr.h:42
{ return std::make_shared<gr_demod_b200>(QRL_DEMOD_DMR, sps, samp_rate, 0, 5000, 0, n_channels, max_samples, device); }

// ---- batched modulator
class gr_mod_b200 {
public:
    gr_mod_b200(int kind, int sps, int samp_rate, int carrier_freq, int filter_width, int flag, int n_channels, long max_items, int device)
        : _C(n_channels)
    {
        if (qrl_tx_create(kind, sps, samp_rate, carrier_freq, filter_width, flag, n_channels, max_items, device, &_h) != QRL_OK)
            throw std::runtime_error(std::string("qrl_tx_create: ") + qrl_last_error(nullptr));
    }
    ~gr_mod_b200() { qrl_tx_destroy(_h); }
    gr_mod_b200(const gr_mod_b200&) = delete;
    gr_mod_b200& operator=(const gr_mod_b200&) = delete;
    void set_bb_gain(float v) { qrl_tx_set_param(_h, -1, QRL_PARAM_BB_GAIN, v); }
    void set_filter_width(int fw) { qrl_tx_set_param(_h, -1, QRL_PARAM_FILTER_WIDTH, fw); }     // gr_mod_nbfm / _ssb / _am
    // gr_mod_dmr: the "zero_samples" tag gr_dmr_source attaches to a byte of the stream (gr_dmr_source.cpp:148)
    int zero_samples(int channel, long long byte_offset, long n_samples) { return qrl_tx_zero_samples(_h, channel, byte_offset, n_samples); }
    // what gr_byte_source::set_data hands over: [channels][n] frame bytes -> [channels][n_out] gr_complex at 1 Msps
    int work(const unsigned char* bytes, long n, long stride, std::vector<gr_complex>& out, long* n_out)
    {
        if (qrl_tx_work(_h, bytes, n, stride, 0) != QRL_OK) return WORK_DONE;
        float* d; long st, no;
        qrl_tx_out_device(_h, &d, &st, &no);
        out.resize(static_cast<size_t>(no) * _C);
        if (qrl_tx_read(_h, reinterpret_cast<float*>(out.data()), no, n_out, 0) != QRL_OK) return WORK_DONE;
        return static_cast<int>(*n_out);
    }
private:
    qrl_tx* _h = nullptr;
    int _C;
};
using gr_mod_b200_sptr = std::shared_ptr<gr_mod_b200>;
inline gr_mod_b200_sptr make_gr_mod_4fsk(int sps, int samp_rate, int carrier_freq, int filter_width, bool fm,
                                         int n_channels = 1, long max_items = 4096, int device = 0)
{ return std::make_shared<gr_mod_b200>(QRL_MOD_4FSK, sps, samp_rate, carrier_freq, filter_width, fm ? 1 : 0, n_channels, max_items, device); }
inline gr_mod_b200_sptr make_gr_mod_qpsk(int sps, int samp_rate, int carrier_freq, int filter_width,
                                         int n_channels = 1, long max_items = 4096, int device = 0)
{ return std::make_shared<gr_mod_b200>(QRL_MOD_QPSK, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_items, device); }

inline gr_mod_b200_sptr make_gr_mod_bpsk(int sps, int samp_rate, int carrier_freq, int filter_width,
                                         int n_channels = 1, long max_items = 4096, int device = 0)
{ return std::make_shared<gr_mod_b200>(QRL_MOD_BPSK, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_items, device); }
inline gr_mod_b200_sptr make_gr_mod_2fsk(int sps, int samp_rate, int carrier_freq, int filter_width, bool fm,
                                         int n_channels = 1, long max_items = 4096, int device = 0)
{ return std::make_shared<gr_mod_b200>(QRL_MOD_2FSK, sps, samp_rate, carrier_freq, filter_width, fm ? 1 : 0, n_channels, max_items, device); }

inline gr_mod_b200_sptr make_gr_mod_m17(int sps = 125, int samp_rate = 1000000, int carrier_freq = 1700, int filter_width = 9000,
                                        int n_channels = 1, long max_items = 4096, int device = 0)               // src/gr/gr_mod_m17.h:43-44
{ return std::make_shared<gr_mod_b200>(QRL_MOD_M17, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_items, device); }

inline gr_mod_b200_sptr make_gr_mod_am(int sps = 125, int samp_rate = 1000000, int carrier_freq = 1700, int filter_width = 5000,
                                       int n_channels = 1, long max_items = 4096, int device = 0)                 // instance gr_mod_base.cpp:167
{ return std::make_shared<gr_mod_b200>(QRL_MOD_AM, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_items, device); }
inline gr_mod_b200_sptr make_gr_mod_dsss(int sps = 25, int samp_rate = 1000000, int carrier_freq = 1700, int filter_width = 200,
                                         int n_channels = 1, long max_items = 8, int device = 0)                  // instance gr_mod_base.cpp:170
{ return std::make_shared<gr_mod_b200>(QRL_MOD_DSSS, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_items, device); }
inline gr_mod_b200_sptr make_gr_mod_dmr(int sps = 125, int samp_rate = 1000000, int carrier_freq = 1700, int filter_width = 5000,
                                        int n_channels = 1, long max_items = 4096, int device = 0)               // src/gr/gr_mod_dmr.h:37-38
{ return std::make_shared<gr_mod_b200>(QRL_MOD_DMR, sps, samp_rate, carrier_freq, filter_width, 0, n_channels, max_items, device); }

// ---- TX front end: what gr_mod_base connects between the modulator and the SDR sink (gr_mod_base.cpp:38,211-290):
// _rotator (set_carrier_offset, :799-805) and, at samp_rate >= 2 Msps, the xN _resampler.  1 Msps gr_complex in, samp_rate out,
// as gr_complex (QRL_TXFRONT_FC32) or interleaved int16 I/Q (QRL_TXFRONT_SC16, per component clamp(rint(x * sc16_scale))).
class tx_frontend_b200 {
public:
    tx_frontend_b200(int samp_rate, int n_channels = 1, long max_in = 1 << 20, int out_format = QRL_TXFRONT_FC32, float sc16_scale = 32767.0f, int device = 0)
        : _C(n_channels), _N(samp_rate / 1000000), _fmt(out_format)
    {
        if (qrl_txfront_create(samp_rate, n_channels, max_in, out_format, sc16_scale, device, &_h) != QRL_OK)
            throw std::runtime_error(std::string("qrl_txfront_create: ") + qrl_last_error(nullptr));
    }
    ~tx_frontend_b200() { qrl_txfront_destroy(_h); }
    tx_frontend_b200(const tx_frontend_b200&) = delete;
    tx_frontend_b200& operator=(const tx_frontend_b200&) = delete;
    int set_carrier_offset(double offset_hz, int channel = -1) { return qrl_txfront_set_carrier_offset(_h, channel, offset_hz); }
    int interpolation() const { return _N; }
    // host path: [channels][stride] gr_complex at 1 Msps -> [channels][N n] items of the output format in `out` (fc32: 2 floats,
    // sc16: 2 int16 per item); returns N n, or WORK_DONE on a shim error
    template <class T>
    int work(const gr_complex* in, long n, long stride, std::vector<T>& out)
    {
        static_assert(sizeof(T) == 8 || sizeof(T) == 4, "gr_complex or a pair of int16 per item");
        long n_out = 0;
        if ((sizeof(T) == 8) != (_fmt == QRL_TXFRONT_FC32)) return WORK_DONE;
        if (qrl_txfront_work(_h, reinterpret_cast<const float*>(in), n, stride, 0, &n_out) != QRL_OK) return WORK_DONE;
        out.resize(static_cast<size_t>(n_out) * _C);
        if (n_out > 0 && qrl_txfront_read(_h, out.data(), n_out) != QRL_OK) return WORK_DONE;
        return static_cast<int>(n_out);
    }
    // device path (e.g. the modulator's qrl_tx_out_device buffer): the output stays on the device, see out_device
    long work_device(const float* d_in, long n, long stride)
    {
        long n_out = 0;
        return qrl_txfront_work(_h, d_in, n, stride, 1, &n_out) == QRL_OK ? n_out : WORK_DONE;
    }
    int out_device(void** data, long* stride, long* n_out) { return qrl_txfront_out_device(_h, data, stride, n_out); }
private:
    qrl_txfront* _h = nullptr;
    int _C, _N, _fmt;
};

}  // namespace qrl_gr
