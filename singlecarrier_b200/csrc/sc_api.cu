// sc_api.cu -- host side of libsinglecarrier_b200.so: the modem bank handle and the C ABI.
//
// Host logic only: state ownership, the per-call launch sequence, slab/stream pipelining and
// host<->device staging.  All modem arithmetic runs in the sm_100a kernels; the two scalars the
// reference takes from glibc (cosf/sinf of the NCO step, qpsk.c:376,428) are evaluated here with
// the same libm, everything else (the phasor recurrences included) is done on the device.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <tuple>
#include <mutex>
#include <new>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "sc_kernels.h"
#include "sc_common.cuh"

namespace sc {
std::atomic<unsigned long long> g_launch_count{0};
}

// NVTX range for the lifetime of a scope (SURVEY section 5: ranges around K1..K4 and the copies; visible to
// ncu --nvtx / any NVTX consumer, a few ns when no tool is attached)
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

using namespace sc;

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

// A failed runtime call also sets the runtime's last error, which every launcher returns: clear it, so that a
// refused allocation does not fail the next launch on this thread.
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            cudaGetLastError();                                                                    \
            return fail(e_ == cudaErrorMemoryAllocation ? SC_ENOMEM : SC_ECUDA, "%s:%d %s: %s",    \
                        __FILE__, __LINE__, #call, cudaGetErrorString(e_));                        \
        }                                                                                          \
    } while (0)

// Device resources owned by the handle or a cache entry, released with their device current.
template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;                                 // elements
    DevBuf() = default;
    DevBuf(DevBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr, o.cap = 0; }
    DevBuf &operator=(DevBuf &&o) noexcept { std::swap(p, o.p), std::swap(cap, o.cap); return *this; }
    ~DevBuf() { if (p) cudaFree(p); }
    operator T *() const { return p; }
    // room for n elements; the contents are discarded when n exceeds the capacity
    cudaError_t reserve(size_t n) {
        if (cap >= n) return cudaSuccess;
        cudaError_t e = p ? cudaFree(p) : cudaSuccess;
        p = nullptr, cap = 0;
        if (e == cudaSuccess && (e = cudaMalloc(&p, n * sizeof(T))) == cudaSuccess) cap = n;
        return e;
    }
};

template <typename H, cudaError_t (*Destroy)(H)>
struct Owned {
    H h = nullptr;
    Owned() = default;
    Owned(Owned &&o) noexcept : h(o.h) { o.h = nullptr; }
    Owned &operator=(Owned &&) = delete;
    ~Owned() { if (h) Destroy(h); }
    operator H() const { return h; }
};
// create() does nothing when the object exists, so lazily built scratch that failed part-way is completed later
struct Stream : Owned<cudaStream_t, cudaStreamDestroy> {
    cudaError_t create() { return h ? cudaSuccess : cudaStreamCreateWithFlags(&h, cudaStreamNonBlocking); }
};
struct Event : Owned<cudaEvent_t, cudaEventDestroy> {
    cudaError_t create(unsigned flags = cudaEventDisableTiming) { return h ? cudaSuccess : cudaEventCreateWithFlags(&h, flags); }
};

static const int N_PIPE = 3;        // internal CUDA streams (slabs in flight)
static const int TAB_HEAD = 2;      // phasor-table frames generated before the first call starts
static const int OV_RING = 4;       // overlapped chains: calls whose hand-over buffers are live at once
static const int TAB_CHUNK = 4;     // ... the rest in pieces of this many frames, each with its own event
static const int H2D_FIRST = 80, H2D_COUNT = 1624;   // sample columns of a frame the RX chain can read (host path)
static const int SYM_FLOATS = 2 * NDATA;                // one record of sc_rx_frames_soft_*: 31 complex floats
static const size_t SYM_BYTES = SYM_FLOATS * sizeof(float);

struct sc_modem {
    int device = 0;
    int64_t n = 0;                  // streams
    int64_t n_pad = 0;              // rounded up to 128 for the tiled window layout
    uint32_t flags = 0;
    float foffset = 0.f;
    bool wide = false, debug_eq = false;
    uint32_t call = 0;              // qpsk_rx_frame() calls made so far
    uint16_t lfsr_rx = 0x4A80;      // RXMemory, src/scramble.c:42, seeded at qpsk.c:434
    float2 rx_rect, tx_rect;

    // per-stream device state (SURVEY appendix B)
    DevBuf<int> timing[2];                  // rx_timing at entry of call n in timing[n & 1]
    DevBuf<int> timing_cold;                // FINE_TIMING_OFFSET for every stream (source of resets)
    DevBuf<float2> win;                     // tracker windows, tiles of 32 streams x WIN_ROWS
    DevBuf<int> max_index;
    DevBuf<float> max_value;
    // frames before the batch that the receiver reads: call-1 (the front-end), call-2 (packet mode), call-3 (ACQ)
    int hist_depth = 1;                     // H
    DevBuf<int16_t> hist;                   // frames call-H .. call-1, [H][n][1880]

    // shared tables
    DevBuf<float2> rx_phase;                // fbb_rx_phase (device scalar)
    DevBuf<float2> mix_table;               // phasors of frames call-H .., this batch's from table_slot(m, 1)
    DevBuf<float2> unit_phase;              // constant 1+0i: the cold phasor of a transmission (qpsk.c:375)
    float *state_dbg = nullptr;             // drop-in shim: full tracker state after the last call, [n][48] (not owned)
    std::vector<uint64_t> kw;               // keystream words of the batch being queued

    Stream pipe[N_PIPE];
    Event ev_start, ev_done[N_PIPE];
    // the phasor table is generated by one thread (a sequential float recurrence): the first TAB_HEAD
    // frames on pipe[0], the rest on tab_stream while the first calls already run
    Stream tab_stream;
    Event ev_tab1, ev_tab2;
    int tab_split = 0;                      // table slots 1..tab_split are ready once pipe[0]'s part is done
    std::vector<Event> ev_tabc;             // piece c (slots tab_split + 1 + TAB_CHUNK c ..) is ready at ev_tabc[c]

    // staging for the host entry point
    DevBuf<int16_t> stage_in[N_PIPE];
    DevBuf<sc_frame_result> stage_res[N_PIPE];
    DevBuf<float> stage_eq[N_PIPE];
    DevBuf<float> stage_sym[N_PIPE];

    // packet mode (SC_FLAG_PACKET, extension): the rx_timing snapshots and per-pipe scratch for the packet pass
    bool packet = false;
    bool packet_dd = false;                 // SC_FLAG_PACKET_DD: packets decoded by the decision-directed equalizer
    bool packet_acq = false;                // SC_FLAG_PACKET_ACQ: packets found by acquisition on the samples
    DevBuf<int4> acq_info[N_PIPE];          // SC_FLAG_PACKET_ACQ: per-pipe grid start, rho and nu0 of the listed packets
    DevBuf<int> pk_t_before[N_PIPE], pk_t_at[N_PIPE];         // [slab] rx_timing at entry of calls call0-1 / call0
    DevBuf<int2> pk_list[N_PIPE];
    DevBuf<int> pk_count[N_PIPE];
    DevBuf<float2> pk_sym[N_PIPE];
    Stream pk_stream[N_PIPE];               // the packet passes run beside the call chain, not inside it
    Event pk_ev_go[N_PIPE], pk_ev_done[N_PIPE];
    bool pk_ready = false;
    DevBuf<unsigned long long> pk_n_host_dev;                  // packet counter of the host entry point
    DevBuf<sc_packet_result> pk_stage;
    DevBuf<float2> pk_sym_stage;            // packet symbols of the host entry point, PK_DATA per record
    PacketKey pk_key;

    // A batch call that failed after its first launch leaves some streams advanced and others not:
    // the handle refuses further work (SC_ESTATE) until sc_reset() or sc_state_import().
    bool poisoned = false;
    bool in_flight = false;
    uint64_t h2d_bytes = 0, d2h_bytes = 0;  // bytes queued by sc_rx_frames_host since sc_create (sc_transfer_bytes)

    // options / per-kernel profiling (bench.py's roofline leg)
    int h2d_mode = SC_H2D_COLUMNS;
    const void *search_a_table = nullptr;   // A fragments of the tensor-core search proposer (per device, not owned)
    bool fe_search_mma = false;             // SC_OPT_FE_SEARCH: any tensor-core mode (the serial chain is used)
    bool fe_search_umma = false;            //   ... SC_FE_SEARCH_TCGEN05: frontend_umma_kernel (sc_frontend_umma.cu)
    const void *search_umma_master = nullptr;   // its A-operand master (per device, not owned)
    int slab_parts = 0;                     // 0 = default (2 x N_PIPE slabs)
    bool profile = false;
    int tracker = SC_TRACKER_AUTO;

    // overlapped chains (SC_OPT_OVERLAP): tall windows, search results, the tracker hand-over and rx_timing in rings of
    // OV_RING calls; two chain streams (the pipe and a partner) and a stream for the data steps per pipe; event rings
    int overlap = SC_OVERLAP_AUTO;
    DevBuf<float2> ov_win[OV_RING];
    DevBuf<int> ov_max_index[OV_RING];
    DevBuf<float> ov_max_value[OV_RING];
    DevBuf<float> ov_state[OV_RING];
    DevBuf<int> ov_timing[OV_RING];
    Stream ov_stream[N_PIPE], ov_data[N_PIPE][2];
    Event ov_ev_fe[N_PIPE][OV_RING], ov_ev_train[N_PIPE][OV_RING], ov_ev_data[N_PIPE][OV_RING];
    Event ov_ev_first[N_PIPE], ov_join[N_PIPE][3];
    bool ov_ready = false;
    std::vector<Event> ev_fe, ev_tk;        // (start, stop) pairs
};

// ---- scrambler keystream (integer LFSR, src/scramble.c:57-69) ----------------------------------
static inline unsigned lfsr_step(uint16_t &m) {
    unsigned out = ((m >> 1) ^ m) & 1u;
    m = (uint16_t) ((m >> 1) | (out << 14));
    return out;
}
static uint64_t keystream_next_word(uint16_t &m) {
    uint64_t w = 0;
    for (int j = 0; j < SC_BITS_PER_CALL; j++) w |= (uint64_t) lfsr_step(m) << j;
    return w;
}

// The 15-bit LFSR x^15 + x^14 + 1 is maximal length: its state sequence has period 32767, so the register
// before call n is the seed stepped (62 n mod 32767) times.
static uint16_t lfsr_at_call(uint32_t call_index) {
    uint16_t m = 0x4A80;
    const uint32_t steps = (uint32_t) (((uint64_t) call_index * SC_BITS_PER_CALL) % 32767u);
    for (uint32_t k = 0; k < steps; k++) lfsr_step(m);
    return m;
}

extern "C" uint64_t sc_keystream_word(uint32_t call_index) {
    uint16_t m = lfsr_at_call(call_index);
    return keystream_next_word(m);
}

// cmplx(TAU * f / FS), headers/qpsk_internal.h:60,67: TAU is a double because glibc's M_PI is
static float2 nco_rect(float freq_hz) {
    double tau = 2.0f * M_PI;
    float x = (float) (tau * freq_hz / 8000.0f);
    return make_float2(cosf(x), sinf(x));
}

extern "C" const char *sc_last_error(void) { return g_err; }
extern "C" const char *sc_version(void) { return "singlecarrier_b200 0.2 (sm_100a)"; }
extern "C" uint64_t sc_launch_count(void) { return g_launch_count; }
extern "C" int sc_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}
extern "C" int64_t sc_n_streams(const sc_modem *m) { return m ? m->n : 0; }
extern "C" uint32_t sc_call_index(const sc_modem *m) { return m ? m->call : 0; }

static int modem_cold(sc_modem *m) {
    CU(cudaSetDevice(m->device));
    const int64_t np = m->n_pad;
    // rx_timing = FINE_TIMING_OFFSET (qpsk.c:53); windows of calls 0 and 1 are the zero-initialised
    // decimated_frame (qpsk.c:42), whose search gives max_index 0 / max_value 0.0
    // (hist needs no reset: it is only read by a batch that continues a previous one, which saved it)
    CU(cudaMemcpyAsync(m->timing[0], m->timing_cold, np * sizeof(int), cudaMemcpyDeviceToDevice, m->pipe[0]));
    CU(cudaMemcpyAsync(m->timing[1], m->timing_cold, np * sizeof(int), cudaMemcpyDeviceToDevice, m->pipe[0]));
    CU(cudaMemsetAsync(m->win, 0, (size_t) (np / 32) * WIN_ROWS * 32 * sizeof(float2), m->pipe[0]));
    CU(cudaMemsetAsync(m->max_index, 0, np * sizeof(int), m->pipe[0]));
    CU(cudaMemsetAsync(m->max_value, 0, np * sizeof(float), m->pipe[0]));
    const float2 one = make_float2(1.0f, 0.0f);                         // cmplx(0.0f), qpsk.c:427
    CU(cudaMemcpyAsync(m->rx_phase, &one, sizeof one, cudaMemcpyHostToDevice, m->pipe[0]));
    CU(cudaStreamSynchronize(m->pipe[0]));
    m->call = 0;
    m->lfsr_rx = 0x4A80;
    m->poisoned = m->in_flight = false;
    return SC_OK;
}

static int search_table(int device, const void **out);
static int search_umma_master(int device, const void **out);

extern "C" int sc_create(sc_modem **out, int device, int64_t n_streams, uint32_t flags, float foffset_hz) {
    if (!out || n_streams <= 0 || n_streams > (int64_t) 1 << 30) return fail(SC_EINVAL, "sc_create: bad arguments");
    *out = nullptr;
    if ((flags & SC_FLAG_PACKET_DD) && !(flags & SC_FLAG_PACKET))
        return fail(SC_EINVAL, "sc_create: SC_FLAG_PACKET_DD needs SC_FLAG_PACKET");
    if ((flags & SC_FLAG_PACKET_ACQ) && !((flags & SC_FLAG_PACKET) && (flags & SC_FLAG_PACKET_DD)))
        return fail(SC_EINVAL, "sc_create: SC_FLAG_PACKET_ACQ needs SC_FLAG_PACKET and SC_FLAG_PACKET_DD");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(SC_ECUDA, "sc_create: no CUDA device (this library has no CPU path)");
    }
    if (device < 0 || device >= ndev) return fail(SC_EINVAL, "sc_create: device %d of %d", device, ndev);
    sc_modem *m = new (std::nothrow) sc_modem();
    if (!m) return fail(SC_ENOMEM, "sc_create: host allocation");
    m->device = device;
    m->n = n_streams;
    m->n_pad = (n_streams + 127) / 128 * 128;
    m->flags = flags;
    m->wide = (flags & SC_FLAG_WIDE) != 0;
    m->debug_eq = (flags & SC_FLAG_DEBUG_EQ) != 0;
    m->packet = (flags & SC_FLAG_PACKET) != 0;
    m->packet_dd = (flags & SC_FLAG_PACKET_DD) != 0;
    m->packet_acq = (flags & SC_FLAG_PACKET_ACQ) != 0;
    m->hist_depth = 1 + m->packet + m->packet_acq;
    {
        uint16_t r = 0x4A80;                                             // scramble_init per packet
        for (int f = 0; f < 8; f++) m->pk_key.k[f] = keystream_next_word(r);
    }
    m->foffset = foffset_hz;
    if (const char *e = getenv("SC_SLAB_PARTS")) m->slab_parts = atoi(e);
    if (const char *e = getenv("SC_OVERLAP")) m->overlap = std::max(0, std::min(atoi(e), (int) SC_OVERLAP_ON));
    m->rx_rect = nco_rect(-1100.0f + foffset_hz);                       // qpsk.c:428
    m->tx_rect = nco_rect(1100.0f);                                     // qpsk.c:376
    int rc = SC_OK;
    auto body = [&]() -> int {
        CU(cudaSetDevice(device));
        const int64_t np = m->n_pad;
        CU(m->timing[0].reserve(np));
        CU(m->timing[1].reserve(np));
        CU(m->timing_cold.reserve(np));
        {
            std::vector<int> t(np, 3);
            CU(cudaMemcpy(m->timing_cold, t.data(), np * sizeof(int), cudaMemcpyHostToDevice));
        }
        CU(m->win.reserve((size_t) (np / 32) * WIN_ROWS * 32));
        CU(m->max_index.reserve(np));
        CU(m->max_value.reserve(np));
        const size_t hist_len = (size_t) m->hist_depth * m->n * FRAME;
        CU(m->hist.reserve(hist_len));
        CU(cudaMemset(m->hist, 0, hist_len * sizeof(int16_t)));
        CU(m->rx_phase.reserve(1));
        if (m->packet) CU(m->pk_n_host_dev.reserve(1));
        CU(m->unit_phase.reserve(1));
        {
            const float2 one = make_float2(1.0f, 0.0f);
            CU(cudaMemcpy(m->unit_phase, &one, sizeof one, cudaMemcpyHostToDevice));
        }
        if (const char *e = getenv("SC_FE_SEARCH")) {
            m->fe_search_umma = strcmp(e, "tcgen05") == 0;
            m->fe_search_mma = m->fe_search_umma || strcmp(e, "mma") == 0;
        }
        if (const char *e = getenv("SC_H2D_MODE")) m->h2d_mode = std::max(0, std::min(atoi(e), (int) SC_H2D_COLUMNS_3D));
        for (int i = 0; i < N_PIPE; i++) {
            CU(m->pipe[i].create());
            CU(m->ev_done[i].create());
        }
        CU(m->ev_start.create());
        CU(m->tab_stream.create());
        CU(m->ev_tab1.create());
        CU(m->ev_tab2.create());
        return modem_cold(m);
    };
    rc = body();
    if (rc != SC_OK) {
        sc_destroy(m);
        return rc;
    }
    *out = m;
    return SC_OK;
}

// The device-wide synchronisation also covers the caller's streams, on which a device-path batch queues work that
// touches handle memory.
extern "C" void sc_destroy(sc_modem *m) {
    if (!m) return;
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    delete m;
    cudaGetLastError();
}

// Wait for everything queued on the handle's own streams (a batch that failed part-way may have left the overlapped
// chains' side streams unjoined: every successful batch joins them into the pipes).
static int drain(sc_modem *m) {
    CU(cudaSetDevice(m->device));
    for (int i = 0; i < N_PIPE; i++) CU(cudaStreamSynchronize(m->pipe[i]));
    CU(cudaStreamSynchronize(m->tab_stream));
    if (m->ov_ready)
        for (int i = 0; i < N_PIPE; i++) {
            CU(cudaStreamSynchronize(m->ov_stream[i]));
            CU(cudaStreamSynchronize(m->ov_data[i][0]));
            CU(cudaStreamSynchronize(m->ov_data[i][1]));
        }
    return SC_OK;
}

extern "C" int sc_reset(sc_modem *m) {
    if (!m) return fail(SC_EINVAL, "sc_reset: null handle");
    int rc = drain(m);
    return rc != SC_OK ? rc : modem_cold(m);
}

// SC_OV_TRACE=1: time stamps (CUDA events) after every launch of the overlapped chains, printed per batch -- a
// development aid (the events themselves cost a few microseconds per call)
struct OvTrace {
    bool on = getenv("SC_OV_TRACE") != nullptr;
    std::vector<std::tuple<const char *, uint32_t, int, cudaEvent_t>> ev;
    void mark(const char *what, uint32_t n, int q, cudaStream_t st) {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        ev.emplace_back(what, n, q, e);
    }
    void dump() {
        if (!on || ev.empty()) return;
        cudaDeviceSynchronize();
        for (auto &t : ev) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, std::get<3>(ev[0]), std::get<3>(t));
            fprintf(stderr, "ovtrace %-8s call %3u stream %d  %9.1f us\n", std::get<0>(t), std::get<1>(t), std::get<2>(t), ms * 1e3);
        }
        for (auto &t : ev) cudaEventDestroy(std::get<3>(t));
        ev.clear();
    }
};
static OvTrace g_trace;

// The phasor table of batch slot `slot`: slot 0 is frame call-1, slots 1.. this batch's frames; the history's older
// frames precede slot 0, so the table of frame call-1-k is table_slot(m, -k) for k < H.
static float2 *table_slot(const sc_modem *m, int slot) {
    return m->mix_table + (size_t) (m->hist_depth - 1 + slot) * FRAME;
}

// Make sure the mix table can hold the H history slots + n_frames frames and generate this batch's phasors
// (calls call .. call+n_frames-1 into slots 1..n_frames) on stream st.
static int prepare_tables(sc_modem *m, int n_frames, cudaStream_t st) {
    const size_t hist_bytes = (size_t) m->hist_depth * FRAME * sizeof(float2);
    if (m->mix_table.cap < (size_t) (m->hist_depth + n_frames) * FRAME) {     // a larger table, keeping the history
        DevBuf<float2> nt;
        CU(nt.reserve((size_t) (m->hist_depth + n_frames) * FRAME));
        if (m->mix_table) {
            CU(cudaMemcpyAsync(nt, m->mix_table, hist_bytes, cudaMemcpyDeviceToDevice, st));
            CU(cudaStreamSynchronize(st));
        } else {
            CU(cudaMemsetAsync(nt, 0, hist_bytes, st));
        }
        m->mix_table = std::move(nt);                                   // the old table goes with nt
    }
    // stored pre-multiplied by 1/16384: phasor*((float)in/16384) == (phasor/16384)*(float)in exactly.
    // Head on st (the calls wait for it); the rest on tab_stream in pieces, so that a call waits only for the piece
    // that holds its frame: one thread generates a frame in ~12 us, a small bank consumes one in ~40 us, and a single
    // tail kernel (~0.5 ms for 42 frames) would stall the chain right after the head.
    const int head = std::min(n_frames, TAB_HEAD);
    CU(launch_nco_table(m->rx_phase, m->rx_rect, NCO_RX, 0, head, 1.0f / 16384.0f, table_slot(m, 1), st));
    CU(cudaEventRecord(m->ev_tab1, st));
    g_trace.mark("tabhead", (uint32_t) head, 0, st);
    CU(cudaStreamWaitEvent(m->tab_stream, m->ev_tab1, 0));
    for (int f = head, c = 0; f < n_frames; f += TAB_CHUNK, c++) {
        if ((int) m->ev_tabc.size() <= c) m->ev_tabc.emplace_back();
        CU(m->ev_tabc[c].create());
        CU(launch_nco_table(m->rx_phase, m->rx_rect, NCO_RX, 0, std::min(TAB_CHUNK, n_frames - f), 1.0f / 16384.0f,
                            table_slot(m, f + 1), m->tab_stream));
        CU(cudaEventRecord(m->ev_tabc[c], m->tab_stream));
        g_trace.mark("table", (uint32_t) (f + TAB_CHUNK), 9, m->tab_stream);
    }
    CU(cudaEventRecord(m->ev_tab2, m->tab_stream));
    m->tab_split = head;
    return SC_OK;
}

// Order stream st after the generation of table slot `slot` (waited = the latest piece st already waits for, -1 at first)
static int table_wait(sc_modem *m, cudaStream_t st, int slot, int &waited) {
    if (slot <= m->tab_split) return SC_OK;
    const int c = (slot - m->tab_split - 1) / TAB_CHUNK;
    if (c > waited) {
        CU(cudaStreamWaitEvent(st, m->ev_tabc[c], 0));
        waited = c;
    }
    return SC_OK;
}

static cudaError_t prof_mark(std::vector<Event> &v, cudaStream_t st) {
    Event e;
    cudaError_t rc = e.create(cudaEventDefault);
    if (rc != cudaSuccess) return rc;
    v.push_back(std::move(e));
    return cudaEventRecord(v.back(), st);
}

struct PacketSink {
    sc_packet_result *packets = nullptr;    // device
    int64_t capacity = 0;
    unsigned long long *n_packets = nullptr;   // device, accumulated into
    float2 *symbols = nullptr;              // device or nullptr: PK_DATA equalizer outputs per record slot
};
static const int PK_CAP = 65536;            // listed packets per pass; slabs are at most this many streams in packet mode

// scratch of the packet pass, once per handle
static int packet_scratch(sc_modem *m) {
    if (m->pk_ready) return SC_OK;
    for (int i = 0; i < N_PIPE; i++) {
        CU(m->pk_t_before[i].reserve(PK_CAP));
        CU(m->pk_t_at[i].reserve(PK_CAP));
        CU(m->pk_list[i].reserve(PK_CAP));
        CU(m->pk_count[i].reserve(1));
        CU(m->pk_sym[i].reserve((size_t) (PK_CAP / 32) * PK_SYMS * 32));
        if (m->packet_acq) CU(m->acq_info[i].reserve(PK_CAP));
        CU(m->pk_stream[i].create());
        CU(m->pk_ev_go[i].create());
        CU(m->pk_ev_done[i].create());
    }
    m->pk_ready = true;
    return SC_OK;
}

// scratch of the overlapped chains, once per handle
static int overlap_scratch(sc_modem *m) {
    if (m->ov_ready) return SC_OK;
    const int64_t np = m->n_pad;
    for (int q = 0; q < OV_RING; q++) {
        CU(m->ov_win[q].reserve((size_t) (np / 32) * WIN_ROWS_OV * 32));
        CU(m->ov_max_index[q].reserve(np));
        CU(m->ov_max_value[q].reserve(np));
        CU(m->ov_state[q].reserve((size_t) np * TRK_STATE_WORDS));
        CU(m->ov_timing[q].reserve(np));
    }
    for (int i = 0; i < N_PIPE; i++) {
        CU(m->ov_stream[i].create());
        for (int q = 0; q < 2; q++) CU(m->ov_data[i][q].create());
        CU(m->ov_ev_first[i].create());
        for (int q = 0; q < 3; q++) CU(m->ov_join[i][q].create());
        for (int q = 0; q < OV_RING; q++) {
            CU(m->ov_ev_fe[i][q].create());
            CU(m->ov_ev_train[i][q].create());
            CU(m->ov_ev_data[i][q].create());
        }
    }
    m->ov_ready = true;
    return SC_OK;
}

// One slab of streams [s0, s0+ns) over one block of frames, queued on st.  `in` points at stream s0's first sample of
// the block's first frame, `results`/`eq_dbg`/`sym` at stream s0's record of the block's first call.  The block begins
// slot0 frames into the batch: its first call is m->call + slot0, with keystream word m->kw[slot0], and filters the
// frame whose phasors are in table slot slot0.
struct Slab {
    cudaStream_t st;
    int pipe;
    int64_t s0;
    int ns;
    const int16_t *in;
    int64_t stride;
    int n_frames;
    int slot0;
    sc_frame_result *results;
    int64_t result_stride;
    float *eq_dbg, *sym;
    const PacketSink *pk;
};

// slot k of stream s0's sample history: frame c-H+k, c the first call of the block that reads it
static int16_t *hist_slot(const sc_modem *m, int k, int64_t s0) {
    return m->hist + ((size_t) k * m->n + s0) * FRAME;
}

// the frame fe(n) filters, for call n = call0 + j: frame j-1 of the block, or the last one of the previous block
static const int16_t *fe_frame(const sc_modem *m, const Slab &s, int j, int64_t &fstride) {
    fstride = j >= 1 ? s.stride : FRAME;
    return j >= 1 ? s.in + (size_t) (j - 1) * FRAME : hist_slot(m, m->hist_depth - 1, s.s0);
}

// The block's last H frames become the history of the next block: slot k takes block frame nf-H+k, or, when the block
// is shorter than that, the frame the previous block saved in slot nf+k (above k, so read before it is overwritten).
static int store_history(sc_modem *m, const Slab &s) {
    const size_t pitch = FRAME * sizeof(int16_t);
    for (int k = 0; k < m->hist_depth; k++) {
        const int f = s.n_frames - m->hist_depth + k;
        if (f >= 0)
            CU(cudaMemcpy2DAsync(hist_slot(m, k, s.s0), pitch, s.in + (size_t) f * FRAME, (size_t) s.stride * sizeof(int16_t),
                                 pitch, (size_t) s.ns, cudaMemcpyDeviceToDevice, s.st));
        else
            CU(cudaMemcpyAsync(hist_slot(m, k, s.s0), hist_slot(m, s.n_frames + k, s.s0), (size_t) s.ns * pitch,
                               cudaMemcpyDeviceToDevice, s.st));
    }
    return SC_OK;
}

// The call loop of one slab as two chains (include/singlecarrier_b200.h, SC_OPT_OVERLAP).  With
//   fe(n):    frame n-1, rx_timing T_n                     -> window(n-1), max_index      [the window call n+1 reads]
//   train(n): window(n-2)                                  -> tracker after the preamble, matches
//   data(n):  that tracker, window(n-2), T_n               -> result(n)
//   T_{n+1} = matches(n) > 98 ? max_index(n) + 128 : T_n                                  [qpsk.c:196,219]
// the only path from call to call is rx_timing, and it does not pass through the 31 data steps:
//   T_n -> fe(n) -> train(n+1) -> T_{n+2}, given T_{n+1} from the other parity's chain.
// fe(n) evaluates T_n itself from what train(n-1) and fe(n-1) left.  So the calls form two chains
//   C[p]:  ... fe(n) -> train(n+1) -> fe(n+2) -> train(n+3) ...        (n + 1 of parity p)
// on two streams, fe(n) waiting for fe(n-1) of the other chain, and the data steps run beside them on two more
// streams (a data kernel, one thread per stream among the chains' warps, takes about as long as a call).  What call k consumes (window, max_index, tracker, T_k) lives in slot k % OV_RING; slot k is rewritten by
// fe(k+3), which therefore waits for data(k).
// The batch's first call runs the uncut tracker on the window the previous batch left (m->win, the serial layout) and
// the last call's front-end writes that layout again, so the state between batches does not depend on the mode.
static int run_slab_overlapped(sc_modem *m, const Slab &s, bool coop) {
    int rc = overlap_scratch(m);
    if (rc != SC_OK) return rc;
    const cudaStream_t st = s.st;
    const int pipe = s.pipe, ns = s.ns, n_frames = s.n_frames, slot0 = s.slot0;
    const int64_t s0 = s.s0;
    const uint32_t call0 = m->call + (uint32_t) slot0;
    const uint64_t *kw = m->kw.data() + slot0;
    const float2 *mix0 = table_slot(m, slot0);
    cudaStream_t C[2];
    const Stream *Dn = m->ov_data[pipe];
    C[call0 & 1] = st;
    C[(call0 & 1) ^ 1] = m->ov_stream[pipe];
    CU(cudaEventRecord(m->ov_join[pipe][0], st));                   // the other streams start where st stands
    CU(cudaStreamWaitEvent(m->ov_stream[pipe], m->ov_join[pipe][0], 0));
    CU(cudaStreamWaitEvent(Dn[0], m->ov_join[pipe][0], 0));
    CU(cudaStreamWaitEvent(Dn[1], m->ov_join[pipe][0], 0));
    int tab_waited[2] = {-1, -1}, tab_waited_d = -1;
    OvTrace &trace = g_trace;
    trace.mark("start", call0, call0 & 1, st);
    const size_t tile_ov = (size_t) (s0 / 32) * WIN_ROWS_OV * 32;
    float2 *win = m->win + (size_t) (s0 / 32) * WIN_ROWS * 32;
    const uint32_t last = call0 + (uint32_t) n_frames - 1;
    auto state_of = [&](uint32_t k) { return m->ov_state[k % OV_RING] + (coop ? (size_t) s0 * TRK_STATE_WORDS : (size_t) s0); };
    // T_k derived from what call k-1 left in its slot (k - 1 > call0: call0 itself runs the uncut tracker, which stores)
    auto timing_src = [&](uint32_t k, int *store) {
        TimingSrc ts;
        if (k >= call0 + 2) {
            ts.matches = state_of(k - 1) + (coop ? 55 : 35 * m->n_pad);
            ts.mstride = coop ? TRK_STATE_WORDS : 1;
            ts.max_index = m->ov_max_index[(k - 1) % OV_RING] + s0;
            ts.timing_prev = m->ov_timing[(k - 1) % OV_RING] + s0;
            ts.timing_out = store;
        }
        return ts;
    };

    // ---- the first call, and the window the second one reads
    {
        const int p = (int) (call0 & 1), q = p ^ 1;
        NvtxRange range("sc:track_kernel");
        CU(launch_track(false, win, m->max_index + s0, m->max_value + s0, m->timing[p] + s0,
                        m->ov_timing[(call0 + 1) % OV_RING] + s0, s.results, s.result_stride, nullptr, nullptr, call0, kw[0],
                        ns, C[p], coop, s.sym));
        trace.mark("track", call0, p, C[p]);
        CU(cudaEventRecord(m->ov_ev_first[pipe], C[p]));
        const uint32_t k = call0 + 1;                               // consumer of fe(call0)
        if (call0 >= 1) {
            int64_t fstride;
            const int16_t *frame = fe_frame(m, s, 0, fstride);
            if ((rc = table_wait(m, C[q], slot0, tab_waited[q])) != SC_OK) return rc;
            NvtxRange range2("sc:frontend_kernel");
            CU(launch_frontend(m->wide, frame, fstride, mix0, m->timing[p] + s0, nullptr, m->ov_win[k % OV_RING] + tile_ov,
                               m->ov_max_index[k % OV_RING] + s0, m->ov_max_value[k % OV_RING] + s0, ns, C[q], nullptr));
            trace.mark("fe_ov", call0, q, C[q]);
        } else {                                                    // the zero-initialised decimated_frame, qpsk.c:42
            CU(cudaMemsetAsync(m->ov_win[k % OV_RING] + tile_ov, 0, (size_t) ((ns + 31) / 32) * WIN_ROWS_OV * 32 * sizeof(float2), C[q]));
            CU(cudaMemsetAsync(m->ov_max_index[k % OV_RING] + s0, 0, (size_t) ns * sizeof(int), C[q]));
            CU(cudaMemsetAsync(m->ov_max_value[k % OV_RING] + s0, 0, (size_t) ns * sizeof(float), C[q]));
        }
        CU(cudaEventRecord(m->ov_ev_fe[pipe][call0 % OV_RING], C[q]));
    }
    for (uint32_t n = call0 + 1; n <= last; n++) {
        const int j = (int) (n - call0), p = (int) (n & 1), q = p ^ 1, r = (int) (n % OV_RING);
        {
            NvtxRange range("sc:track_train");
            CU(launch_track_train(m->ov_win[r] + tile_ov, state_of(n), m->n_pad, ns, C[p], coop));
            trace.mark("train", n, p, C[p]);
            CU(cudaEventRecord(m->ov_ev_train[pipe][r], C[p]));
        }
        if (n < last) {
            // fe(n) on the other chain, behind train(n-1) (or the first call): T_n from slot n-1, or as the first call stored it
            const uint32_t k = n + 1;
            int64_t fstride;
            const int16_t *frame = fe_frame(m, s, j, fstride);
            CU(cudaStreamWaitEvent(C[q], m->ov_ev_fe[pipe][(n - 1) % OV_RING], 0));       // T_{n-1}
            if (n >= call0 + 4) CU(cudaStreamWaitEvent(C[q], m->ov_ev_data[pipe][(n - 3) % OV_RING], 0));   // slot k is free
            if ((rc = table_wait(m, C[q], slot0 + j, tab_waited[q])) != SC_OK) return rc;
            const TimingSrc ts = timing_src(n, m->ov_timing[r] + s0);
            NvtxRange range("sc:frontend_kernel");
            CU(launch_frontend(m->wide, frame, fstride, mix0 + (size_t) j * FRAME, m->ov_timing[r] + s0, nullptr,
                               m->ov_win[k % OV_RING] + tile_ov, m->ov_max_index[k % OV_RING] + s0,
                               m->ov_max_value[k % OV_RING] + s0, ns, C[q], nullptr, &ts));
            trace.mark("fe_ov", n, q, C[q]);
            CU(cudaEventRecord(m->ov_ev_fe[pipe][r], C[q]));
        }
        {
            // data(n) beside the chains; the last call also leaves T_n and T_{n+1} where the next batch looks for them
            cudaStream_t D = Dn[p];
            CU(cudaStreamWaitEvent(D, m->ov_ev_train[pipe][r], 0));
            if (n < last) CU(cudaStreamWaitEvent(D, m->ov_ev_fe[pipe][r], 0));             // T_n
            else if (n == call0 + 1) CU(cudaStreamWaitEvent(D, m->ov_ev_first[pipe], 0));
            else {                                                                         // T_n from slot n-1
                CU(cudaStreamWaitEvent(D, m->ov_ev_fe[pipe][(n - 1) % OV_RING], 0));
                CU(cudaStreamWaitEvent(D, m->ov_ev_train[pipe][(n - 1) % OV_RING], 0));
            }
            const TimingSrc ts = n < last ? TimingSrc() : timing_src(n, nullptr);
            NvtxRange range("sc:track_data");
            CU(launch_track_data(m->ov_win[r] + tile_ov, state_of(n), m->n_pad, m->ov_max_index[r] + s0, m->ov_max_value[r] + s0,
                                 m->ov_timing[r] + s0, n == last ? m->timing[(n + 1) & 1] + s0 : nullptr, s.results + j,
                                 s.result_stride, n, kw[j], ns, D, coop, &ts, n == last ? m->timing[n & 1] + s0 : nullptr,
                                 s.sym ? s.sym + (size_t) j * SYM_FLOATS : nullptr));
            trace.mark("data", n, 2 + p, D);
            CU(cudaEventRecord(m->ov_ev_data[pipe][r], D));
        }
    }
    {
        // the last call's front-end in the serial layout: window, max_index and both rx_timing arrays for the next batch
        cudaStream_t D = Dn[last & 1];
        int64_t fstride;
        const int16_t *frame = fe_frame(m, s, n_frames - 1, fstride);
        if ((rc = table_wait(m, D, slot0 + n_frames - 1, tab_waited_d)) != SC_OK) return rc;
        NvtxRange range("sc:frontend_kernel");
        CU(launch_frontend(m->wide, frame, fstride, mix0 + (size_t) (n_frames - 1) * FRAME, m->timing[last & 1] + s0,
                           m->timing[(last + 1) & 1] + s0, win, m->max_index + s0, m->max_value + s0, ns, D, nullptr));
        trace.mark("fe_std", last, 2, D);
    }
    CU(cudaEventRecord(m->ov_join[pipe][0], m->ov_stream[pipe]));
    CU(cudaEventRecord(m->ov_join[pipe][1], Dn[0]));
    CU(cudaEventRecord(m->ov_join[pipe][2], Dn[1]));
    for (int q = 0; q < 3; q++) CU(cudaStreamWaitEvent(st, m->ov_join[pipe][q], 0));
    trace.dump();
    return SC_OK;
}

// The call loop of one slab; afterwards the block's last frames are saved for the block that follows.
static int run_slab(sc_modem *m, const Slab &s) {
    const cudaStream_t st = s.st;
    const int pipe = s.pipe, ns = s.ns, n_frames = s.n_frames, slot0 = s.slot0;
    const int64_t s0 = s.s0;
    const PacketSink *pk = s.pk;
    float *eq_dbg = s.eq_dbg;
    const uint32_t call0 = m->call + (uint32_t) slot0;
    const uint64_t *kw = m->kw.data() + slot0;
    const float2 *mix0 = table_slot(m, slot0);
    float2 *win = m->win + (size_t) (s0 / 32) * WIN_ROWS * 32;
    int tab_waited = -1;
    PacketSrc psrc;
    int pk_chunk = 0, pk_done = 0;
    if (pk) {
        if (ns > PK_CAP) return fail(SC_ESTATE, "packet mode: slab larger than the packet scratch");
        // rx_timing at entry of calls call0-1 and call0 (the ping-pong arrays are overwritten as the calls run)
        CU(cudaMemcpyAsync(m->pk_t_before[pipe], m->timing[(call0 + 1) & 1] + s0, (size_t) ns * sizeof(int), cudaMemcpyDeviceToDevice, st));
        CU(cudaMemcpyAsync(m->pk_t_at[pipe], m->timing[call0 & 1] + s0, (size_t) ns * sizeof(int), cudaMemcpyDeviceToDevice, st));
        psrc.results = s.results;
        psrc.result_stride = s.result_stride;
        psrc.in = s.in;
        psrc.stride = s.stride;
        psrc.hist = hist_slot(m, m->hist_depth - 1, s0);
        psrc.hist_pitch = m->n * FRAME;
        psrc.mix0 = mix0;
        psrc.timing_before_call0 = m->pk_t_before[pipe];
        psrc.timing_at_call0 = m->pk_t_at[pipe];
        psrc.call0 = call0;
        psrc.stream0 = (int) s0;
        psrc.wide = m->wide;
        pk_chunk = std::max(1, PK_CAP / ns);                // every call of a pass may be valid
    }
    const bool tracker_coop = m->tracker == SC_TRACKER_COOP || (m->tracker == SC_TRACKER_AUTO && ns <= SC_TRACKER_COOP_MAX);
    const bool plain = !pk && !m->packet && !m->profile && !m->fe_search_mma && !eq_dbg && !m->state_dbg;
    if (plain && n_frames >= 2 && (m->overlap == SC_OVERLAP_ON || (m->overlap == SC_OVERLAP_AUTO && m->n <= SC_OVERLAP_MAX))) {
        int rc = run_slab_overlapped(m, s, tracker_coop);
        return rc != SC_OK ? rc : store_history(m, s);
    }
    for (int j = 0; j < n_frames; j++) {
        const uint32_t n = call0 + (uint32_t) j;
        int *tc = m->timing[n & 1] + s0, *tn = m->timing[(n + 1) & 1] + s0;
        if (m->profile) CU(prof_mark(m->ev_tk, st));
        {
            NvtxRange range("sc:track_kernel");
            CU(launch_track(m->debug_eq && eq_dbg != nullptr, win, m->max_index + s0, m->max_value + s0, tc, tn,
                            s.results + j, s.result_stride, eq_dbg ? eq_dbg + (size_t) j * 10 : nullptr,
                            m->state_dbg ? m->state_dbg + (size_t) s0 * TRACK_STATE_FLOATS : nullptr, n, kw[j], ns, st, tracker_coop,
                            s.sym ? s.sym + (size_t) j * SYM_FLOATS : nullptr));
        }
        if (m->profile) CU(prof_mark(m->ev_tk, st));
        if (n >= 1) {
            int64_t fstride;
            const int16_t *frame = fe_frame(m, s, j, fstride);
            int rcw = table_wait(m, st, slot0 + j, tab_waited);
            if (rcw != SC_OK) return rcw;
            if (m->profile) CU(prof_mark(m->ev_fe, st));
            {
                NvtxRange range("sc:frontend_kernel");
                if (m->fe_search_umma && frontend_umma_eligible(frame, fstride))
                    CU(launch_frontend_umma(m->wide, frame, fstride, mix0 + (size_t) j * FRAME, tc, tn, win, m->max_index + s0,
                                            m->max_value + s0, ns, st, m->search_umma_master));
                else
                    CU(launch_frontend(m->wide, frame, fstride, mix0 + (size_t) j * FRAME, tc, tn, win, m->max_index + s0,
                                       m->max_value + s0, ns, st,
                                       m->fe_search_mma && !m->fe_search_umma ? m->search_a_table : nullptr));
            }
            if (m->profile) CU(prof_mark(m->ev_fe, st));
        }
        if (pk && (j + 1 - pk_done == pk_chunk || j + 1 == n_frames)) {
            // The pass only READS what the calls up to j produced (results, frames, tables), so it runs on a side
            // stream beside the call chain: its 376-step serial kernel would otherwise sit on every call's critical path.
            NvtxRange range("sc:packet_pass");
            // the pass reads the tables of frames up to call j-1, acquisition up to call j
            int rcw = table_wait(m, st, slot0 + j + (m->packet_acq ? 1 : 0), tab_waited);
            if (rcw != SC_OK) return rcw;
            CU(cudaEventRecord(m->pk_ev_go[pipe], st));
            CU(cudaStreamWaitEvent(m->pk_stream[pipe], m->pk_ev_go[pipe], 0));
            const AcqScratch acq = {m->acq_info[pipe].p};
            CU(launch_packet_pass(psrc, ns, pk_done, j + 1, PK_CAP, m->pk_list[pipe], m->pk_count[pipe], m->pk_sym[pipe],
                                  m->pk_key, pk->packets, pk->capacity, pk->n_packets, pk->symbols, m->packet_dd,
                                  m->packet_acq ? &acq : nullptr, m->pk_stream[pipe]));
            pk_done = j + 1;
        }
    }
    if (pk) {                                                       // join before the frames / history are reused
        CU(cudaEventRecord(m->pk_ev_done[pipe], m->pk_stream[pipe]));
        CU(cudaStreamWaitEvent(st, m->pk_ev_done[pipe], 0));
    }
    return store_history(m, s);
}

static int64_t pick_slab(int64_t n, int64_t lo, int64_t parts) {
    int64_t s = (n + parts - 1) / parts;
    s = std::max<int64_t>(s, lo);
    s = (s + 127) / 128 * 128;
    return s;
}

// One batch of any of the eight RX entry points (include/singlecarrier_b200.h): device or host buffers, the optional
// equalizer outputs (eq_dbg of debug banks, sym of the soft forms) and, for the packet entry points, the records.
struct RxBatch {
    const char *who;
    const int16_t *in;
    int64_t stream_stride;
    int n_frames;
    sc_frame_result *results;
    int64_t result_stride;
    float *eq_dbg = nullptr, *sym = nullptr;
    bool host = false;
    cudaStream_t stream = nullptr;          // the caller's stream (device buffers)
    bool packet_mode = false;
    sc_packet_result *packets = nullptr;
    int64_t capacity = 0;
    uint64_t *n_packets = nullptr;
    float *packet_symbols = nullptr;
};

// Generate the batch's phasor tables on pipe[0] and order the other pipes after them.  The batch is in flight from
// here: a failure from now on may leave some streams advanced and others not.
static int start_tables(sc_modem *m, int n_frames) {
    m->in_flight = true;
    int rc = prepare_tables(m, n_frames, m->pipe[0]);
    if (rc != SC_OK) return rc;
    CU(cudaEventRecord(m->ev_start, m->pipe[0]));
    for (int i = 1; i < N_PIPE; i++) CU(cudaStreamWaitEvent(m->pipe[i], m->ev_start, 0));
    return SC_OK;
}

// The tables of the batch's last H frames become the next batch's history: history slot k (frame call-H+k) takes the
// table n_frames slots above it, from this batch or, when the batch is shorter than H-k, from a higher history slot.
static int rotate_tables(sc_modem *m, int n_frames, cudaStream_t st) {
    for (int k = 0; k < m->hist_depth; k++)
        CU(cudaMemcpyAsync(m->mix_table + (size_t) k * FRAME, m->mix_table + (size_t) (n_frames + k) * FRAME,
                           FRAME * sizeof(float2), cudaMemcpyDeviceToDevice, st));
    return SC_OK;
}

static int rx_dev_body(sc_modem *m, const RxBatch &b, const PacketSink *pk) {
    CU(cudaSetDevice(m->device));
    // order after the caller's stream, build the tables once, fan out over the pipe streams
    CU(cudaEventRecord(m->ev_start, b.stream));
    CU(cudaStreamWaitEvent(m->pipe[0], m->ev_start, 0));
    int rc = start_tables(m, b.n_frames);
    if (rc != SC_OK) return rc;

    // default: two slabs, each on its own stream, so one slab's tail waves overlap the other's kernels
    int64_t slab = pick_slab(m->n, m->slab_parts > 0 ? 128 : 8192, m->slab_parts > 0 ? m->slab_parts : 2);
    if (pk) slab = std::min<int64_t>(slab, PK_CAP);
    int k = 0;
    for (int64_t s0 = 0; s0 < m->n; s0 += slab, k++) {
        const Slab s = {m->pipe[k % N_PIPE], k % N_PIPE, s0, (int) std::min<int64_t>(slab, m->n - s0),
                        b.in + (size_t) s0 * b.stream_stride, b.stream_stride, b.n_frames, 0,
                        b.results + (size_t) s0 * b.result_stride, b.result_stride,
                        b.eq_dbg ? b.eq_dbg + (size_t) s0 * b.result_stride * 10 : nullptr,
                        b.sym ? b.sym + (size_t) s0 * b.result_stride * SYM_FLOATS : nullptr, pk};
        if ((rc = run_slab(m, s)) != SC_OK) return rc;
    }
    for (int i = 0; i < N_PIPE; i++) {
        CU(cudaEventRecord(m->ev_done[i], m->pipe[i]));
        CU(cudaStreamWaitEvent(b.stream, m->ev_done[i], 0));
    }
    CU(cudaStreamWaitEvent(b.stream, m->ev_tab2, 0));
    if ((rc = rotate_tables(m, b.n_frames, b.stream)) != SC_OK) return rc;
    CU(cudaEventRecord(m->ev_start, b.stream));
    for (int i = 0; i < N_PIPE; i++) CU(cudaStreamWaitEvent(m->pipe[i], m->ev_start, 0));
    return SC_OK;
}

// Host -> device copy of frames [f0, f0 + nf) of streams [s0, s0 + ns) into a staging buffer laid out
// [ns][nf * 1880].  Only samples [80, 1704) of a frame can influence any output: rx_timing is 128..255 after
// the first call, so the front-end reads samples rx_timing-48 .. rx_timing+1445 (+ pair slack) and nothing
// else (DESIGN.md section 3); the staging columns that are not copied are never read.
//   SC_H2D_COLUMNS     one 2-D copy per frame of the block: ns rows of 3,248 bytes (86 % of the bytes)
//   SC_H2D_COLUMNS_3D  the same bytes as ONE 3-D copy per block (needs stream_stride % 1880 == 0)
//   SC_H2D_ROWS        one 2-D copy per block: ns rows from sample 80 of the first frame to sample 1703 of
//                      the last (nf * 3760 - 512 bytes each)
//   SC_H2D_FULL        whole frames: one 2-D copy per block, or one plain 1-D copy when the block covers every
//                      frame of contiguous streams
static int h2d_block(sc_modem *m, int mode, int16_t *stage, const int16_t *in, int64_t stream_stride, int64_t s0,
                     int ns, int f0, int nf, cudaStream_t st) {
    NvtxRange range("sc:h2d");
    const size_t spitch = (size_t) stream_stride * sizeof(int16_t);
    const size_t dpitch = (size_t) nf * FRAME * sizeof(int16_t);
    const int16_t *src = in + (size_t) s0 * stream_stride + (size_t) f0 * FRAME;
    if (mode == SC_H2D_COLUMNS_3D && stream_stride % FRAME != 0) mode = SC_H2D_COLUMNS;
    switch (mode) {
        case SC_H2D_FULL: m->h2d_bytes += dpitch * (size_t) ns; break;
        case SC_H2D_ROWS: m->h2d_bytes += (dpitch - (size_t) (FRAME - H2D_COUNT) * sizeof(int16_t)) * (size_t) ns; break;
        default: m->h2d_bytes += (size_t) H2D_COUNT * sizeof(int16_t) * (size_t) nf * (size_t) ns;
    }
    switch (mode) {
        case SC_H2D_FULL:
            if (spitch == dpitch)
                CU(cudaMemcpyAsync(stage, src, dpitch * (size_t) ns, cudaMemcpyHostToDevice, st));
            else
                CU(cudaMemcpy2DAsync(stage, dpitch, src, spitch, dpitch, (size_t) ns, cudaMemcpyHostToDevice, st));
            break;
        case SC_H2D_ROWS:
            CU(cudaMemcpy2DAsync(stage + H2D_FIRST, dpitch, src + H2D_FIRST, spitch,
                                 dpitch - (size_t) (FRAME - H2D_COUNT) * sizeof(int16_t), (size_t) ns,
                                 cudaMemcpyHostToDevice, st));
            break;
        case SC_H2D_COLUMNS_3D: {
            cudaMemcpy3DParms p;
            memset(&p, 0, sizeof p);
            const size_t fpitch = FRAME * sizeof(int16_t);
            p.srcPtr = make_cudaPitchedPtr((void *) (src + H2D_FIRST), fpitch, fpitch, (size_t) (stream_stride / FRAME));
            p.dstPtr = make_cudaPitchedPtr((void *) (stage + H2D_FIRST), fpitch, fpitch, (size_t) nf);
            p.extent = make_cudaExtent((size_t) H2D_COUNT * sizeof(int16_t), (size_t) nf, (size_t) ns);
            p.kind = cudaMemcpyHostToDevice;
            CU(cudaMemcpy3DAsync(&p, st));
            break;
        }
        default:
            for (int j = 0; j < nf; j++)
                CU(cudaMemcpy2DAsync(stage + (size_t) j * FRAME + H2D_FIRST, dpitch, src + (size_t) j * FRAME + H2D_FIRST,
                                     spitch, (size_t) H2D_COUNT * sizeof(int16_t), (size_t) ns, cudaMemcpyHostToDevice, st));
    }
    return SC_OK;
}

extern "C" int sc_transfer_bytes(const sc_modem *m, uint64_t out[2]) {
    if (!m || !out) return fail(SC_EINVAL, "sc_transfer_bytes: bad arguments");
    out[0] = m->h2d_bytes;
    out[1] = m->d2h_bytes;
    return SC_OK;
}

static const size_t STAGE_BYTES = (size_t) 768 << 20;     // staging per pipe stream

static int rx_host_body(sc_modem *m, const RxBatch &b, const PacketSink *pk) {
    CU(cudaSetDevice(m->device));
    // slabs of streams x blocks of frames; slab k always runs on pipe k % N_PIPE, so its blocks
    // stay in order and the staging buffer of that pipe is reused safely (stream order)
    const int n_frames = b.n_frames;
    const size_t frame_bytes = FRAME * sizeof(int16_t);
    int64_t slab;
    int fblk;
    // packet mode reads whole frames (the 248 data symbols reach past the columns the ordinary chain needs)
    const int h2d_mode = m->packet ? (int) SC_H2D_FULL : m->h2d_mode;
    const bool contiguous = h2d_mode == SC_H2D_FULL && b.stream_stride == (int64_t) n_frames * FRAME &&
                            (size_t) n_frames * frame_bytes * 128 <= STAGE_BYTES;
    if (contiguous && m->slab_parts <= 0) {
        // all frames of a slab in one plain copy: as many streams as the staging buffer holds
        fblk = n_frames;
        slab = (int64_t) (STAGE_BYTES / ((size_t) n_frames * frame_bytes)) / 128 * 128;
        slab = std::min<int64_t>(slab, pick_slab(m->n, 128, 2 * N_PIPE));
        if (pk) slab = std::min<int64_t>(slab, PK_CAP);
    } else {
        slab = pick_slab(m->n, m->slab_parts > 0 ? 128 : 4096, m->slab_parts > 0 ? m->slab_parts : 2 * N_PIPE);
        if (pk) slab = std::min<int64_t>(slab, PK_CAP);
        fblk = (int) std::max<int64_t>(1, std::min<int64_t>(n_frames, (int64_t) STAGE_BYTES / (slab * (int64_t) frame_bytes)));
    }
    const size_t records = (size_t) slab * fblk;
    for (int p = 0; p < N_PIPE; p++) {
        CU(m->stage_in[p].reserve(records * FRAME));
        CU(m->stage_res[p].reserve(records));
        if (b.eq_dbg) CU(m->stage_eq[p].reserve(records * 10));
        if (b.sym) CU(m->stage_sym[p].reserve(records * SYM_FLOATS));
    }
    int rc = start_tables(m, n_frames);
    if (rc != SC_OK) return rc;

    for (int f0 = 0; f0 < n_frames; f0 += fblk) {
        const int nf = std::min(fblk, n_frames - f0);
        int k = 0;
        for (int64_t s0 = 0; s0 < m->n; s0 += slab, k++) {
            const int p = k % N_PIPE;
            cudaStream_t st = m->pipe[p];
            const int ns = (int) std::min<int64_t>(slab, m->n - s0);
            if ((rc = h2d_block(m, h2d_mode, m->stage_in[p], b.in, b.stream_stride, s0, ns, f0, nf, st)) != SC_OK) return rc;
            const Slab s = {st, p, s0, ns, m->stage_in[p], (int64_t) nf * FRAME, nf, f0, m->stage_res[p], nf,
                            b.eq_dbg ? m->stage_eq[p].p : nullptr, b.sym ? m->stage_sym[p].p : nullptr, pk};
            if ((rc = run_slab(m, s)) != SC_OK) return rc;
            NvtxRange range("sc:d2h");
            m->d2h_bytes += (size_t) nf * sizeof(sc_frame_result) * (size_t) ns + (b.eq_dbg ? (size_t) nf * 10 * sizeof(float) * (size_t) ns : 0) +
                            (b.sym ? (size_t) nf * SYM_BYTES * (size_t) ns : 0);
            CU(cudaMemcpy2DAsync(b.results + (size_t) s0 * b.result_stride + f0, (size_t) b.result_stride * sizeof(sc_frame_result),
                                 m->stage_res[p], (size_t) nf * sizeof(sc_frame_result),
                                 (size_t) nf * sizeof(sc_frame_result), (size_t) ns, cudaMemcpyDeviceToHost, st));
            if (b.eq_dbg)
                CU(cudaMemcpy2DAsync(b.eq_dbg + ((size_t) s0 * b.result_stride + f0) * 10, (size_t) b.result_stride * 10 * sizeof(float),
                                     m->stage_eq[p], (size_t) nf * 10 * sizeof(float), (size_t) nf * 10 * sizeof(float),
                                     (size_t) ns, cudaMemcpyDeviceToHost, st));
            if (b.sym)
                CU(cudaMemcpy2DAsync(b.sym + ((size_t) s0 * b.result_stride + f0) * SYM_FLOATS, (size_t) b.result_stride * SYM_BYTES,
                                     m->stage_sym[p], (size_t) nf * SYM_BYTES, (size_t) nf * SYM_BYTES, (size_t) ns,
                                     cudaMemcpyDeviceToHost, st));
        }
    }
    for (int i = 0; i < N_PIPE; i++) CU(cudaStreamSynchronize(m->pipe[i]));
    CU(cudaStreamSynchronize(m->tab_stream));
    if ((rc = rotate_tables(m, n_frames, m->pipe[0])) != SC_OK) return rc;
    CU(cudaStreamSynchronize(m->pipe[0]));
    return SC_OK;
}

// Checks, the batch's keystream words and the packet sink, then the device or host body.  The words are drawn from a
// COPY of the descrambler register, which is committed together with the call index only when the whole batch has
// been queued (a failing call must not leave RXMemory ahead of m->call).
static int rx_batch(sc_modem *m, const RxBatch &b) {
    const char *who = b.who;
    if (b.packet_mode) {
        if (!m || !b.packets || b.capacity < 0 || !b.n_packets) return fail(SC_EINVAL, "%s: bad arguments", who);
        if (!m->packet) return fail(SC_EINVAL, "%s: the bank was not created with SC_FLAG_PACKET", who);
        int rc = packet_scratch(m);
        if (rc != SC_OK) return rc;
        if (b.host) *b.n_packets = 0;
    }
    if (!m || !b.in || !b.results || b.n_frames < 0) return fail(SC_EINVAL, "%s: bad arguments", who);
    if (m->poisoned) return fail(SC_ESTATE, "%s: an earlier batch failed part-way; call sc_reset() first", who);
    if (b.n_frames == 0) return SC_OK;
    if (b.stream_stride < (int64_t) b.n_frames * FRAME || b.result_stride < b.n_frames)
        return fail(SC_EINVAL, "%s: stride smaller than the batch", who);
    if (b.eq_dbg && !m->debug_eq) return fail(SC_EINVAL, "%s: eq_dbg needs SC_FLAG_DEBUG_EQ", who);
    if (m->fe_search_mma) {                 // per batch, not per handle: sc_release_caches() may have freed the table
        int rc = m->fe_search_umma ? search_umma_master(m->device, &m->search_umma_master)
                                   : search_table(m->device, &m->search_a_table);
        if (rc != SC_OK) return rc;
    }
    uint16_t lfsr = m->lfsr_rx;
    m->kw.resize(b.n_frames);
    for (int j = 0; j < b.n_frames; j++) m->kw[j] = keystream_next_word(lfsr);
    NvtxRange range(who);

    PacketSink sink;
    if (b.packet_mode && b.host) {          // the records are staged on the device and read back below
        CU(cudaSetDevice(m->device));
        CU(m->pk_stage.reserve((size_t) b.capacity));
        if (b.packet_symbols) CU(m->pk_sym_stage.reserve((size_t) b.capacity * PK_DATA));
        CU(cudaMemset(m->pk_n_host_dev, 0, sizeof(unsigned long long)));
        sink = {m->pk_stage, b.capacity, m->pk_n_host_dev, b.packet_symbols ? m->pk_sym_stage.p : nullptr};
    } else if (b.packet_mode) {
        sink = {b.packets, b.capacity, (unsigned long long *) b.n_packets, reinterpret_cast<float2 *>(b.packet_symbols)};
    }
    const PacketSink *pk = b.packet_mode ? &sink : nullptr;
    int rc = b.host ? rx_host_body(m, b, pk) : rx_dev_body(m, b, pk);
    if (rc == SC_OK && b.packet_mode && b.host) {
        unsigned long long n = 0;
        cudaError_t e = cudaMemcpy(&n, m->pk_n_host_dev, sizeof n, cudaMemcpyDeviceToHost);
        const size_t kept = (size_t) std::min<unsigned long long>(n, (unsigned long long) b.capacity);
        if (e == cudaSuccess && n > 0)
            e = cudaMemcpy(b.packets, m->pk_stage, kept * sizeof(sc_packet_result), cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && n > 0 && b.packet_symbols)
            e = cudaMemcpy(b.packet_symbols, m->pk_sym_stage, kept * PK_DATA * sizeof(float2), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) {
            cudaGetLastError();
            rc = fail(SC_ECUDA, "%s: %s", who, cudaGetErrorString(e));
        }
        *b.n_packets = n;
    }
    if (rc != SC_OK) {
        if (m->in_flight) m->poisoned = true;      // something was launched: per-stream state is inconsistent
        m->in_flight = false;
        return rc;
    }
    m->in_flight = false;
    m->lfsr_rx = lfsr;
    m->call += (uint32_t) b.n_frames;
    return SC_OK;
}

extern "C" int sc_rx_frames_dev(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                                sc_frame_result *results, int64_t result_stride, float *eq_dbg, void *stream) {
    RxBatch b = {"sc_rx_frames_dev", in, stream_stride, n_frames, results, result_stride};
    b.eq_dbg = eq_dbg;
    b.stream = (cudaStream_t) stream;
    return rx_batch(m, b);
}

extern "C" int sc_rx_frames_host(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                                 sc_frame_result *results, int64_t result_stride, float *eq_dbg) {
    RxBatch b = {"sc_rx_frames_host", in, stream_stride, n_frames, results, result_stride};
    b.eq_dbg = eq_dbg;
    b.host = true;
    return rx_batch(m, b);
}

// The same calls with the equalizer outputs of the data steps (include/singlecarrier_b200.h).  Nothing else changes:
// the soft kernels are the plain ones with one extra store per step, on the same schedules.
extern "C" int sc_rx_frames_soft_dev(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                                     sc_frame_result *results, int64_t result_stride, float *symbols, void *stream) {
    if (!symbols) return fail(SC_EINVAL, "sc_rx_frames_soft_dev: symbols is NULL");
    if (((uintptr_t) symbols & 7) != 0) return fail(SC_EINVAL, "sc_rx_frames_soft_dev: symbols not 8-byte aligned");
    RxBatch b = {"sc_rx_frames_soft_dev", in, stream_stride, n_frames, results, result_stride};
    b.sym = symbols;
    b.stream = (cudaStream_t) stream;
    return rx_batch(m, b);
}

extern "C" int sc_rx_frames_soft_host(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                                      sc_frame_result *results, int64_t result_stride, float *symbols) {
    if (!symbols) return fail(SC_EINVAL, "sc_rx_frames_soft_host: symbols is NULL");
    RxBatch b = {"sc_rx_frames_soft_host", in, stream_stride, n_frames, results, result_stride};
    b.sym = symbols;
    b.host = true;
    return rx_batch(m, b);
}

// The packet entry points and their soft forms.  symbols (per call) and packet_symbols are nullptr for the plain ones.
static RxBatch packet_batch(const char *who, const int16_t *in, int64_t stream_stride, int n_frames,
                            sc_frame_result *results, int64_t result_stride, float *symbols, sc_packet_result *packets,
                            int64_t capacity, uint64_t *n_packets, float *packet_symbols) {
    RxBatch b = {who, in, stream_stride, n_frames, results, result_stride};
    b.sym = symbols;
    b.packet_mode = true;
    b.packets = packets;
    b.capacity = capacity;
    b.n_packets = n_packets;
    b.packet_symbols = packet_symbols;
    return b;
}

extern "C" int sc_rx_packets_dev(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                                 sc_frame_result *results, int64_t result_stride, sc_packet_result *packets,
                                 int64_t capacity, uint64_t *n_packets, void *stream) {
    RxBatch b = packet_batch("sc_rx_packets_dev", in, stream_stride, n_frames, results, result_stride, nullptr, packets,
                             capacity, n_packets, nullptr);
    b.stream = (cudaStream_t) stream;
    return rx_batch(m, b);
}

extern "C" int sc_rx_packets_host(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                                  sc_frame_result *results, int64_t result_stride, sc_packet_result *packets,
                                  int64_t capacity, uint64_t *n_packets) {
    RxBatch b = packet_batch("sc_rx_packets_host", in, stream_stride, n_frames, results, result_stride, nullptr, packets,
                             capacity, n_packets, nullptr);
    b.host = true;
    return rx_batch(m, b);
}

// Packet mode with the equalizer outputs (include/singlecarrier_b200.h): the 248 of every packet record, and, when
// symbols is not NULL, the 31 of every call.  Records, results and state are those of sc_rx_packets_*.
extern "C" int sc_rx_packets_soft_dev(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                                      sc_frame_result *results, int64_t result_stride, float *symbols,
                                      sc_packet_result *packets, int64_t capacity, uint64_t *n_packets,
                                      float *packet_symbols, void *stream) {
    if (!packet_symbols) return fail(SC_EINVAL, "sc_rx_packets_soft_dev: packet_symbols is NULL");
    if (((uintptr_t) packet_symbols & 7) != 0)
        return fail(SC_EINVAL, "sc_rx_packets_soft_dev: packet_symbols not 8-byte aligned");
    if (((uintptr_t) symbols & 7) != 0) return fail(SC_EINVAL, "sc_rx_packets_soft_dev: symbols not 8-byte aligned");
    RxBatch b = packet_batch("sc_rx_packets_soft_dev", in, stream_stride, n_frames, results, result_stride, symbols,
                             packets, capacity, n_packets, packet_symbols);
    b.stream = (cudaStream_t) stream;
    return rx_batch(m, b);
}

extern "C" int sc_rx_packets_soft_host(sc_modem *m, const int16_t *in, int64_t stream_stride, int n_frames,
                                       sc_frame_result *results, int64_t result_stride, float *symbols,
                                       sc_packet_result *packets, int64_t capacity, uint64_t *n_packets,
                                       float *packet_symbols) {
    if (!packet_symbols) return fail(SC_EINVAL, "sc_rx_packets_soft_host: packet_symbols is NULL");
    RxBatch b = packet_batch("sc_rx_packets_soft_host", in, stream_stride, n_frames, results, result_stride, symbols,
                             packets, capacity, n_packets, packet_symbols);
    b.host = true;
    return rx_batch(m, b);
}

extern "C" uint64_t sc_packet_keystream_word(int frame) {
    if (frame < 0 || frame >= 8) return 0;
    uint16_t r = 0x4A80;                                                 // scramble_init per packet
    uint64_t w = 0;
    for (int f = 0; f <= frame; f++) w = keystream_next_word(r);
    return w;
}

extern "C" void sc_unpack_bits(const sc_frame_result *results, int64_t n_records, uint8_t *rows) {
    for (int64_t k = 0; k < n_records; k++) {
        if (!results[k].valid) continue;
        const uint64_t w = results[k].bits;
        uint8_t *row = rows + k * SC_BITS_PER_CALL;
        for (int j = 0; j < SC_BITS_PER_CALL; j++) row[j] = (uint8_t) ((w >> j) & 1u);
    }
}

// stream-ordered device scratch that is released on every return path
template <typename T>
struct AsyncBuf {
    T *p = nullptr;
    cudaStream_t st;
    explicit AsyncBuf(cudaStream_t s) : st(s) {}
    AsyncBuf(const AsyncBuf &) = delete;
    AsyncBuf &operator=(const AsyncBuf &) = delete;
    ~AsyncBuf() { if (p) cudaFreeAsync(p, st); }
    cudaError_t alloc(size_t n) { return cudaMallocAsync((void **) &p, std::max<size_t>(n, 1) * sizeof(T), st); }
};

extern "C" int sc_nco_table_host(sc_modem *m, int tx, uint32_t first_call, int n_calls, float *out) {
    if (!m || !out || n_calls <= 0) return fail(SC_EINVAL, "sc_nco_table_host: bad arguments");
    CU(cudaSetDevice(m->device));
    // The phasor is a float recurrence: frames before first_call have to be stepped through, but only a
    // bounded scratch of them is ever materialised.
    const int CHUNK = 64;
    const int segs_per_call = tx ? 9 : 1;               // TX "call" = one packet: 640 + 8 x 155 samples
    const int pattern = tx ? NCO_TX_PACKET : NCO_RX;
    const float2 rect = tx ? m->tx_rect : m->rx_rect;
    cudaStream_t st = 0;
    AsyncBuf<float2> d_ph(st), d_out(st);
    CU(d_ph.alloc(1));
    CU(d_out.alloc((size_t) std::max(std::min<int64_t>(first_call, CHUNK), (int64_t) n_calls) * FRAME));
    CU(cudaMemcpyAsync(d_ph.p, m->unit_phase, sizeof(float2), cudaMemcpyDeviceToDevice, st));
    for (uint32_t c = 0; c < first_call; c += CHUNK) {
        const int k = (int) std::min<uint32_t>(CHUNK, first_call - c);
        CU(launch_nco_table(d_ph.p, rect, pattern, 0, k * segs_per_call, 1.0f, d_out.p, st));
    }
    CU(launch_nco_table(d_ph.p, rect, pattern, 0, n_calls * segs_per_call, 1.0f, d_out.p, st));
    CU(cudaMemcpyAsync(out, d_out.p, (size_t) n_calls * FRAME * sizeof(float2), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return SC_OK;
}

// ---- accessors used by the TX / stage translation units ----------------------------------------
namespace sc {
int modem_device(const sc_modem *m) { return m->device; }
int64_t modem_n(const sc_modem *m) { return m->n; }
bool modem_wide(const sc_modem *m) { return m->wide; }
float2 modem_tx_rect(const sc_modem *m) { return m->tx_rect; }
int api_fail(int code, const char *msg) { return fail(code, "%s", msg); }
// drop-in shim (sc_legacy_dev.cu): the reference's qpsk_rx_frame() and scramble()/data_eq() share RXMemory
// (src/scramble.c:42, src/equalizer.c:87) and leave the Kalman globals behind (src/kalman.c:19-35)
uint16_t modem_lfsr_rx(const sc_modem *m) { return m->lfsr_rx; }
void modem_set_lfsr_rx(sc_modem *m, uint16_t v) { m->lfsr_rx = v; }
void modem_set_state_dbg(sc_modem *m, float *p) { m->state_dbg = p; }
}  // namespace sc

// ---- TX ---------------------------------------------------------------------------------------
static int tx_common(sc_modem *m, const uint8_t *bits, uint8_t *bits_out, uint64_t seed, int n_packets,
                     int gap_samples, const int32_t *lead_in, const sc_channel *ch, int16_t *out,
                     int64_t stream_stride, int64_t samples_per_stream, void *stream) {
    if (!m || !out || n_packets < 0 || gap_samples < 0 || samples_per_stream < 0 || stream_stride < samples_per_stream)
        return fail(SC_EINVAL, "sc_tx: bad arguments");
    CU(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t) stream;
    // TX phasor table from the cold phasor: renormalised after every qpsk_tx_frame() call, i.e.
    // after the 640-sample preamble and after each 155-sample data frame (qpsk.c:306).  Everything
    // is stream ordered: no host temporaries, no synchronisation.
    AsyncBuf<float2> d_ph(st), d_tab(st);
    CU(d_ph.alloc(1));
    CU(d_tab.alloc((size_t) n_packets * FRAME));
    CU(cudaMemcpyAsync(d_ph.p, m->unit_phase, sizeof(float2), cudaMemcpyDeviceToDevice, st));   // cmplx(0.0f), qpsk.c:375
    if (n_packets > 0) CU(launch_nco_table(d_ph.p, m->tx_rect, NCO_TX_PACKET, 0, n_packets * 9, 1.0f, d_tab.p, st));
    TxArgs a;
    a.bits = bits;
    a.bits_out = bits_out;
    a.seed = seed;
    a.n_packets = n_packets;
    a.gap_samples = gap_samples;
    a.lead_in = lead_in;
    a.tx_table = d_tab.p;
    a.out = out;
    a.stream_stride = stream_stride;
    a.samples_per_stream = samples_per_stream;
    a.n_streams = m->n;
    a.wide = m->wide;
    a.use_channel = ch != nullptr;
    a.scramble = m->packet;
    a.key = m->pk_key;
    memset(&a.ch, 0, sizeof a.ch);
    if (ch) a.ch = *ch;
    CU(launch_tx(a, st));
    return SC_OK;
}

extern "C" int sc_tx_packets_dev(sc_modem *m, const uint8_t *bits, uint8_t *bits_out, uint64_t seed, int n_packets,
                                 int gap_samples, const int32_t *lead_in, int16_t *out, int64_t stream_stride,
                                 int64_t samples_per_stream, void *stream) {
    return tx_common(m, bits, bits_out, seed, n_packets, gap_samples, lead_in, nullptr, out, stream_stride,
                     samples_per_stream, stream);
}

extern "C" int sc_tx_channel_dev(sc_modem *m, const uint8_t *bits, uint8_t *bits_out, uint64_t seed, int n_packets,
                                 int gap_samples, const int32_t *lead_in, const sc_channel *ch, int16_t *out,
                                 int64_t stream_stride, int64_t samples_per_stream, void *stream) {
    if (!ch) return fail(SC_EINVAL, "sc_tx_channel_dev: null channel");
    return tx_common(m, bits, bits_out, seed, n_packets, gap_samples, lead_in, ch, out, stream_stride,
                     samples_per_stream, stream);
}

// ---- stage entry points -----------------------------------------------------------------------
static int stage_device(int device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(SC_ECUDA, "no CUDA device (this library has no CPU path)");
    }
    if (device < 0 || device >= ndev) return fail(SC_EINVAL, "device %d of %d", device, ndev);
    CU(cudaSetDevice(device));
    return SC_OK;
}

extern "C" int sc_fir_batch_dev(int device, int64_t n_streams, int wide, float *memory, float *sample,
                                int64_t sample_stride, int length, void *stream) {
    if (n_streams < 0 || !memory || !sample || length < 0 || sample_stride < length)
        return fail(SC_EINVAL, "sc_fir_batch_dev: bad arguments");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (n_streams == 0 || length == 0) return SC_OK;
    CU(launch_fir_batch((wide & 1) != 0, n_streams, (float2 *) memory, (float2 *) sample, sample_stride, length,
                        (cudaStream_t) stream, (wide & SC_FIR_FAST) != 0));
    return SC_OK;
}

// Immutable per-device tables, shared by every call and stream, built on first use and freed by sc_release_caches():
// the search proposers' operand tables and the FFT tables.  The map is never destroyed: freeing device memory while
// the process exits would race the CUDA runtime's own teardown.
enum TableKind { TAB_SEARCH_MMA, TAB_SEARCH_UMMA, TAB_SEARCH_FFT, TAB_FFT_TW, TAB_FFT_SUPER_TW, TAB_FFT_PERM };
using TableKey = std::tuple<int, int, int, int, int>;     // (kind, device, n, inverse, real)
static std::mutex g_tables_mu;
static std::map<TableKey, DevBuf<char>> &g_tables = *new std::map<TableKey, DevBuf<char>>();

// The table `key` on its device, `count` elements of T written by make() on the host when it is built.
template <typename T, typename Make>
static int device_table(const TableKey &key, size_t count, Make make, const void **out) {
    std::lock_guard<std::mutex> lock(g_tables_mu);
    auto it = g_tables.find(key);
    if (it == g_tables.end()) {
        std::vector<T> h(count);
        make(h.data());
        DevBuf<char> d;                     // released, with its device current, if it is not completed
        CU(cudaSetDevice(std::get<1>(key)));
        CU(d.reserve(count * sizeof(T)));
        CU(cudaMemcpy(d, h.data(), count * sizeof(T), cudaMemcpyHostToDevice));
        it = g_tables.emplace(key, std::move(d)).first;
    }
    *out = it->second.p;
    return SC_OK;
}

// A fragments of the tensor-core proposer (sc_search_mma.cuh) and the fused tcgen05 proposer's A-operand master
// (sc_frontend_umma.cu)
static int search_table(int device, const void **out) {
    return device_table<uint32_t>(TableKey(TAB_SEARCH_MMA, device, 0, 0, 0), (size_t) 9 * 32 * 4, search_mma_make_table, out);
}

static int search_umma_master(int device, const void **out) {
    return device_table<uint16_t>(TableKey(TAB_SEARCH_UMMA, device, 0, 0, 0), (size_t) SU_A_WORDS4 * 8,
                                  search_umma_make_master, out);
}

static int search_args(int64_t n_streams, const float *symbols, int64_t symbol_stride, int32_t *max_index, float *max_value) {
    if (n_streams < 0 || !symbols || !max_index || !max_value || symbol_stride < 255)
        return fail(SC_EINVAL, "sc_preamble_search_batch_dev: bad arguments");
    return SC_OK;
}

// proposer on tcgen05 / tensor memory with TMA loads when the windows allow it (256 symbols per window, 16-byte
// aligned: sc_search_umma.cu), else on mma.sync; identical results
extern "C" int sc_preamble_search_batch_dev(int device, int64_t n_streams, const float *symbols, int64_t symbol_stride,
                                            int32_t *max_index, float *max_value, void *stream) {
    int rc = search_args(n_streams, symbols, symbol_stride, max_index, max_value);
    if (rc != SC_OK) return rc;
    if ((rc = stage_device(device)) != SC_OK) return rc;
    if (n_streams == 0) return SC_OK;
    const void *table = nullptr;
    if (search_umma_eligible((const float2 *) symbols, symbol_stride) && !getenv("SC_SEARCH_NO_TCGEN05")) {
        CU(launch_search_umma_batch(n_streams, (const float2 *) symbols, symbol_stride, max_index, max_value, nullptr,
                                    (cudaStream_t) stream));
        return SC_OK;
    }
    if ((rc = search_table(device, &table)) != SC_OK) return rc;
    CU(launch_search_mma_batch(n_streams, (const float2 *) symbols, symbol_stride, table, max_index, max_value,
                               (cudaStream_t) stream));
    return SC_OK;
}

extern "C" int sc_preamble_search_mma_batch_dev(int device, int64_t n_streams, const float *symbols, int64_t symbol_stride,
                                                int32_t *max_index, float *max_value, void *stream) {
    int rc = search_args(n_streams, symbols, symbol_stride, max_index, max_value);
    if (rc != SC_OK) return rc;
    if ((rc = stage_device(device)) != SC_OK) return rc;
    if (n_streams == 0) return SC_OK;
    const void *table = nullptr;
    if ((rc = search_table(device, &table)) != SC_OK) return rc;
    CU(launch_search_mma_batch(n_streams, (const float2 *) symbols, symbol_stride, table, max_index, max_value,
                               (cudaStream_t) stream));
    return SC_OK;
}

// the tcgen05 kernel only; approx (optional, [n_streams][128]) receives the PROPOSED |correlation|^2 of every lag
extern "C" int sc_preamble_search_tcgen05_batch_dev(int device, int64_t n_streams, const float *symbols, int64_t symbol_stride,
                                                    int32_t *max_index, float *max_value, float *approx, void *stream) {
    int rc = search_args(n_streams, symbols, symbol_stride, max_index, max_value);
    if (rc != SC_OK) return rc;
    if (!search_umma_eligible((const float2 *) symbols, symbol_stride))
        return fail(SC_EINVAL, "sc_preamble_search_tcgen05_batch_dev: needs symbol_stride >= 256, even, and a 16-byte aligned array");
    if ((rc = stage_device(device)) != SC_OK) return rc;
    if (n_streams == 0) return SC_OK;
    CU(launch_search_umma_batch(n_streams, (const float2 *) symbols, symbol_stride, max_index, max_value, approx,
                                (cudaStream_t) stream));
    return SC_OK;
}

extern "C" int sc_preamble_search_direct_batch_dev(int device, int64_t n_streams, const float *symbols,
                                                   int64_t symbol_stride, int32_t *max_index, float *max_value, void *stream) {
    int rc = search_args(n_streams, symbols, symbol_stride, max_index, max_value);
    if (rc != SC_OK) return rc;
    if ((rc = stage_device(device)) != SC_OK) return rc;
    if (n_streams == 0) return SC_OK;
    CU(launch_search_batch(n_streams, (const float2 *) symbols, symbol_stride, max_index, max_value,
                           (cudaStream_t) stream));
    return SC_OK;
}

extern "C" int sc_track_decide_batch_dev(int device, int64_t n_streams, const float *symbols, int64_t symbol_stride,
                                         const int32_t *max_index, const float *max_value, int32_t *rx_timing,
                                         uint32_t call_index, sc_frame_result *results, float *eq_dbg, void *stream) {
    if (n_streams < 0 || !symbols || !max_index || !rx_timing || !results || symbol_stride < WIN)
        return fail(SC_EINVAL, "sc_track_decide_batch_dev: bad arguments");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (n_streams == 0) return SC_OK;
    CU(launch_track_window_batch(n_streams, (const float2 *) symbols, symbol_stride, max_index, max_value, rx_timing,
                                 call_index, sc_keystream_word(call_index), results, eq_dbg, (cudaStream_t) stream));
    return SC_OK;
}

// ---- FFT (fft.h) --------------------------------------------------------------------------------
// kf_factor(), src/fft.c:433-459: radix 4 first, then 2, 3, 5, 7, ...; p > floor(sqrt(n)) => p = n
namespace sc {
void fft_make_plan(int n, int inverse, FftPlan *plan) {
    plan->n = n;
    plan->inverse = inverse ? 1 : 0;
    int p = 4, k = 0;
    const float floor_sqrt = floorf(sqrtf((float) n));
    do {
        while (n % p) {
            switch (p) {
                case 4: p = 2; break;
                case 2: p = 3; break;
                default: p += 2;
            }
            if (p > floor_sqrt) p = n;
        }
        n /= p;
        plan->p[k] = p;
        plan->m[k] = n;
        k++;
    } while (n > 1);
    plan->n_stages = k;
}

// Leaves of kf_work() (src/fft.c:399-404): element i of the working array is input element perm[i]
// (mixed-radix digit reversal of the plan's factors).
void fft_make_permutation(const FftPlan &plan, int *perm) {
    for (int i = 0; i < plan.n; i++) {
        int rem = i, src = 0, mult = 1;
        for (int l = 0; l < plan.n_stages; l++) {
            const int q = rem / plan.m[l];
            rem -= q * plan.m[l];
            src += q * mult;
            mult *= plan.p[l];
        }
        perm[i] = src;
    }
}

// twiddles exactly as fft_alloc() computes them (src/fft.c:70-77), same libm as the reference
void fft_make_twiddles(int n, int inverse, float2 *tw) {
    const double tau = 2.0f * M_PI;
    for (int i = 0; i < n; i++) {
        float phase = (float) (-tau * (float) i / (float) n);
        if (inverse) phase *= -1.0f;
        tw[i] = make_float2(cosf(phase), sinf(phase));
    }
}

// super twiddles of fftr_alloc() (src/fft.c:118-126); ncfft = nfft/2
void fft_make_super_twiddles(int ncfft, int inverse, float2 *tw) {
    for (int i = 0; i < ncfft / 2; i++) {
        float phase = (float) (-M_PI * ((float) (i + 1) / (float) ncfft + .5f));
        if (inverse) phase *= -1.0f;
        tw[i] = make_float2(cosf(phase), sinf(phase));
    }
}
}  // namespace sc

// Per-(device, n, direction) FFT tables: twiddles, the real-FFT super twiddles and the digit-reversal permutation of
// kf_work()'s leaves.  Working storage is NOT cached: transforms too long for shared memory get stream-ordered scratch
// per call (two calls on two streams must not share it).
struct FftDeviceTables {
    const void *tw = nullptr, *super_tw = nullptr, *perm = nullptr;
};

static int fft_tables(int device, int n, int inverse, bool real, FftDeviceTables *t) {
    inverse = inverse ? 1 : 0;
    auto key = [&](int kind) { return TableKey(kind, device, n, inverse, real ? 1 : 0); };
    int rc = device_table<float2>(key(TAB_FFT_TW), n, [&](float2 *h) { fft_make_twiddles(n, inverse, h); }, &t->tw);
    if (rc == SC_OK && real)
        rc = device_table<float2>(key(TAB_FFT_SUPER_TW), std::max(n / 2, 1),
                                  [&](float2 *h) { fft_make_super_twiddles(n, inverse, h); }, &t->super_tw);
    if (rc == SC_OK)
        rc = device_table<int>(key(TAB_FFT_PERM), n, [&](int *h) {
            FftPlan plan;
            fft_make_plan(n, inverse, &plan);
            fft_make_permutation(plan, h);
        }, &t->perm);
    return rc;
}

static int fft_run(int device, int64_t n_batches, int n_core, int inverse, int mode, const void *in, void *out,
                   void *stream) {
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (n_batches == 0) return SC_OK;
    FftDeviceTables t;
    if ((rc = fft_tables(device, n_core, inverse, mode != 0, &t)) != SC_OK) return rc;
    FftPlan plan;
    fft_make_plan(n_core, inverse, &plan);
    cudaStream_t st = (cudaStream_t) stream;
    AsyncBuf<float2> scratch(st);
    if (fft_needs_scratch(n_core)) CU(scratch.alloc((size_t) FFT_SCRATCH_CTAS * 2 * n_core));
    CU(launch_fft(plan, (const float2 *) t.tw, (const float2 *) t.super_tw, (const int *) t.perm, mode, in, out, scratch.p,
                  n_batches, st));
    return SC_OK;
}

extern "C" int sc_release_caches(void) {
    std::lock_guard<std::mutex> lock(g_tables_mu);
    int dev0 = 0;
    cudaGetDevice(&dev0);
    while (!g_tables.empty()) {
        cudaSetDevice(std::get<1>(g_tables.begin()->first));
        g_tables.erase(g_tables.begin());
    }
    cudaSetDevice(dev0);
    cudaGetLastError();
    return SC_OK;
}

extern "C" int sc_fft_batch_dev(int device, int64_t n_batches, int nfft, int inverse, const float *in, float *out,
                                void *stream) {
    if (n_batches < 0 || !in || !out || nfft < 1 || nfft > (1 << 20))
        return fail(SC_EINVAL, "sc_fft_batch_dev: bad arguments");
    return fft_run(device, n_batches, nfft, inverse, 0, in, out, stream);
}

extern "C" int sc_fftr_batch_dev(int device, int64_t n_batches, int nfft, const float *in, float *out, void *stream) {
    if (n_batches < 0 || !in || !out || nfft < 2 || (nfft & 1) || nfft > (1 << 21))
        return fail(SC_EINVAL, "sc_fftr_batch_dev: nfft must be even");
    return fft_run(device, n_batches, nfft / 2, 0, 1, in, out, stream);
}

extern "C" int sc_fftri_batch_dev(int device, int64_t n_batches, int nfft, const float *in, float *out, void *stream) {
    if (n_batches < 0 || !in || !out || nfft < 2 || (nfft & 1) || nfft > (1 << 21))
        return fail(SC_EINVAL, "sc_fftri_batch_dev: nfft must be even");
    return fft_run(device, n_batches, nfft / 2, 1, 2, in, out, stream);
}

// the FFT proposer's spectrum of the preamble (sc_stage_kernels.cu), one immutable table per device
extern "C" int sc_preamble_search_fft_batch_dev(int device, int64_t n_streams, const float *symbols, int64_t symbol_stride,
                                                int32_t *max_index, float *max_value, void *stream) {
    int rc = search_args(n_streams, symbols, symbol_stride, max_index, max_value);
    if (rc != SC_OK) return rc;
    if ((rc = stage_device(device)) != SC_OK) return rc;
    if (n_streams == 0) return SC_OK;
    FftDeviceTables t;
    if ((rc = fft_tables(device, 256, 0, false, &t)) != SC_OK) return rc;
    const void *ptab = nullptr;
    if ((rc = device_table<float>(TableKey(TAB_SEARCH_FFT, device, 0, 0, 0), (size_t) 8 * 32 * 2, search_fft_make_table,
                                  &ptab)) != SC_OK)
        return rc;
    CU(launch_search_fft_batch(n_streams, (const float2 *) symbols, symbol_stride, (const float2 *) t.tw, ptab, max_index, max_value,
                               (cudaStream_t) stream));
    return SC_OK;
}

extern "C" int sc_lock_stats_dev(int device, const sc_frame_result *results, int64_t n_streams, int64_t result_stride,
                                 int n_frames, uint64_t *counters, void *stream) {
    if (!results || !counters || n_streams < 0 || n_frames < 0 || result_stride < n_frames)
        return fail(SC_EINVAL, "sc_lock_stats_dev: bad arguments");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (n_streams == 0 || n_frames == 0) return SC_OK;
    CU(launch_lock_stats(results, n_streams, result_stride, n_frames, (unsigned long long *) counters,
                         (cudaStream_t) stream));
    return SC_OK;
}

extern "C" int sc_ber_stats_dev(int device, const sc_frame_result *results, int64_t n_streams, int64_t result_stride,
                                int n_frames, const uint8_t *tx_bits, int n_packets, const int32_t *lead_in,
                                int gap_samples, const int32_t *group, int n_groups, uint64_t *counters, void *stream) {
    if (!results || !tx_bits || !counters || n_streams < 0 || n_frames < 0 || result_stride < n_frames || n_packets < 1 ||
        gap_samples < 0 || n_groups < 1)
        return fail(SC_EINVAL, "sc_ber_stats_dev: bad arguments");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (n_streams == 0 || n_frames == 0) return SC_OK;
    CU(launch_ber_stats(results, n_streams, result_stride, n_frames, tx_bits, n_packets, lead_in, gap_samples, group,
                        n_groups, (unsigned long long *) counters, (cudaStream_t) stream));
    return SC_OK;
}

extern "C" int sc_packet_ber_stats_dev(int device, const sc_packet_result *packets, int64_t capacity,
                                       const uint64_t *n_found, const sc_frame_result *results, int64_t n_streams,
                                       int64_t result_stride, int n_frames, const uint8_t *tx_bits, int n_packets,
                                       const int32_t *lead_in, int gap_samples, const int32_t *group, int n_groups,
                                       uint64_t *counters, void *stream) {
    if (!packets || !n_found || !results || !tx_bits || !counters || capacity < 0 || n_streams < 0 || n_frames < 0 ||
        result_stride < n_frames || n_packets < 1 || gap_samples < 0 || n_groups < 1)
        return fail(SC_EINVAL, "sc_packet_ber_stats_dev: bad arguments");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (capacity == 0 || n_streams == 0 || n_frames < 3) return SC_OK;
    CU(launch_packet_ber_stats(packets, capacity, (const unsigned long long *) n_found, results, n_streams,
                               result_stride, n_frames, tx_bits, n_packets, lead_in, gap_samples, group, n_groups,
                               (unsigned long long *) counters, (cudaStream_t) stream));
    return SC_OK;
}

// ---- coded payload (DESIGN.md section 8c) -------------------------------------------------------
extern "C" int sc_packet_encode_dev(int device, const uint8_t *payload, int64_t n, uint8_t *bits, void *stream) {
    if (!payload || !bits || n < 0) return fail(SC_EINVAL, "sc_packet_encode_dev: bad arguments");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (n == 0) return SC_OK;
    CU(launch_packet_encode(payload, n, bits, (cudaStream_t) stream));
    return SC_OK;
}

extern "C" int sc_packet_llr_dev(int device, const float *packet_symbols, int64_t capacity, const uint64_t *n_found,
                                 float *llr, void *stream) {
    if (!packet_symbols || !n_found || !llr || capacity < 0) return fail(SC_EINVAL, "sc_packet_llr_dev: bad arguments");
    if (((uintptr_t) packet_symbols & 7) != 0 || ((uintptr_t) llr & 7) != 0)
        return fail(SC_EINVAL, "sc_packet_llr_dev: packet_symbols and llr must be 8-byte aligned");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (capacity == 0) return SC_OK;
    PacketKey key;
    for (int f = 0; f < 8; f++) key.k[f] = sc_packet_keystream_word(f);
    CU(launch_packet_llr(packet_symbols, capacity, (const unsigned long long *) n_found, llr, key, (cudaStream_t) stream));
    return SC_OK;
}

extern "C" int sc_packet_decode_dev(int device, const float *llr, int64_t capacity, const uint64_t *n_found,
                                    sc_packet_payload *out, void *stream) {
    if (!llr || !n_found || !out || capacity < 0) return fail(SC_EINVAL, "sc_packet_decode_dev: bad arguments");
    if (((uintptr_t) llr & 7) != 0 || ((uintptr_t) out & 3) != 0)
        return fail(SC_EINVAL, "sc_packet_decode_dev: llr must be 8-byte and out 4-byte aligned");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (capacity == 0) return SC_OK;
    CU(launch_packet_decode(llr, capacity, (const unsigned long long *) n_found, out, (cudaStream_t) stream));
    return SC_OK;
}

extern "C" int sc_packet_payload_bytes(int code) {
    return code == SC_PACKET_CODE_R12 ? 27 : code == SC_PACKET_CODE_R23 ? 36 : code == SC_PACKET_CODE_R34 ? 41 : 0;
}

extern "C" int sc_packet_encode_ex_dev(int device, const uint8_t *payload, int64_t n_streams, int n_packets,
                                       const uint8_t *stream_code, uint8_t *bits, void *stream) {
    if (!payload || !stream_code || !bits || n_streams < 0 || n_packets < 1)
        return fail(SC_EINVAL, "sc_packet_encode_ex_dev: bad arguments");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (n_streams == 0) return SC_OK;
    CU(launch_packet_encode_ex(payload, n_streams, n_packets, stream_code, bits, (cudaStream_t) stream));
    return SC_OK;
}

extern "C" int sc_packet_decode_ex_dev(int device, const float *llr, const sc_packet_result *packets, int64_t capacity,
                                       const uint64_t *n_found, const uint8_t *stream_code, int64_t n_streams,
                                       sc_packet_payload_ex *out, void *stream) {
    if (!llr || !packets || !n_found || !stream_code || !out || capacity < 0 || n_streams < 0)
        return fail(SC_EINVAL, "sc_packet_decode_ex_dev: bad arguments");
    if (((uintptr_t) llr & 7) != 0 || ((uintptr_t) out & 3) != 0)
        return fail(SC_EINVAL, "sc_packet_decode_ex_dev: llr must be 8-byte and out 4-byte aligned");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (capacity == 0) return SC_OK;
    CU(launch_packet_decode_ex(llr, packets, capacity, (const unsigned long long *) n_found, stream_code, n_streams, out,
                               (cudaStream_t) stream));
    return SC_OK;
}

extern "C" int sc_packet_decode_blind_dev(int device, const float *llr, int64_t capacity, const uint64_t *n_found,
                                          unsigned code_mask, sc_packet_payload_ex *out, void *stream) {
    if (!llr || !n_found || !out || capacity < 0 || code_mask == 0u || (code_mask & ~7u) != 0u)
        return fail(SC_EINVAL, "sc_packet_decode_blind_dev: bad arguments");
    if (((uintptr_t) llr & 7) != 0 || ((uintptr_t) out & 3) != 0)
        return fail(SC_EINVAL, "sc_packet_decode_blind_dev: llr must be 8-byte and out 4-byte aligned");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    if (capacity == 0) return SC_OK;
    CU(launch_packet_decode_blind(llr, capacity, (const unsigned long long *) n_found, code_mask, out,
                                  (cudaStream_t) stream));
    return SC_OK;
}

// ---- checkpoint / resume ------------------------------------------------------------------------
namespace {
struct StateHeader {
    uint32_t magic, version;
    int64_t n, n_pad;
    uint32_t flags, call;
    float foffset;
    uint16_t lfsr_rx, pad;
    float2 rx_phase;
};
const uint32_t STATE_MAGIC = 0x53433242u, STATE_VERSION = 1;   // "SC2B"

struct StateLayout {
    size_t off_timing, off_maxi, off_maxv, off_win, off_hist, off_mix, total;
};
StateLayout state_layout(const sc_modem *m) {
    StateLayout L;
    size_t o = (sizeof(StateHeader) + 15) / 16 * 16;
    auto take = [&](size_t bytes) { size_t at = o; o = (o + bytes + 15) / 16 * 16; return at; };
    L.off_timing = take((size_t) m->n_pad * sizeof(int));
    L.off_maxi = take((size_t) m->n_pad * sizeof(int));
    L.off_maxv = take((size_t) m->n_pad * sizeof(float));
    L.off_win = take((size_t) (m->n_pad / 32) * WIN_ROWS * 32 * sizeof(float2));
    L.off_hist = take((size_t) m->n * FRAME * sizeof(int16_t));
    L.off_mix = take((size_t) FRAME * sizeof(float2));
    L.total = o;
    return L;
}
}  // namespace

extern "C" int64_t sc_state_size(const sc_modem *m) { return m ? (int64_t) state_layout(m).total : 0; }

extern "C" int sc_state_export(sc_modem *m, void *buf, int64_t buf_bytes) {
    if (!m || !buf) return fail(SC_EINVAL, "sc_state_export: bad arguments");
    if (m->poisoned) return fail(SC_ESTATE, "sc_state_export: the bank is in a failed-batch state");
    if (m->packet) return fail(SC_EINVAL, "sc_state_export: not available for SC_FLAG_PACKET banks");
    const StateLayout L = state_layout(m);
    if (buf_bytes < (int64_t) L.total) return fail(SC_EINVAL, "sc_state_export: buffer smaller than sc_state_size()");
    int rc = drain(m);
    if (rc != SC_OK) return rc;
    CU(cudaDeviceSynchronize());                           // the caller's stream may still be writing state
    char *b = (char *) buf;
    StateHeader h;
    memset(&h, 0, sizeof h);
    h.magic = STATE_MAGIC;
    h.version = STATE_VERSION;
    h.n = m->n;
    h.n_pad = m->n_pad;
    h.flags = m->flags;
    h.call = m->call;
    h.foffset = m->foffset;
    h.lfsr_rx = m->lfsr_rx;
    CU(cudaMemcpy(&h.rx_phase, m->rx_phase, sizeof(float2), cudaMemcpyDeviceToHost));
    memcpy(b, &h, sizeof h);
    CU(cudaMemcpy(b + L.off_timing, m->timing[m->call & 1], (size_t) m->n_pad * sizeof(int), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(b + L.off_maxi, m->max_index, (size_t) m->n_pad * sizeof(int), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(b + L.off_maxv, m->max_value, (size_t) m->n_pad * sizeof(float), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(b + L.off_win, m->win, (size_t) (m->n_pad / 32) * WIN_ROWS * 32 * sizeof(float2), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(b + L.off_hist, m->hist, (size_t) m->n * FRAME * sizeof(int16_t), cudaMemcpyDeviceToHost));
    if (m->mix_table) CU(cudaMemcpy(b + L.off_mix, m->mix_table, (size_t) FRAME * sizeof(float2), cudaMemcpyDeviceToHost));
    else memset(b + L.off_mix, 0, (size_t) FRAME * sizeof(float2));
    return SC_OK;
}

extern "C" int sc_state_import(sc_modem *m, const void *buf, int64_t buf_bytes) {
    if (!m || !buf) return fail(SC_EINVAL, "sc_state_import: bad arguments");
    if (m->packet) return fail(SC_EINVAL, "sc_state_import: not available for SC_FLAG_PACKET banks");
    const StateLayout L = state_layout(m);
    if (buf_bytes < (int64_t) L.total) return fail(SC_EINVAL, "sc_state_import: buffer smaller than sc_state_size()");
    const char *b = (const char *) buf;
    StateHeader h;
    memcpy(&h, b, sizeof h);
    if (h.magic != STATE_MAGIC || h.version != STATE_VERSION) return fail(SC_EINVAL, "sc_state_import: not a state image");
    if (h.n != m->n || h.n_pad != m->n_pad || h.flags != m->flags || h.foffset != m->foffset)
        return fail(SC_EINVAL, "sc_state_import: the image was taken from a bank with other parameters");
    int rc = drain(m);
    if (rc != SC_OK) return rc;
    CU(m->mix_table.reserve(FRAME));
    CU(cudaMemcpy(m->rx_phase, &h.rx_phase, sizeof(float2), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(m->timing[h.call & 1], b + L.off_timing, (size_t) m->n_pad * sizeof(int), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(m->max_index, b + L.off_maxi, (size_t) m->n_pad * sizeof(int), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(m->max_value, b + L.off_maxv, (size_t) m->n_pad * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(m->win, b + L.off_win, (size_t) (m->n_pad / 32) * WIN_ROWS * 32 * sizeof(float2), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(m->hist, b + L.off_hist, (size_t) m->n * FRAME * sizeof(int16_t), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(m->mix_table, b + L.off_mix, (size_t) FRAME * sizeof(float2), cudaMemcpyHostToDevice));
    m->call = h.call;
    m->lfsr_rx = h.lfsr_rx;
    m->poisoned = m->in_flight = false;
    return SC_OK;
}

// ---- options and per-kernel profiling ----------------------------------------------------------
extern "C" int sc_set_option(sc_modem *m, int option, int64_t value) {
    if (!m) return fail(SC_EINVAL, "sc_set_option: null handle");
    switch (option) {
        case SC_OPT_SLAB_PARTS:
            if (value < 0 || value > 1024) return fail(SC_EINVAL, "sc_set_option: slab parts out of range");
            m->slab_parts = (int) value;
            return SC_OK;
        case SC_OPT_PROFILE:
            m->profile = value != 0;
            return SC_OK;
        case SC_OPT_FE_SEARCH:
            if (value != SC_FE_SEARCH_DIRECT && value != SC_FE_SEARCH_MMA && value != SC_FE_SEARCH_TCGEN05)
                return fail(SC_EINVAL, "sc_set_option: unknown search mode");
            m->fe_search_mma = value != SC_FE_SEARCH_DIRECT;
            m->fe_search_umma = value == SC_FE_SEARCH_TCGEN05;
            return SC_OK;
        case SC_OPT_TRACKER:
            if (value < SC_TRACKER_AUTO || value > SC_TRACKER_COOP) return fail(SC_EINVAL, "sc_set_option: unknown tracker");
            m->tracker = (int) value;
            return SC_OK;
        case SC_OPT_OVERLAP:
            if (value < SC_OVERLAP_AUTO || value > SC_OVERLAP_ON) return fail(SC_EINVAL, "sc_set_option: unknown overlap mode");
            m->overlap = (int) value;
            return SC_OK;
        case SC_OPT_H2D_MODE:
            if (value < SC_H2D_COLUMNS || value > SC_H2D_COLUMNS_3D) return fail(SC_EINVAL, "sc_set_option: unknown H2D mode");
            m->h2d_mode = (int) value;
            return SC_OK;
        default:
            return fail(SC_EINVAL, "sc_set_option: unknown option %d", option);
    }
}

static int prof_sum(std::vector<Event> &v, double *ms, double *count) {
    *ms = 0.0;
    *count = 0.0;
    for (size_t i = 0; i + 1 < v.size(); i += 2) {
        float t = 0.f;
        CU(cudaEventElapsedTime(&t, v[i], v[i + 1]));
        *ms += t;
        *count += 1.0;
    }
    v.clear();
    return SC_OK;
}

extern "C" int sc_profile_read(sc_modem *m, double out[4]) {
    if (!m || !out) return fail(SC_EINVAL, "sc_profile_read: bad arguments");
    CU(cudaSetDevice(m->device));
    CU(cudaDeviceSynchronize());
    int rc = prof_sum(m->ev_fe, &out[0], &out[1]);
    if (rc != SC_OK) return rc;
    return prof_sum(m->ev_tk, &out[2], &out[3]);
}

// Self-test hook (tests/test_stage_gpu.py): counts float bit patterns in [lo_bits, hi_bits] for which
// the tracker's branch-free reciprocal differs from __frcp_rn.  *mismatches is a device uint64.
extern "C" int sc_selftest_rcp_dev(int device, uint32_t lo_bits, uint32_t hi_bits, uint64_t *mismatches, void *stream) {
    if (!mismatches || hi_bits < lo_bits) return fail(SC_EINVAL, "sc_selftest_rcp_dev: bad arguments");
    int rc = stage_device(device);
    if (rc != SC_OK) return rc;
    CU(launch_selftest_rcp(lo_bits, hi_bits, (unsigned long long *) mismatches, (cudaStream_t) stream));
    return SC_OK;
}
