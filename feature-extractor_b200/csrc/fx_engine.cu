// fx_engine.cu -- host side of libfxb200.so: the C ABI of include/fx_engine.h over the kernels in
// fx_analyse.cu / fx_post.cu.  No CPU fallback: every analysis call runs the CUDA path or fails.
//
// Per-track state kept resident in HBM between calls (all ping-ponged so that chunks of one call may read
// the carry-in while another chunk writes the carry-out):
//   tail   [T][N-H]   fp32  overlap of the framer            (RealTimeAudioDataOverlapper, RealTimeAudioAnalysis.h:194-242)
//   prev   [T][M]     fp32  Re spectrum of the last non-silent frame (previousBinMagnitudes, SpectralCharacteristics.h:203)
//   hist   [T][32][12] fp32 last raw feature rows            (AudioFeatures / ValueHistory, RealTimeAnalyser.h:70-92)
// The ping-pong side and the hop count live per TRACK GROUP: the groups of the real-time path advance independently.
//
// Real-time path (threading contract in include/fx_engine.h):
//   audio thread   fx_push_block -> fx::TrackRings::push into the pinned ring (AudioDataCollector's 4096-float ring,
//                  AudioDataCollector.h:24, becomes ring_hops hops per track) + one futex wake per group that completed a hop
//   group worker   rt_batch: cudaMemcpy2DAsync ring -> device on the group's stream, K1..K3, smoothed vectors back, seqlock
//                  publish (replaces the two juce::Threads per track, RealTimeAnalyser.h:97-127)
// Every buffer of that path is allocated in fx_engine_create; a batch performs no allocation and synchronises only its own
// stream.
#include "fx_kernels.cuh"
#include "fx_fft.cuh"
#include "fx_rt_host.h"
#include "fx_tables.h"
#include <arpa/inet.h>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace {
thread_local std::string g_create_error;
constexpr size_t kLatestWords = FX_NUM_FEATURES + 2;      // 12 smoothed floats + the 64-bit hop count as two words
constexpr int    kMaxGroups = 256;                        // fx_push_block keeps one flag per group on its stack
}

// the buffers one run of K1 -> K1b -> K2 -> K3 hands from kernel to kernel
struct fx_scratch
{
    unsigned char* rec = nullptr;       // [tracks][frames] records of fx::frame_rec_bytes (window)
    float* first_spec = nullptr;        // [tracks * chunks][M]
    float* last_spec = nullptr;
    int*   first_idx = nullptr;         // [tracks * chunks]
};

struct fx_group
{
    int          t0 = 0, n = 0;          // track range
    // carried-state bookkeeping of this group's tracks
    int          flip = 0;
    long         frames_done = 0;        // hops analysed since the last reset
    // real-time path (allocated when ring_hops > 0)
    cudaStream_t stream = nullptr;
    float*       d_stage = nullptr;      // [n][stage_hops * H] newly complete hops
    float*       d_raw = nullptr;        // [n][stage_hops][12]
    float*       d_smooth = nullptr;
    fx_scratch   scratch;
    int          max_chunks = 1;
    float*       h_latest = nullptr;     // pinned [n][14], landing zone of the smoothed vectors
    fx::SeqBlock latest;                 // what fx_poll_features reads
    std::mutex   batch_mutex;            // held by a batch and by the parameter calls (never by the audio thread)
    fx::WakeWord wake;
    std::thread  worker;
    bool         params_dirty = true;    // this group's slice of the per-track parameter arrays must be uploaded
    bool         ratio_pending = false;  // a gain change: the carried overlap must be rescaled before the next hop
    std::string  worker_error;
    std::atomic<int> worker_status { 0 };
};

struct fx_engine
{
    fx_config cfg{};
    int N = 0, H = 0, M = 0, NB = 0, log2_hop = 0, sm_count = 148, ctas_per_sm = 2;
    cudaStream_t stream = nullptr;
    std::string err;
    std::mutex err_mutex;
    std::mutex api_mutex;                // offline calls, parameter calls, fx_process, start / stop
    std::atomic<uint64_t> launches{0};

    float2 *d_tw2 = nullptr, *d_tw1f = nullptr;
    double *d_ex_tab = nullptr;
    int    *d_ex_off = nullptr;
    short  *d_her_tab = nullptr;
    size_t ex_tab_len = 0;
    short   f0bin_pow2[16] = {};
    double bin_var = 0.0;
    float  iir_c1 = 0.0f, iir_c2 = 0.0f;

    // per-track parameters
    std::vector<float> h_gain, h_mult, h_ratio;
    std::vector<int>   h_type, h_hist;
    std::vector<long>  h_reset, h_start;
    float *d_gain = nullptr, *d_mult = nullptr, *d_ratio = nullptr;
    int   *d_type = nullptr, *d_hist = nullptr;
    long  *d_reset = nullptr, *d_start = nullptr;

    // carried state
    float* d_tail[2] = { nullptr, nullptr };
    float* d_prev[2] = { nullptr, nullptr };
    float* d_hrows[2] = { nullptr, nullptr };
    cudaEvent_t ev_last = nullptr;       // end of the last offline call's device work (cross-stream ordering of the carried state)

    // offline scratch (grown on demand)
    fx_scratch scratch;
    long  chunk_capacity = 0;           // in (track, chunk) pairs
    long  rec_capacity = 0;             // frames per track
    float *d_raw = nullptr, *d_smooth = nullptr, *d_diag = nullptr;
    long  result_capacity = 0;          // frames per track
    float *d_latest = nullptr, *h_latest = nullptr;      // [T][14]

    // host API pipeline
    float* d_audio_slot[3] = { nullptr, nullptr, nullptr };
    long   audio_slot_floats = 0;
    unsigned char* d_pcm_slot[3] = { nullptr, nullptr, nullptr };     // file ingest: raw PCM rows of one track group
    long   pcm_slot_bytes = 0;
    cudaStream_t pipe_stream[3] = { nullptr, nullptr, nullptr };      // upload, analysis, download
    cudaEvent_t  ev_ready[3] = { nullptr, nullptr, nullptr }, ev_free[3] = { nullptr, nullptr, nullptr };

    // real-time path
    bool   rt_enabled = false;
    float* h_ring = nullptr;            // pinned [T][ring_len]
    long   ring_len = 0;
    long   stage_hops = 0;
    fx::TrackRings rings;
    std::vector<std::unique_ptr<fx_group>> groups;
    std::atomic<int> rt_running { 0 }, rt_stop { 0 };
    fx_features_callback cb = nullptr;
    void*  cb_user = nullptr;
    std::atomic<uint64_t> st_batches { 0 }, st_hops { 0 }, st_overruns { 0 }, st_ns_sum { 0 }, st_ns_max { 0 };

    // optional per-kernel timing (bench.py roofline; offline calls only)
    bool   profiling = false;
    struct ProfRec { cudaEvent_t a, b, c; };
    std::vector<ProfRec> prof_pending, prof_free;
};

namespace {

using namespace fx;

void set_error (fx_engine* e, const char* what, cudaError_t ce)
{
    char buf[512];
    snprintf (buf, sizeof (buf), "%s: %s", what, cudaGetErrorString (ce));
    if (e) { std::lock_guard<std::mutex> lk (e->err_mutex); e->err = buf; }
    else g_create_error = buf;
}
void set_error (fx_engine* e, const char* text)
{
    std::lock_guard<std::mutex> lk (e->err_mutex);
    e->err = text;
}

#define FX_CUDA(e, call)                                                             \
    do { cudaError_t ce_ = (call); if (ce_ != cudaSuccess) { set_error ((e), #call, ce_); return FX_ERR_CUDA; } } while (0)

int ilog2 (int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

// ---- per-track parameters ----------------------------------------------------------------------------------
// slice [t0, t0 + n) of the parameter arrays, on `s`.  The sources are pageable: cudaMemcpyAsync stages them before it
// returns, so the vectors may change again afterwards.
fx_status upload_params (fx_engine* e, int t0, int n, cudaStream_t s)
{
    const size_t o = (size_t) t0, c = (size_t) n;
    FX_CUDA (e, cudaMemcpyAsync (e->d_gain + o,  e->h_gain.data() + o,  c * sizeof (float), cudaMemcpyHostToDevice, s));
    FX_CUDA (e, cudaMemcpyAsync (e->d_mult + o,  e->h_mult.data() + o,  c * sizeof (float), cudaMemcpyHostToDevice, s));
    FX_CUDA (e, cudaMemcpyAsync (e->d_type + o,  e->h_type.data() + o,  c * sizeof (int),   cudaMemcpyHostToDevice, s));
    FX_CUDA (e, cudaMemcpyAsync (e->d_hist + o,  e->h_hist.data() + o,  c * sizeof (int),   cudaMemcpyHostToDevice, s));
    FX_CUDA (e, cudaMemcpyAsync (e->d_reset + o, e->h_reset.data() + o, c * sizeof (long),  cudaMemcpyHostToDevice, s));
    FX_CUDA (e, cudaMemcpyAsync (e->d_start + o, e->h_start.data() + o, c * sizeof (long),  cudaMemcpyHostToDevice, s));
    return FX_OK;
}

// A gain change (AudioDataCollector.h:88 multiplies on the way out of the ring, so the older part of the next windows keeps
// the old gain; K1 applies the current one to the whole window): rescale the carried overlap of [t0, t0 + n) by old / new.
fx_status apply_gain_ratio (fx_engine* e, int t0, int n, int side, cudaStream_t s)
{
    const size_t o = (size_t) t0;
    FX_CUDA (e, cudaMemcpyAsync (e->d_ratio + o, e->h_ratio.data() + o, (size_t) n * sizeof (float), cudaMemcpyHostToDevice, s));
    FX_CUDA (e, launch_tail_scale (e->d_tail[side] + o * (size_t) (e->N - e->H), e->N - e->H, e->d_ratio + o, n, s));
    for (int t = t0; t < t0 + n; ++t) e->h_ratio[(size_t) t] = 1.0f;
    e->launches += 1;
    return FX_OK;
}

fx_status ensure_chunks (fx_engine* e, long pairs)
{
    if (pairs <= e->chunk_capacity) return FX_OK;
    // grow: earlier work that used the old buffers must have finished
    FX_CUDA (e, cudaDeviceSynchronize());
    cudaFree (e->scratch.first_spec); cudaFree (e->scratch.last_spec); cudaFree (e->scratch.first_idx);
    e->scratch.first_spec = e->scratch.last_spec = nullptr; e->scratch.first_idx = nullptr; e->chunk_capacity = 0;
    FX_CUDA (e, cudaMalloc (&e->scratch.first_spec, (size_t) pairs * e->M * sizeof (float)));
    FX_CUDA (e, cudaMalloc (&e->scratch.last_spec,  (size_t) pairs * e->M * sizeof (float)));
    FX_CUDA (e, cudaMalloc (&e->scratch.first_idx,  (size_t) pairs * sizeof (int)));
    e->chunk_capacity = pairs;
    return FX_OK;
}

fx_status ensure_results (fx_engine* e, long frames)
{
    if (frames <= e->result_capacity) return FX_OK;
    FX_CUDA (e, cudaDeviceSynchronize());
    cudaFree (e->d_raw); cudaFree (e->d_smooth); cudaFree (e->d_diag);
    e->d_raw = e->d_smooth = e->d_diag = nullptr; e->result_capacity = 0;
    const size_t rows = (size_t) e->cfg.n_tracks * (size_t) frames;
    FX_CUDA (e, cudaMalloc (&e->d_raw,    rows * FX_NUM_FEATURES * sizeof (float)));
    FX_CUDA (e, cudaMalloc (&e->d_smooth, rows * FX_NUM_FEATURES * sizeof (float)));
    FX_CUDA (e, cudaMalloc (&e->d_diag,   rows * FX_NUM_DIAG * sizeof (float)));
    e->result_capacity = frames;
    return FX_OK;
}

fx_status ensure_records (fx_engine* e, long frames)
{
    if (frames <= e->rec_capacity) return FX_OK;
    FX_CUDA (e, cudaDeviceSynchronize());
    cudaFree (e->scratch.rec);
    e->scratch.rec = nullptr; e->rec_capacity = 0;
    FX_CUDA (e, cudaMalloc (&e->scratch.rec, (size_t) e->cfg.n_tracks * (size_t) frames * fx::frame_rec_bytes (e->N)));
    e->rec_capacity = frames;
    return FX_OK;
}

// How many chunks per track.  All CTAs carry equal work, so the launch takes ceil (CTAs / resident slots) rounds and an almost
// empty last round costs a whole chunk's time: 4096 tracks on 444 slots are 9.2 rounds as whole tracks but 36.9 as quarters.
// Against that, every chunk start refills the whole window and repeats the prologue (about two frames' worth).  Among the
// chunk counts that give at least a few rounds over the machine take the one with the best fill x (1 - start-up share); never
// chunks shorter than 8 frames.
int choose_chunks (const fx_engine* e, long n_tracks, long frames)
{
    if (frames <= 8 || n_tracks <= 0) return 1;
    const long slots = (long) e->sm_count * e->ctas_per_sm;
    const long target = slots * 6;
    const long max_c = (frames + 7) / 8;
    long c = (target + n_tracks - 1) / n_tracks;
    if (c > max_c) c = max_c;
    if (c < 1) c = 1;
    const double startup_frames = 2.0;
    long best_c = c; double best_score = 0.0;
    for (long k = c; k <= c + 8 && k <= max_c; ++k)
    {
        const long ctas = n_tracks * k, rounds = (ctas + slots - 1) / slots;
        const double fill = (double) ctas / (double) (rounds * slots);
        const double fpc = (double) ((frames + k - 1) / k);
        const double score = fill * fpc / (fpc + startup_frames);
        if (score > best_score + 1e-9) { best_score = score; best_c = k; }
    }
    return (int) best_c;
}

// K1 -> K1b -> K2 -> K3 for tracks [t0, t0 + nt) on `s`, reading the carried state on side `flip` and writing side flip ^ 1;
// `frames_done` hops of these tracks were analysed before.  Output pointers are already offset to track t0's rows; `sc` is
// offset to track t0 as well (rec: t0 * frames, chunk buffers: t0 * n_chunks).  Does NOT advance the bookkeeping.
fx_status run_range (fx_engine* e, int t0, int nt, int n_chunks, int flip, long frames_done, const fx_scratch& sc,
                     const float* d_audio, long track_stride, long frames,
                     float* d_raw, float* d_smooth, float* d_diag, float* d_spec, float* d_latest, cudaStream_t s, bool may_profile)
{
    const int in = flip, out = flip ^ 1;
    const int fpc = (int) ((frames + n_chunks - 1) / n_chunks);

    AnalyseParams a{};
    a.audio = d_audio; a.track_stride = track_stride;
    a.tail_in = e->d_tail[in] + (size_t) t0 * (e->N - e->H);
    a.tail_out = e->d_tail[out] + (size_t) t0 * (e->N - e->H);
    a.first_hop = frames_done;
    a.n_frames = (int) frames; a.frames_per_chunk = fpc; a.n_chunks = n_chunks;
    a.hop = e->H; a.log2_hop = e->log2_hop;
    a.use_bulk = (((uintptr_t) d_audio & 15u) == 0 && (track_stride % 4) == 0 && (e->H % 4) == 0) ? 1 : 0;       // the kernel copies 16-byte pieces (cp.async)
    a.want_margins = d_diag != nullptr ? 1 : 0;
    a.gain = e->d_gain + t0;
    a.sample_rate = e->cfg.sample_rate; a.bin_var = e->bin_var; a.iir_c1 = e->iir_c1; a.iir_c2 = e->iir_c2;
    a.tw2 = e->d_tw2; a.tw1f = e->d_tw1f;
    a.her_tab = e->d_her_tab; a.ex_tab = e->d_ex_tab; a.ex_off = e->d_ex_off;
    for (int k = 0; k < 16; ++k) a.f0bin_pow2[k] = e->f0bin_pow2[k];
    a.rec = sc.rec;
    a.first_spec = sc.first_spec; a.last_spec = sc.last_spec; a.first_idx = sc.first_idx;
    a.spectrum = e->cfg.spectrum;
    a.spec = d_spec;
    const bool prof = may_profile && e->profiling;
    fx_engine::ProfRec pr{};
    if (prof)
    {
        if (! e->prof_free.empty()) { pr = e->prof_free.back(); e->prof_free.pop_back(); }
        else { FX_CUDA (e, cudaEventCreate (&pr.a)); FX_CUDA (e, cudaEventCreate (&pr.b)); FX_CUDA (e, cudaEventCreate (&pr.c)); }
        FX_CUDA (e, cudaEventRecord (pr.a, s));
    }
    FX_CUDA (e, launch_analyse (e->N, nt, a, s));
    if (prof) FX_CUDA (e, cudaEventRecord (pr.b, s));

    FinalizeParams fz{};
    fz.rec = a.rec; fz.n_rows = (long) nt * frames; fz.window = e->N; fz.sample_rate = e->cfg.sample_rate; fz.bin_var = e->bin_var;
    fz.raw = d_raw; fz.diag = d_diag;
    FX_CUDA (e, launch_finalize (fz, s));

    FluxFixParams fp{};
    fp.n_frames = (int) frames; fp.n_chunks = n_chunks; fp.m = e->M;
    fp.first_spec = a.first_spec; fp.last_spec = a.last_spec; fp.first_idx = a.first_idx;
    fp.prev_in = e->d_prev[in] + (size_t) t0 * e->M;
    fp.prev_out = e->d_prev[out] + (size_t) t0 * e->M;
    fp.raw = d_raw;
    FX_CUDA (e, launch_flux_fix (nt, fp, s));

    SmoothParams sp{};
    sp.n_frames = (int) frames; sp.frames_before = frames_done; sp.rms_pushes = e->cfg.rms_pushes_per_frame;
    sp.raw = d_raw; sp.smooth = d_smooth; sp.diag = d_diag;
    sp.hist_in = e->d_hrows[in] + (size_t) t0 * kHistRows * FX_NUM_FEATURES;
    sp.hist_out = e->d_hrows[out] + (size_t) t0 * kHistRows * FX_NUM_FEATURES;
    sp.onset_type = e->d_type + t0; sp.onset_hist = e->d_hist + t0; sp.onset_mult = e->d_mult + t0; sp.onset_reset = e->d_reset + t0;
    sp.track_start = e->d_start + t0;
    sp.latest = d_latest;
    FX_CUDA (e, launch_smooth (nt, sp, s));
    if (prof) { FX_CUDA (e, cudaEventRecord (pr.c, s)); e->prof_pending.push_back (pr); }
    e->launches += 5;
    return FX_OK;
}

// fx_scratch of the engine-wide (offline) buffers, offset to track t0
fx_scratch offline_scratch (const fx_engine* e, long t0, long frames, int n_chunks)
{
    fx_scratch sc;
    const size_t coff = (size_t) t0 * (size_t) n_chunks;
    sc.rec = e->scratch.rec + (size_t) t0 * (size_t) frames * fx::frame_rec_bytes (e->N);
    sc.first_spec = e->scratch.first_spec + coff * e->M;
    sc.last_spec  = e->scratch.last_spec + coff * e->M;
    sc.first_idx  = e->scratch.first_idx + coff;
    return sc;
}

// ---- real-time workers ------------------------------------------------------------------------------------------
void rt_stop_workers (fx_engine* e)
{
    if (! e->rt_running.load()) return;
    e->rt_stop.store (1);
    for (auto& g : e->groups) g->wake.signal();
    for (auto& g : e->groups) if (g->worker.joinable()) g->worker.join();
    e->rt_running.store (0);
    e->rt_stop.store (0);
}

void free_engine (fx_engine* e)
{
    if (! e) return;
    rt_stop_workers (e);
    cudaSetDevice (e->cfg.device);
    cudaDeviceSynchronize();
    cudaFree (e->d_tw2); cudaFree (e->d_tw1f); cudaFree (e->d_her_tab); cudaFree (e->d_ex_tab); cudaFree (e->d_ex_off);
    cudaFree (e->d_gain); cudaFree (e->d_mult); cudaFree (e->d_ratio); cudaFree (e->d_type); cudaFree (e->d_hist); cudaFree (e->d_reset); cudaFree (e->d_start);
    for (int i = 0; i < 2; ++i) { cudaFree (e->d_tail[i]); cudaFree (e->d_prev[i]); cudaFree (e->d_hrows[i]); }
    cudaFree (e->scratch.first_spec); cudaFree (e->scratch.last_spec); cudaFree (e->scratch.first_idx); cudaFree (e->scratch.rec);
    cudaFree (e->d_raw); cudaFree (e->d_smooth); cudaFree (e->d_diag); cudaFree (e->d_latest);
    if (e->h_latest) cudaFreeHost (e->h_latest);
    for (int i = 0; i < 3; ++i) cudaFree (e->d_pcm_slot[i]);
    for (int i = 0; i < 3; ++i) { cudaFree (e->d_audio_slot[i]); if (e->pipe_stream[i]) cudaStreamDestroy (e->pipe_stream[i]); }
    for (int i = 0; i < 3; ++i) { if (e->ev_ready[i]) cudaEventDestroy (e->ev_ready[i]); if (e->ev_free[i]) cudaEventDestroy (e->ev_free[i]); }
    if (e->ev_last) cudaEventDestroy (e->ev_last);
    if (e->h_ring) cudaFreeHost (e->h_ring);
    for (auto& g : e->groups)
    {
        cudaFree (g->d_stage); cudaFree (g->d_raw); cudaFree (g->d_smooth);
        cudaFree (g->scratch.rec); cudaFree (g->scratch.first_spec); cudaFree (g->scratch.last_spec); cudaFree (g->scratch.first_idx);
        if (g->stream) cudaStreamDestroy (g->stream);
    }
    for (auto* v : { &e->prof_pending, &e->prof_free })
        for (auto& pr : *v) { cudaEventDestroy (pr.a); cudaEventDestroy (pr.b); cudaEventDestroy (pr.c); }
    if (e->stream) cudaStreamDestroy (e->stream);
    delete e;
}

// the published vector of a track that has analysed nothing yet: AudioFeatures::getValue before the first push is 0 / 0
// (RealTimeAnalyser.h:87), hop count 0
void publish_empty (fx_group& g, int local_track)
{
    float nanv = NAN;
    uint32_t nb; memcpy (&nb, &nanv, 4);
    g.latest.write_begin();
    for (size_t k = 0; k < FX_NUM_FEATURES; ++k) g.latest.put ((size_t) local_track * kLatestWords + k, nb);
    g.latest.put ((size_t) local_track * kLatestWords + FX_NUM_FEATURES, 0u);
    g.latest.put ((size_t) local_track * kLatestWords + FX_NUM_FEATURES + 1, 0u);
    g.latest.write_end();
}

fx_status clear_state (fx_engine* e, cudaStream_t s)
{
    const size_t T = (size_t) e->cfg.n_tracks;
    for (int i = 0; i < 2; ++i)
    {
        FX_CUDA (e, cudaMemsetAsync (e->d_tail[i], 0, T * (size_t) (e->N - e->H) * sizeof (float), s));
        FX_CUDA (e, cudaMemsetAsync (e->d_prev[i], 0, T * (size_t) e->M * sizeof (float), s));
        FX_CUDA (e, cudaMemsetAsync (e->d_hrows[i], 0, T * kHistRows * FX_NUM_FEATURES * sizeof (float), s));
    }
    FX_CUDA (e, cudaMemsetAsync (e->d_latest, 0, T * kLatestWords * sizeof (float), s));
    for (auto& g : e->groups)
    {
        g->flip = 0; g->frames_done = 0; g->params_dirty = true; g->ratio_pending = false;
        for (int t = 0; t < g->n; ++t) publish_empty (*g, t);
    }
    std::fill (e->h_ratio.begin(), e->h_ratio.end(), 1.0f);
    return FX_OK;
}

// The offline calls treat all tracks as one stream position: the groups must be in step (they are unless the real-time path
// advanced them independently).
bool groups_in_step (const fx_engine* e)
{
    for (auto& g : e->groups)
        if (g->flip != e->groups[0]->flip || g->frames_done != e->groups[0]->frames_done) return false;
    return true;
}

struct AllGroupsLock      // the batch mutexes of every group, in index order (the workers only ever hold their own)
{
    explicit AllGroupsLock (fx_engine* e_) : e (e_) { for (auto& g : e->groups) g->batch_mutex.lock(); }
    ~AllGroupsLock() { for (size_t i = e->groups.size(); i-- > 0;) e->groups[i]->batch_mutex.unlock(); }
    fx_engine* e;
};

// settle what the parameter calls left for the next analysed hop, for every group, on `s` (offline calls)
fx_status settle_params_offline (fx_engine* e, cudaStream_t s)
{
    for (auto& g : e->groups)
    {
        if (g->params_dirty)
        {
            fx_status st = upload_params (e, g->t0, g->n, s);
            if (st != FX_OK) return st;
            g->params_dirty = false;
        }
        if (g->ratio_pending)
        {
            fx_status st = apply_gain_ratio (e, g->t0, g->n, g->flip, s);
            if (st != FX_OK) return st;
            g->ratio_pending = false;
        }
    }
    return FX_OK;
}

fx_status offline_begin (fx_engine* e, cudaStream_t s)
{
    if (e->rt_running.load()) { set_error (e, "the real-time workers are running (fx_rt_stop first)"); return FX_ERR_INVALID_ARG; }
    if (! groups_in_step (e)) { set_error (e, "track groups are out of step (the real-time path advanced them independently): fx_reset first"); return FX_ERR_INVALID_ARG; }
    // carried state written by the previous offline call, possibly on another stream
    FX_CUDA (e, cudaStreamWaitEvent (s, e->ev_last, 0));
    return settle_params_offline (e, s);
}

fx_status offline_end (fx_engine* e, cudaStream_t s, long frames)
{
    FX_CUDA (e, cudaEventRecord (e->ev_last, s));
    for (auto& g : e->groups) { g->flip ^= 1; g->frames_done += frames; }
    return FX_OK;
}

// ---- one pass of the real-time path over one group ------------------------------------------------------------------
// rt_issue: everything up to the download of the smoothed vectors is queued on the group's stream; rt_finish waits for it,
// releases the ring space and publishes.  Both run with the group's batch mutex held.
fx_status rt_issue (fx_engine* e, fx_group& g, long* hops_out)
{
    *hops_out = 0;
    const long H = e->H, L = e->ring_len;
    const long gi = g.t0 / e->rings.per;
    long hops = e->rings.hops_available (gi, g.t0, g.n, H);
    if (hops > e->stage_hops) hops = e->stage_hops;
    if (hops <= 0) return FX_OK;
    const long r = e->rings.read_pos (gi);
    const long n = hops * H;

    // fx_clear_buffer: samples pushed before the request become zeros (AudioDataCollector.h:122); they are published and
    // not yet released, so only this thread touches them
    for (int t = g.t0; t < g.t0 + g.n; ++t) e->rings.apply_clear (t, r, n);

    if (g.params_dirty)
    {
        fx_status st = upload_params (e, g.t0, g.n, g.stream);
        if (st != FX_OK) return st;
        g.params_dirty = false;
    }
    if (g.ratio_pending)
    {
        fx_status st = apply_gain_ratio (e, g.t0, g.n, g.flip, g.stream);
        if (st != FX_OK) return st;
        g.ratio_pending = false;
    }

    const long o = r % L;
    const long first = (o + n <= L) ? n : L - o;
    const float* src = e->h_ring + (size_t) g.t0 * (size_t) L;
    FX_CUDA (e, cudaMemcpy2DAsync (g.d_stage, (size_t) n * sizeof (float), src + o, (size_t) L * sizeof (float),
                                    (size_t) first * sizeof (float), (size_t) g.n, cudaMemcpyHostToDevice, g.stream));
    if (first < n)
        FX_CUDA (e, cudaMemcpy2DAsync (g.d_stage + first, (size_t) n * sizeof (float), src, (size_t) L * sizeof (float),
                                        (size_t) (n - first) * sizeof (float), (size_t) g.n, cudaMemcpyHostToDevice, g.stream));
    int n_chunks = choose_chunks (e, g.n, hops);
    if (n_chunks > g.max_chunks) n_chunks = g.max_chunks;
    fx_status st = run_range (e, g.t0, g.n, n_chunks, g.flip, g.frames_done, g.scratch, g.d_stage, n, hops, g.d_raw, g.d_smooth,
                              nullptr, nullptr, e->d_latest + (size_t) g.t0 * kLatestWords, g.stream, false);
    if (st != FX_OK) return st;
    FX_CUDA (e, cudaMemcpyAsync (g.h_latest, e->d_latest + (size_t) g.t0 * kLatestWords,
                                  (size_t) g.n * kLatestWords * sizeof (float), cudaMemcpyDeviceToHost, g.stream));
    *hops_out = hops;
    return FX_OK;
}

fx_status rt_finish (fx_engine* e, fx_group& g, long hops)
{
    if (hops <= 0) return FX_OK;
    FX_CUDA (e, cudaStreamSynchronize (g.stream));
    e->rings.consumed (g.t0 / e->rings.per, hops * e->H);          // the producers may overwrite these samples from here on
    g.flip ^= 1;
    g.frames_done += hops;
    const uint32_t* w = reinterpret_cast<const uint32_t*> (g.h_latest);
    g.latest.write_begin();
    for (size_t i = 0; i < (size_t) g.n * kLatestWords; ++i) g.latest.put (i, w[i]);
    g.latest.write_end();
    return FX_OK;
}

void rt_note_batch (fx_engine* e, long hops, std::chrono::steady_clock::time_point t0)
{
    const uint64_t ns = (uint64_t) std::chrono::duration_cast<std::chrono::nanoseconds> (std::chrono::steady_clock::now() - t0).count();
    e->st_batches.fetch_add (1, std::memory_order_relaxed);
    e->st_hops.fetch_add ((uint64_t) hops, std::memory_order_relaxed);
    e->st_ns_sum.fetch_add (ns, std::memory_order_relaxed);
    uint64_t m = e->st_ns_max.load (std::memory_order_relaxed);
    while (ns > m && ! e->st_ns_max.compare_exchange_weak (m, ns, std::memory_order_relaxed)) {}
}

void rt_worker_main (fx_engine* e, fx_group* g)
{
    if (cudaSetDevice (e->cfg.device) != cudaSuccess) { g->worker_error = "cudaSetDevice failed on the worker thread"; g->worker_status.store (FX_ERR_CUDA); return; }
    while (! e->rt_stop.load (std::memory_order_acquire))
    {
        const uint32_t ticket = g->wake.observe();
        long hops = 0;
        fx_status st;
        uint64_t frame_index = 0;
        const auto t0 = std::chrono::steady_clock::now();
        {
            std::lock_guard<std::mutex> lk (g->batch_mutex);
            st = rt_issue (e, *g, &hops);
            if (st == FX_OK) st = rt_finish (e, *g, hops);
            frame_index = (uint64_t) g->frames_done;
        }
        if (st != FX_OK)
        {
            { std::lock_guard<std::mutex> lk (e->err_mutex); g->worker_error = e->err; }
            g->worker_status.store (st);
            return;
        }
        if (hops > 0)
        {
            rt_note_batch (e, hops, t0);
            if (e->cb) e->cb (e->cb_user, g->t0, g->n, frame_index, (int) hops);
        }
        else
            g->wake.wait (ticket, 100);
    }
}

fx_status rebuild_rate_tables (fx_engine* e, double sample_rate, bool allocate)
{
    std::vector<short> her_tab;
    build_lag_tables (e->N, sample_rate, her_tab);
    for (int k = 0; k < 16 && (1 << k) <= e->N; ++k) e->f0bin_pow2[k] = her_tab[(size_t) (1 << k) * FX_HER_TAB_STRIDE + 18];
    std::vector<double> ex_tab; std::vector<int> ex_off;
    build_exact_ratio_table (e->N, sample_rate, ex_tab, ex_off);
    if (allocate)
    {
        FX_CUDA (e, cudaMalloc (&e->d_ex_tab, ex_tab.size() * sizeof (double)));
        FX_CUDA (e, cudaMalloc (&e->d_ex_off, ex_off.size() * sizeof (int)));
        FX_CUDA (e, cudaMalloc (&e->d_her_tab, her_tab.size() * sizeof (short)));
        e->ex_tab_len = ex_tab.size();
    }
    else if (ex_tab.size() != e->ex_tab_len) { set_error (e, "exact-ratio table changed size"); return FX_ERR_CUDA; }    // its layout depends on the window only
    FX_CUDA (e, cudaMemcpy (e->d_ex_tab, ex_tab.data(), ex_tab.size() * sizeof (double), cudaMemcpyHostToDevice));
    FX_CUDA (e, cudaMemcpy (e->d_ex_off, ex_off.data(), ex_off.size() * sizeof (int), cudaMemcpyHostToDevice));
    FX_CUDA (e, cudaMemcpy (e->d_her_tab, her_tab.data(), her_tab.size() * sizeof (short), cudaMemcpyHostToDevice));
    return FX_OK;
}

} // namespace

extern "C" {

void fx_default_config (fx_config* c)
{
    c->n_tracks = 1;
    c->window = 2048;                 // AnalyserTrackController.h:20-21
    c->hop = 1024;                    // RealTimeAudioAnalysis.h:207
    c->sample_rate = 48000.0;         // RealTimeAnalyser.h:100
    c->device = 0;
    c->rms_pushes_per_frame = 2;      // RealTimeAnalyser.h:150,209
    c->onset_type = 1;                // SpectralCharacteristics.h:240
    c->onset_hist = 5;                // SpectralCharacteristics.h:238-239
    c->onset_multiplier = 1.7f;       // SpectralCharacteristics.h:311
    c->gain = 1.0f;                   // AudioDataCollector.h:129
    c->max_frames_per_call = 0;       // grow on demand
    c->ring_hops = 16;
    c->tracks_per_group = 0;
    c->spectrum = FX_SPECTRUM_RE_SQUARED;   // the reference's Re(X)^2
}

const char* fx_version (void) { return "fxb200 0.2 (sm_100a)"; }

const char* fx_last_error (const fx_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

fx_status fx_engine_create (const fx_config* cfg, fx_engine** out)
{
    if (! cfg || ! out) { g_create_error = "null argument"; return FX_ERR_INVALID_ARG; }
    *out = nullptr;
    const int N = cfg->window, H = cfg->hop;
    if (N != 1024 && N != 2048 && N != 4096) { g_create_error = "window must be 1024, 2048 or 4096"; return FX_ERR_UNSUPPORTED; }
    if (H < 16 || H > N || (N % H) != 0 || (H & (H - 1)) != 0) { g_create_error = "hop must be a power of two >= 16 dividing the window"; return FX_ERR_UNSUPPORTED; }
    if (cfg->n_tracks < 1) { g_create_error = "n_tracks must be >= 1"; return FX_ERR_INVALID_ARG; }
    if (cfg->onset_hist < 1 || cfg->onset_hist > kMaxOnsetHist) { g_create_error = "onset_hist must be in 1..16"; return FX_ERR_INVALID_ARG; }
    if (cfg->rms_pushes_per_frame != 1 && cfg->rms_pushes_per_frame != 2) { g_create_error = "rms_pushes_per_frame must be 1 or 2"; return FX_ERR_INVALID_ARG; }
    if (cfg->ring_hops < 0 || cfg->tracks_per_group < 0) { g_create_error = "ring_hops and tracks_per_group must be >= 0"; return FX_ERR_INVALID_ARG; }
    if (! (cfg->sample_rate > 0.0)) { g_create_error = "sample_rate must be positive"; return FX_ERR_INVALID_ARG; }
    if (cfg->spectrum != FX_SPECTRUM_RE_SQUARED && cfg->spectrum != FX_SPECTRUM_POWER) { g_create_error = "spectrum must be FX_SPECTRUM_RE_SQUARED or FX_SPECTRUM_POWER"; return FX_ERR_INVALID_ARG; }

    int ndev = 0;
    if (cudaGetDeviceCount (&ndev) != cudaSuccess || ndev == 0) { g_create_error = "no CUDA device (this library has no CPU fallback)"; return FX_ERR_NO_DEVICE; }
    if (cfg->device < 0 || cfg->device >= ndev) { g_create_error = "device ordinal out of range"; return FX_ERR_INVALID_ARG; }

    fx_engine* e = new fx_engine();
    e->cfg = *cfg; e->N = N; e->H = H; e->M = N / 2; e->NB = N / H; e->log2_hop = ilog2 (H);
    e->ctas_per_sm = analyse_ctas_per_sm (N);
    const size_t T = (size_t) cfg->n_tracks;

#define FX_CREATE(call) do { cudaError_t ce_ = (call); if (ce_ != cudaSuccess) { set_error (nullptr, #call, ce_); free_engine (e); return FX_ERR_CUDA; } } while (0)
#define FX_CREATE_ST(call) do { if ((call) != FX_OK) { g_create_error = e->err; free_engine (e); return FX_ERR_CUDA; } } while (0)
    FX_CREATE (cudaSetDevice (cfg->device));
    cudaDeviceProp prop{};
    FX_CREATE (cudaGetDeviceProperties (&prop, cfg->device));
    e->sm_count = prop.multiProcessorCount;
    FX_CREATE (configure_analyse (N));
    FX_CREATE (cudaStreamCreateWithFlags (&e->stream, cudaStreamNonBlocking));
    FX_CREATE (cudaEventCreateWithFlags (&e->ev_last, cudaEventDisableTiming));

    std::vector<float2> tw2, tw1f;
    build_twiddles (N, tw2, tw1f);
    FX_CREATE (cudaMalloc (&e->d_tw2, tw2.size() * sizeof (float2)));
    FX_CREATE (cudaMemcpy (e->d_tw2, tw2.data(), tw2.size() * sizeof (float2), cudaMemcpyHostToDevice));
    FX_CREATE (cudaMalloc (&e->d_tw1f, tw1f.size() * sizeof (float2)));
    FX_CREATE (cudaMemcpy (e->d_tw1f, tw1f.data(), tw1f.size() * sizeof (float2), cudaMemcpyHostToDevice));
    FX_CREATE_ST (rebuild_rate_tables (e, cfg->sample_rate, true));

    // SpectralCharacteristics.h:180-189: binVar accumulated sequentially in double
    {
        double bv = 0.0;
        const int M = e->M;
        for (double i = 0.0; i < M; i++) { const double ni = i / (double) M; bv += (ni - 0.5) * (ni - 0.5); }
        e->bin_var = bv / (double) M;
    }
    // RealTimeAudioAnalysis.h:122,127: (float_Pi / m) and exp (-float_Pi / m), m = 2, in fp32
    {
        const float pi_f = 3.14159265358979323846f, m = 2.0f;
        e->iir_c1 = pi_f / m;
        e->iir_c2 = expf (-pi_f / m);
    }

    e->h_gain.assign (T, cfg->gain); e->h_mult.assign (T, cfg->onset_multiplier); e->h_ratio.assign (T, 1.0f);
    e->h_type.assign (T, cfg->onset_type); e->h_hist.assign (T, cfg->onset_hist); e->h_reset.assign (T, 0); e->h_start.assign (T, 0);
    FX_CREATE (cudaMalloc (&e->d_gain, T * sizeof (float)));
    FX_CREATE (cudaMalloc (&e->d_mult, T * sizeof (float)));
    FX_CREATE (cudaMalloc (&e->d_ratio, T * sizeof (float)));
    FX_CREATE (cudaMalloc (&e->d_type, T * sizeof (int)));
    FX_CREATE (cudaMalloc (&e->d_hist, T * sizeof (int)));
    FX_CREATE (cudaMalloc (&e->d_reset, T * sizeof (long)));
    FX_CREATE (cudaMalloc (&e->d_start, T * sizeof (long)));
    for (int i = 0; i < 2; ++i)
    {
        FX_CREATE (cudaMalloc (&e->d_tail[i], T * (size_t) (N - H + 4) * sizeof (float)));
        FX_CREATE (cudaMalloc (&e->d_prev[i], T * (size_t) e->M * sizeof (float)));
        FX_CREATE (cudaMalloc (&e->d_hrows[i], T * kHistRows * FX_NUM_FEATURES * sizeof (float)));
    }
    FX_CREATE (cudaMalloc (&e->d_latest, T * kLatestWords * sizeof (float)));
    FX_CREATE (cudaHostAlloc (&e->h_latest, T * kLatestWords * sizeof (float), cudaHostAllocDefault));
    memset (e->h_latest, 0, T * kLatestWords * sizeof (float));

    // track groups: the unit of the real-time path (one stream, one worker, one ring read position each) and of the
    // carried-state bookkeeping
    {
        int per = cfg->tracks_per_group > 0 ? cfg->tracks_per_group : cfg->n_tracks;
        if ((cfg->n_tracks + per - 1) / per > kMaxGroups) per = (cfg->n_tracks + kMaxGroups - 1) / kMaxGroups;
        e->rt_enabled = cfg->ring_hops > 0;
        const int rh = cfg->ring_hops >= e->NB + 2 ? cfg->ring_hops : e->NB + 2;
        e->ring_len = (long) rh * H;
        e->stage_hops = rh;
        if (e->rt_enabled)
        {
            FX_CREATE (cudaHostAlloc (&e->h_ring, T * (size_t) e->ring_len * sizeof (float), cudaHostAllocDefault));
            memset (e->h_ring, 0, T * (size_t) e->ring_len * sizeof (float));
            e->rings.init (e->h_ring, (long) T, e->ring_len, per);
        }
        for (int t0 = 0; t0 < cfg->n_tracks; t0 += per)
        {
            std::unique_ptr<fx_group> g (new fx_group());
            g->t0 = t0; g->n = (t0 + per <= cfg->n_tracks) ? per : cfg->n_tracks - t0;
            g->latest.init ((size_t) g->n * kLatestWords);
            g->h_latest = e->h_latest + (size_t) t0 * kLatestWords;
            fx_group* gp = g.get();
            e->groups.push_back (std::move (g));
            if (! e->rt_enabled) continue;
            const size_t rows = (size_t) gp->n * (size_t) e->stage_hops;
            gp->max_chunks = (int) ((e->stage_hops + 7) / 8);
            FX_CREATE (cudaStreamCreateWithFlags (&gp->stream, cudaStreamNonBlocking));
            FX_CREATE (cudaMalloc (&gp->d_stage, rows * H * sizeof (float)));
            FX_CREATE (cudaMalloc (&gp->d_raw, rows * FX_NUM_FEATURES * sizeof (float)));
            FX_CREATE (cudaMalloc (&gp->d_smooth, rows * FX_NUM_FEATURES * sizeof (float)));
            FX_CREATE (cudaMalloc (&gp->scratch.rec, rows * fx::frame_rec_bytes (e->N)));
            const size_t pairs = (size_t) gp->n * (size_t) gp->max_chunks;
            FX_CREATE (cudaMalloc (&gp->scratch.first_spec, pairs * e->M * sizeof (float)));
            FX_CREATE (cudaMalloc (&gp->scratch.last_spec,  pairs * e->M * sizeof (float)));
            FX_CREATE (cudaMalloc (&gp->scratch.first_idx,  pairs * sizeof (int)));
        }
    }
    FX_CREATE_ST (clear_state (e, e->stream));
    FX_CREATE (cudaEventRecord (e->ev_last, e->stream));
    if (cfg->max_frames_per_call > 0)
    {
        FX_CREATE_ST (ensure_results (e, cfg->max_frames_per_call));
        FX_CREATE_ST (ensure_records (e, cfg->max_frames_per_call));
    }
    FX_CREATE (cudaStreamSynchronize (e->stream));
#undef FX_CREATE
#undef FX_CREATE_ST
    *out = e;
    return FX_OK;
}

fx_status fx_engine_destroy (fx_engine* e)
{
    free_engine (e);
    return FX_OK;
}

// ---- runtime parameter surface ---------------------------------------------------------------------------------
fx_status fx_set_gain (fx_engine* e, int track, float gain)
{
    if (! e || track < -1 || track >= e->cfg.n_tracks) return FX_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> api (e->api_mutex);
    const int a = track < 0 ? 0 : track, b = track < 0 ? e->cfg.n_tracks : track + 1;
    for (auto& g : e->groups)
    {
        if (g->t0 >= b || g->t0 + g->n <= a) continue;
        std::lock_guard<std::mutex> lk (g->batch_mutex);
        for (int t = (a > g->t0 ? a : g->t0); t < b && t < g->t0 + g->n; ++t)
        {
            const float old = e->h_gain[(size_t) t];
            if (old == gain) continue;
            // the samples already collected keep the gain they were collected with (AudioDataCollector.h:88); a gain of
            // exactly zero cannot be carried through the rescaling: the overlap then counts as silence
            e->h_ratio[(size_t) t] = (gain == 0.0f || old == 0.0f) ? 0.0f : e->h_ratio[(size_t) t] * (old / gain);
            e->h_gain[(size_t) t] = gain;
            g->params_dirty = true;
            g->ratio_pending = true;
        }
    }
    return FX_OK;
}

fx_status fx_set_onset (fx_engine* e, int track, int type, int hist_len, float multiplier)
{
    if (! e || track < -1 || track >= e->cfg.n_tracks) return FX_ERR_INVALID_ARG;
    if (type < 0 || type > 2 || hist_len < 1 || hist_len > kMaxOnsetHist) { set_error (e, "onset type must be 0..2 and hist_len 1..16"); return FX_ERR_INVALID_ARG; }
    std::lock_guard<std::mutex> api (e->api_mutex);
    const int a = track < 0 ? 0 : track, b = track < 0 ? e->cfg.n_tracks : track + 1;
    for (auto& g : e->groups)
    {
        if (g->t0 >= b || g->t0 + g->n <= a) continue;
        std::lock_guard<std::mutex> lk (g->batch_mutex);
        for (int t = (a > g->t0 ? a : g->t0); t < b && t < g->t0 + g->n; ++t)
        {
            e->h_type[(size_t) t] = type;
            e->h_mult[(size_t) t] = multiplier;
            if (e->h_hist[(size_t) t] != hist_len)
            {
                // RealTimeSpectralAnalyser::setOnsetWindowLength -> ValueHistory::setHistoryLength clears (RealTimeAudioAnalysis.h:73-81)
                e->h_hist[(size_t) t] = hist_len;
                e->h_reset[(size_t) t] = g->frames_done;
            }
        }
        g->params_dirty = true;
    }
    return FX_OK;
}

fx_status fx_set_sample_rate (fx_engine* e, double sample_rate)
{
    if (! e || ! (sample_rate > 0.0)) return FX_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> api (e->api_mutex);
    if (sample_rate == e->cfg.sample_rate) return FX_OK;
    FX_CUDA (e, cudaSetDevice (e->cfg.device));
    AllGroupsLock all (e);                                   // between two batches of every group = at a hop boundary
    FX_CUDA (e, cudaEventSynchronize (e->ev_last));          // and after the last offline call's kernels
    fx_status st = rebuild_rate_tables (e, sample_rate, false);
    if (st != FX_OK) return st;
    e->cfg.sample_rate = sample_rate;
    return FX_OK;
}

fx_status fx_set_track_active (fx_engine* e, int track, int active, int reset_state)
{
    if (! e || track < -1 || track >= e->cfg.n_tracks) return FX_ERR_INVALID_ARG;
    if (! e->rt_enabled) { set_error (e, "the engine was created without the real-time path (ring_hops = 0)"); return FX_ERR_INVALID_ARG; }
    std::lock_guard<std::mutex> api (e->api_mutex);
    FX_CUDA (e, cudaSetDevice (e->cfg.device));
    const int a = track < 0 ? 0 : track, b = track < 0 ? e->cfg.n_tracks : track + 1;
    for (auto& g : e->groups)
    {
        if (g->t0 >= b || g->t0 + g->n <= a) continue;
        std::lock_guard<std::mutex> lk (g->batch_mutex);
        for (int t = (a > g->t0 ? a : g->t0); t < b && t < g->t0 + g->n; ++t)
        {
            const size_t ts = (size_t) t;
            if (! active) { e->rings.deactivate (t); continue; }       // from here on the track is fed silence
            if (reset_state)
            {
                // a freshly constructed AnalyserTrackController: zero overlap buffer (RealTimeAudioAnalysis.h:202), zero
                // previous spectrum (SpectralCharacteristics.h:34-38), empty feature / onset histories (RealTimeAnalyser.h:70-74)
                FX_CUDA (e, cudaMemsetAsync (e->d_tail[g->flip] + ts * (size_t) (e->N - e->H), 0, (size_t) (e->N - e->H) * sizeof (float), g->stream));
                FX_CUDA (e, cudaMemsetAsync (e->d_prev[g->flip] + ts * (size_t) e->M, 0, (size_t) e->M * sizeof (float), g->stream));
                FX_CUDA (e, cudaStreamSynchronize (g->stream));
                e->h_start[ts] = g->frames_done;
                e->h_ratio[ts] = 1.0f;
                g->params_dirty = true;
                publish_empty (*g, t - g->t0);
            }
            e->rings.activate (t);                                      // its stream starts at the group's read position
        }
    }
    return FX_OK;
}

fx_status fx_clear_buffer (fx_engine* e, int track)
{
    if (! e || track < -1 || track >= e->cfg.n_tracks) return FX_ERR_INVALID_ARG;
    if (! e->rt_enabled) return FX_OK;
    const int a = track < 0 ? 0 : track, b = track < 0 ? e->cfg.n_tracks : track + 1;
    for (int t = a; t < b; ++t) e->rings.request_clear (t);
    return FX_OK;
}

fx_status fx_reset (fx_engine* e)
{
    if (! e) return FX_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> api (e->api_mutex);
    FX_CUDA (e, cudaSetDevice (e->cfg.device));
    AllGroupsLock all (e);
    FX_CUDA (e, cudaDeviceSynchronize());
    fx_status st = clear_state (e, e->stream);
    if (st != FX_OK) return st;
    std::fill (e->h_reset.begin(), e->h_reset.end(), 0L);
    std::fill (e->h_start.begin(), e->h_start.end(), 0L);
    if (e->rt_enabled) e->rings.reset();
    FX_CUDA (e, cudaEventRecord (e->ev_last, e->stream));
    FX_CUDA (e, cudaStreamSynchronize (e->stream));
    return FX_OK;
}

// ---- offline / batch analysis ------------------------------------------------------------------------------------
fx_status fx_analyse_device_spectrum (fx_engine* e, const float* d_audio, long track_stride, long n_samples,
                                      float* d_raw, float* d_smooth, float* d_diag, float* d_spec, void* stream, long* n_frames)
{
    if (! e || ! d_audio || n_samples < 0 || track_stride < n_samples) return FX_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> api (e->api_mutex);
    if (((uintptr_t) d_spec & 15u) != 0) { set_error (e, "d_spec must be 16-byte aligned"); return FX_ERR_INVALID_ARG; }      // K1 stores 16-byte vectors
    FX_CUDA (e, cudaSetDevice (e->cfg.device));
    cudaStream_t s = stream ? (cudaStream_t) stream : e->stream;
    const long frames = n_samples / e->H;
    if (n_frames) *n_frames = frames;
    if (frames == 0) return FX_OK;
    if (frames > 0x7fffffffL / (FX_NUM_FEATURES * 4)) { set_error (e, "too many frames in one call"); return FX_ERR_INVALID_ARG; }
    const long T = e->cfg.n_tracks;
    // K1 indexes the spectrum rows in 64 bits: T * frames * M floats must have a byte size that a long holds
    if (d_spec && T * frames > 0x7fffffffffffffffL / ((long) e->M * (long) sizeof (float)))
    {
        set_error (e, "the spectrum output is too large for one call"); return FX_ERR_INVALID_ARG;
    }
    fx_status st = offline_begin (e, s);
    if (st != FX_OK) return st;
    const int n_chunks = choose_chunks (e, T, frames);
    st = ensure_chunks (e, T * n_chunks);
    if (st != FX_OK) return st;
    st = ensure_records (e, frames);
    if (st != FX_OK) return st;
    if (! d_raw)
    {
        st = ensure_results (e, frames);
        if (st != FX_OK) return st;
        d_raw = e->d_raw;
    }
    st = run_range (e, 0, (int) T, n_chunks, e->groups[0]->flip, e->groups[0]->frames_done, offline_scratch (e, 0, frames, n_chunks),
                    d_audio, track_stride, frames, d_raw, d_smooth, d_diag, d_spec, e->d_latest, s, true);
    if (st != FX_OK) return st;
    return offline_end (e, s, frames);
}

fx_status fx_analyse_device (fx_engine* e, const float* d_audio, long track_stride, long n_samples,
                             float* d_raw, float* d_smooth, float* d_diag, void* stream, long* n_frames)
{
    return fx_analyse_device_spectrum (e, d_audio, track_stride, n_samples, d_raw, d_smooth, d_diag, nullptr, stream, n_frames);
}

namespace {

// Shared body of fx_analyse_host / fx_analyse_host_pcm.  format == 0: `src` is fp32, row stride in bytes = 4 * track_stride.
fx_status analyse_host_pipeline (fx_engine* e, const unsigned char* src, long row_stride_bytes, int format, int n_channels, int channel,
                                 long frames, float* raw, float* smooth, float* diag)
{
    const long T = e->cfg.n_tracks;
    const long used = frames * e->H;                                  // samples per track actually analysed
    const long frame_bytes = format ? (long) n_channels * pcm_bytes_per_sample (format) : (long) sizeof (float);
    const long row_bytes = used * frame_bytes;                        // source bytes per track that cross PCIe
    const bool shared_row = format != 0 && row_stride_bytes == 0;     // every track reads the same interleaved stream

    // Track groups: about fifty per call (the first group's upload and the last group's analysis are the only parts of
    // the pipeline that do not overlap), but never below ~64 MiB of fp32 audio -- small groups would have to cut every
    // track into short chunks to fill the GPU, and each chunk start refills a whole window
    const long want_groups = 48;
    long per = (T + want_groups - 1) / want_groups;
    const long per_min = (64L << 20) / (used * (long) sizeof (float));
    if (per < per_min) per = per_min;
    if (per < 1) per = 1;
    if (per > T) per = T;
    const long n_groups = (T + per - 1) / per;
    const long slot_floats = per * used;
    if (slot_floats > e->audio_slot_floats)
    {
        FX_CUDA (e, cudaDeviceSynchronize());
        for (int i = 0; i < 3; ++i) { cudaFree (e->d_audio_slot[i]); e->d_audio_slot[i] = nullptr; }
        e->audio_slot_floats = 0;
        for (int i = 0; i < 3; ++i) FX_CUDA (e, cudaMalloc (&e->d_audio_slot[i], (size_t) slot_floats * sizeof (float)));
        e->audio_slot_floats = slot_floats;
    }
    // PCM rows keep a 16-byte aligned pitch on the device so that the vector decode path applies whenever the format allows
    const long pcm_pitch = (row_bytes + 15) & ~15L;
    if (format && per * pcm_pitch > e->pcm_slot_bytes)
    {
        FX_CUDA (e, cudaDeviceSynchronize());
        for (int i = 0; i < 3; ++i) { cudaFree (e->d_pcm_slot[i]); e->d_pcm_slot[i] = nullptr; }
        e->pcm_slot_bytes = 0;
        for (int i = 0; i < 3; ++i) FX_CUDA (e, cudaMalloc (&e->d_pcm_slot[i], (size_t) (per * pcm_pitch)));
        e->pcm_slot_bytes = per * pcm_pitch;
    }
    for (int i = 0; i < 3; ++i)
        if (! e->pipe_stream[i]) FX_CUDA (e, cudaStreamCreateWithFlags (&e->pipe_stream[i], cudaStreamNonBlocking));

    fx_status st = offline_begin (e, e->stream);
    if (st != FX_OK) return st;
    FX_CUDA (e, cudaStreamSynchronize (e->stream));
    st = ensure_results (e, frames);
    if (st != FX_OK) return st;
    st = ensure_records (e, frames);
    if (st != FX_OK) return st;
    const int n_chunks = choose_chunks (e, per, frames);
    st = ensure_chunks (e, T * n_chunks);
    if (st != FX_OK) return st;
    const int flip = e->groups[0]->flip;
    const long frames_done = e->groups[0]->frames_done;

    // Three streams, three slots: uploads, kernels and result downloads each run in group order on their own stream and
    // meet through events, so that group g + 1's upload overlaps group g's analysis and the analysis kernels run back to
    // back.  (Launching each group on its own stream lets the hardware interleave the CTAs of three analysis kernels: all
    // three then finish together, their slots free together, and every third upload is exposed.)
    cudaStream_t s_up = e->pipe_stream[0], s_run = e->pipe_stream[1], s_down = e->pipe_stream[2];
    for (int i = 0; i < 3; ++i)
    {
        if (! e->ev_ready[i]) FX_CUDA (e, cudaEventCreateWithFlags (&e->ev_ready[i], cudaEventDisableTiming));
        if (! e->ev_free[i])  FX_CUDA (e, cudaEventCreateWithFlags (&e->ev_free[i], cudaEventDisableTiming));
    }
    // FXB200_PIPE_TRACE=1: per-group device timeline of the pipeline on stderr (diagnostics)
    const bool trace = getenv ("FXB200_PIPE_TRACE") != nullptr;
    std::vector<cudaEvent_t> tev;
    auto mark = [&] (cudaStream_t st_) { if (trace) { cudaEvent_t ev; cudaEventCreate (&ev); cudaEventRecord (ev, st_); tev.push_back (ev); } };
    for (long g = 0; g < n_groups; ++g)
    {
        const int slot = (int) (g % 3);
        const long t0 = g * per, nt = (t0 + per <= T) ? per : T - t0;
        // upload: the slot's previous occupant (group g - 3) must have been analysed
        if (g >= 3) FX_CUDA (e, cudaStreamWaitEvent (s_up, e->ev_free[slot], 0));
        mark (s_up);
        if (format == 0 && row_stride_bytes == row_bytes)      // contiguous rows: one linear copy
            FX_CUDA (e, cudaMemcpyAsync (e->d_audio_slot[slot], src + t0 * row_stride_bytes, (size_t) row_bytes * (size_t) nt, cudaMemcpyHostToDevice, s_up));
        else if (format == 0)
            FX_CUDA (e, cudaMemcpy2DAsync (e->d_audio_slot[slot], (size_t) row_bytes, src + t0 * row_stride_bytes, (size_t) row_stride_bytes,
                                            (size_t) row_bytes, (size_t) nt, cudaMemcpyHostToDevice, s_up));
        else if (shared_row)       // one interleaved stream feeds every track (track t <- channel t % n_channels): upload it once per group
            FX_CUDA (e, cudaMemcpyAsync (e->d_pcm_slot[slot], src, (size_t) row_bytes, cudaMemcpyHostToDevice, s_up));
        else if (row_stride_bytes == row_bytes && pcm_pitch == row_bytes)
            FX_CUDA (e, cudaMemcpyAsync (e->d_pcm_slot[slot], src + t0 * row_stride_bytes, (size_t) row_bytes * (size_t) nt, cudaMemcpyHostToDevice, s_up));
        else
            FX_CUDA (e, cudaMemcpy2DAsync (e->d_pcm_slot[slot], (size_t) pcm_pitch, src + t0 * row_stride_bytes, (size_t) row_stride_bytes,
                                            (size_t) row_bytes, (size_t) nt, cudaMemcpyHostToDevice, s_up));
        mark (s_up);
        FX_CUDA (e, cudaEventRecord (e->ev_ready[slot], s_up));
        // analysis
        FX_CUDA (e, cudaStreamWaitEvent (s_run, e->ev_ready[slot], 0));
        if (format != 0)
        {
            PcmParams pp{};
            pp.pcm = e->d_pcm_slot[slot]; pp.track_stride_bytes = shared_row ? 0 : pcm_pitch; pp.format = format; pp.n_channels = n_channels;
            pp.channel = channel; pp.first_track = t0;
            pp.n_samples = used; pp.n_tracks = nt; pp.audio = e->d_audio_slot[slot]; pp.audio_stride = used;
            FX_CUDA (e, launch_pcm_decode (pp, s_run));
            e->launches += (uint64_t) pcm_launch_count (pp);
        }
        const size_t roff = (size_t) t0 * (size_t) frames;
        float* dr = e->d_raw + roff * FX_NUM_FEATURES;
        float* ds = e->d_smooth + roff * FX_NUM_FEATURES;
        float* dd = e->d_diag + roff * FX_NUM_DIAG;
        st = run_range (e, (int) t0, (int) nt, n_chunks, flip, frames_done, offline_scratch (e, t0, frames, n_chunks),
                        e->d_audio_slot[slot], used, frames, dr, smooth ? ds : nullptr, diag ? dd : nullptr, nullptr,
                        e->d_latest + (size_t) t0 * kLatestWords, s_run, true);
        if (st != FX_OK) return st;
        mark (s_run);
        FX_CUDA (e, cudaEventRecord (e->ev_free[slot], s_run));
        // results (engine-owned result buffers are indexed by track: no reuse inside a call)
        FX_CUDA (e, cudaStreamWaitEvent (s_down, e->ev_free[slot], 0));
        if (raw)    FX_CUDA (e, cudaMemcpyAsync (raw + roff * FX_NUM_FEATURES, dr, (size_t) nt * frames * FX_NUM_FEATURES * sizeof (float), cudaMemcpyDeviceToHost, s_down));
        if (smooth) FX_CUDA (e, cudaMemcpyAsync (smooth + roff * FX_NUM_FEATURES, ds, (size_t) nt * frames * FX_NUM_FEATURES * sizeof (float), cudaMemcpyDeviceToHost, s_down));
        if (diag)   FX_CUDA (e, cudaMemcpyAsync (diag + roff * FX_NUM_DIAG, dd, (size_t) nt * frames * FX_NUM_DIAG * sizeof (float), cudaMemcpyDeviceToHost, s_down));
        mark (s_down);
    }
    for (int i = 0; i < 3; ++i) FX_CUDA (e, cudaStreamSynchronize (e->pipe_stream[i]));
    if (trace)
    {
        for (size_t i = 0; i + 3 < tev.size(); i += 4)
        {
            float a = 0, b = 0, c = 0, d = 0;
            cudaEventElapsedTime (&a, tev[0], tev[i]); cudaEventElapsedTime (&b, tev[0], tev[i + 1]);
            cudaEventElapsedTime (&c, tev[0], tev[i + 2]); cudaEventElapsedTime (&d, tev[0], tev[i + 3]);
            fprintf (stderr, "pipe group %3zu: upload %8.3f .. %8.3f  analysed %8.3f  results out %8.3f ms\n", i / 4, a, b, c, d);
        }
        for (auto ev : tev) cudaEventDestroy (ev);
    }
    return offline_end (e, s_run, frames);
}

fx_status analyse_host_impl (fx_engine* e, const unsigned char* src, long row_stride_bytes, int format, int n_channels, int channel,
                             long n_samples, float* raw, float* smooth, float* diag, long* n_frames)
{
    std::lock_guard<std::mutex> api (e->api_mutex);
    FX_CUDA (e, cudaSetDevice (e->cfg.device));
    const long frames = n_samples / e->H;
    if (n_frames) *n_frames = frames;
    if (frames == 0) return FX_OK;
    const fx_status st = analyse_host_pipeline (e, src, row_stride_bytes, format, n_channels, channel, frames, raw, smooth, diag);
    if (st != FX_OK)
    {
        // the caller's host buffers may still be the target of queued copies: drain the pipeline before handing them back
        for (int i = 0; i < 3; ++i) if (e->pipe_stream[i]) cudaStreamSynchronize (e->pipe_stream[i]);
        cudaStreamSynchronize (e->stream);
    }
    return st;
}

} // namespace

fx_status fx_analyse_host (fx_engine* e, const float* audio, long track_stride, long n_samples,
                           float* raw, float* smooth, float* diag, long* n_frames)
{
    if (! e || ! audio || n_samples < 0 || track_stride < n_samples) return FX_ERR_INVALID_ARG;
    return analyse_host_impl (e, reinterpret_cast<const unsigned char*> (audio), track_stride * (long) sizeof (float), 0, 1, 0,
                              n_samples, raw, smooth, diag, n_frames);
}

// ---- file ingest ----------------------------------------------------------------------------------------
int fx_pcm_bytes_per_sample (int format) { return fx::pcm_bytes_per_sample (format); }

fx_status fx_analyse_host_pcm (fx_engine* e, const void* pcm, int format, int n_channels, int channel,
                               long track_stride_bytes, long n_samples,
                               float* raw, float* smooth, float* diag, long* n_frames)
{
    const int bps = fx::pcm_bytes_per_sample (format);
    if (! e || ! pcm || n_samples < 0 || n_channels < 1 || channel < -1 || channel >= n_channels) return FX_ERR_INVALID_ARG;
    if (bps == 0) return FX_ERR_UNSUPPORTED;
    if (track_stride_bytes != 0 && track_stride_bytes < n_samples * (long) n_channels * bps) return FX_ERR_INVALID_ARG;
    return analyse_host_impl (e, static_cast<const unsigned char*> (pcm), track_stride_bytes, format, n_channels, channel,
                              n_samples, raw, smooth, diag, n_frames);
}

fx_status fx_decode_pcm_device (fx_engine* e, const void* d_pcm, int format, int n_channels, int channel,
                                long track_stride_bytes, long n_samples, long n_tracks,
                                float* d_audio, long audio_stride, void* stream)
{
    const int bps = fx::pcm_bytes_per_sample (format);
    if (! e || ! d_pcm || ! d_audio || n_samples < 0 || n_tracks < 0 || n_channels < 1 || channel < -1 || channel >= n_channels
        || audio_stride < n_samples) return FX_ERR_INVALID_ARG;
    if (bps == 0) return FX_ERR_UNSUPPORTED;
    if (n_tracks > 1 && track_stride_bytes != 0 && track_stride_bytes < n_samples * (long) n_channels * bps) return FX_ERR_INVALID_ARG;
    FX_CUDA (e, cudaSetDevice (e->cfg.device));
    PcmParams pp{};
    pp.pcm = static_cast<const unsigned char*> (d_pcm); pp.track_stride_bytes = track_stride_bytes; pp.format = format;
    pp.n_channels = n_channels; pp.channel = channel; pp.n_samples = n_samples; pp.n_tracks = n_tracks;
    pp.audio = d_audio; pp.audio_stride = audio_stride;
    FX_CUDA (e, launch_pcm_decode (pp, stream ? static_cast<cudaStream_t> (stream) : e->stream));
    e->launches += (uint64_t) pcm_launch_count (pp);
    return FX_OK;
}

// ---- real-time path ---------------------------------------------------------------------------------------
fx_status fx_push_block (fx_engine* e, int first_track, int n_tracks, const float* const* channels, int n_samples)
{
    if (! e || ! channels || first_track < 0 || n_tracks < 0 || first_track + n_tracks > e->cfg.n_tracks || n_samples < 0 || ! e->rt_enabled)
        return FX_ERR_INVALID_ARG;
    if (n_samples > e->ring_len) return FX_ERR_OVERRUN;
    unsigned char crossed[kMaxGroups];
    const long g0 = e->rings.group_of (first_track), g1 = n_tracks > 0 ? e->rings.group_of (first_track + n_tracks - 1) : g0 - 1;
    for (long g = g0; g <= g1; ++g) crossed[g] = 0;
    const bool ok = e->rings.push (first_track, n_tracks, channels, n_samples, e->H, crossed);
    if (! ok) { e->st_overruns.fetch_add (1, std::memory_order_relaxed); return FX_ERR_OVERRUN; }
    if (e->rt_running.load (std::memory_order_relaxed))
        for (long g = g0; g <= g1; ++g) if (crossed[g]) e->groups[(size_t) g]->wake.signal();
    return FX_OK;
}

fx_status fx_process (fx_engine* e, long* n_new_frames)
{
    if (! e) return FX_ERR_INVALID_ARG;
    if (n_new_frames) *n_new_frames = 0;
    if (! e->rt_enabled) { set_error (e, "the engine was created without the real-time path (ring_hops = 0)"); return FX_ERR_INVALID_ARG; }
    std::lock_guard<std::mutex> api (e->api_mutex);
    if (e->rt_running.load()) { set_error (e, "fx_process while the workers run (fx_rt_stop first)"); return FX_ERR_INVALID_ARG; }
    FX_CUDA (e, cudaSetDevice (e->cfg.device));
    AllGroupsLock all (e);
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<long> hops (e->groups.size(), 0);
    long most = 0, total = 0;
    fx_status st = FX_OK;
    for (size_t i = 0; i < e->groups.size() && st == FX_OK; ++i) st = rt_issue (e, *e->groups[i], &hops[i]);     // every group's work is queued ...
    for (size_t i = 0; i < e->groups.size(); ++i)                                                                  // ... before the first wait
    {
        const fx_status s2 = rt_finish (e, *e->groups[i], hops[i]);
        if (st == FX_OK) st = s2;
        if (hops[i] > most) most = hops[i];
        total += hops[i];
    }
    if (st != FX_OK) return st;
    if (total > 0) rt_note_batch (e, total, t0);
    if (n_new_frames) *n_new_frames = most;
    if (e->cb)
        for (size_t i = 0; i < e->groups.size(); ++i)
            if (hops[i] > 0) e->cb (e->cb_user, e->groups[i]->t0, e->groups[i]->n, (uint64_t) e->groups[i]->frames_done, (int) hops[i]);
    return FX_OK;
}

fx_status fx_rt_start (fx_engine* e)
{
    if (! e) return FX_ERR_INVALID_ARG;
    if (! e->rt_enabled) { set_error (e, "the engine was created without the real-time path (ring_hops = 0)"); return FX_ERR_INVALID_ARG; }
    std::lock_guard<std::mutex> api (e->api_mutex);
    if (e->rt_running.load()) return FX_OK;
    e->rt_stop.store (0);
    for (auto& g : e->groups)
    {
        g->worker_status.store (0);
        g->worker = std::thread (rt_worker_main, e, g.get());
    }
    e->rt_running.store (1);
    return FX_OK;
}

fx_status fx_rt_stop (fx_engine* e)
{
    if (! e) return FX_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> api (e->api_mutex);
    rt_stop_workers (e);
    for (auto& g : e->groups)
        if (g->worker_status.load() != 0) { set_error (e, g->worker_error.c_str()); return (fx_status) g->worker_status.load(); }
    return FX_OK;
}

fx_status fx_set_features_callback (fx_engine* e, fx_features_callback cb, void* user)
{
    if (! e) return FX_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> api (e->api_mutex);
    if (e->rt_running.load()) { set_error (e, "set the features callback before fx_rt_start"); return FX_ERR_INVALID_ARG; }
    e->cb = cb; e->cb_user = user;
    return FX_OK;
}

fx_status fx_rt_get_stats (fx_engine* e, fx_rt_stats* out, int reset)
{
    if (! e || ! out) return FX_ERR_INVALID_ARG;
    out->batches = e->st_batches.load(); out->hops = e->st_hops.load(); out->overruns = e->st_overruns.load();
    out->batch_ms_mean = out->batches ? 1e-6 * (double) e->st_ns_sum.load() / (double) out->batches : 0.0;
    out->batch_ms_max = 1e-6 * (double) e->st_ns_max.load();
    if (reset) { e->st_batches.store (0); e->st_hops.store (0); e->st_overruns.store (0); e->st_ns_sum.store (0); e->st_ns_max.store (0); }
    return FX_OK;
}

fx_status fx_poll_block (fx_engine* e, int first_track, int n_tracks, float* out, uint64_t* frame_index)
{
    if (! e || ! out || first_track < 0 || n_tracks < 0 || first_track + n_tracks > e->cfg.n_tracks) return FX_ERR_INVALID_ARG;
    const int per = e->groups[0]->n;
    for (int i = 0; i < n_tracks;)
    {
        const int t = first_track + i;
        fx_group& g = *e->groups[(size_t) (t / per)];
        int run = g.t0 + g.n - t;
        if (run > n_tracks - i) run = n_tracks - i;
        // one consistent read per group run
        uint32_t w[64 * kLatestWords];
        for (int done = 0; done < run;)
        {
            const int c = run - done < 64 ? run - done : 64;
            g.latest.read ((size_t) (t - g.t0 + done) * kLatestWords, (size_t) c * kLatestWords, w);
            for (int k = 0; k < c; ++k)
            {
                memcpy (out + (size_t) (i + done + k) * FX_NUM_FEATURES, w + (size_t) k * kLatestWords, FX_NUM_FEATURES * sizeof (float));
                if (frame_index)
                    frame_index[i + done + k] = ((uint64_t) w[(size_t) k * kLatestWords + FX_NUM_FEATURES + 1] << 32) | w[(size_t) k * kLatestWords + FX_NUM_FEATURES];
            }
            done += c;
        }
        i += run;
    }
    return FX_OK;
}

fx_status fx_poll_features (fx_engine* e, int track, float out12[FX_NUM_FEATURES], uint64_t* frame_index)
{
    if (! e || track < 0 || track >= e->cfg.n_tracks || ! out12) return FX_ERR_INVALID_ARG;
    return fx_poll_block (e, track, 1, out12, frame_index);
}

fx_status fx_flush (fx_engine* e)
{
    if (! e) return FX_ERR_INVALID_ARG;
    FX_CUDA (e, cudaSetDevice (e->cfg.device));
    for (auto& g : e->groups) if (g->stream) FX_CUDA (e, cudaStreamSynchronize (g->stream));
    for (int i = 0; i < 3; ++i) if (e->pipe_stream[i]) FX_CUDA (e, cudaStreamSynchronize (e->pipe_stream[i]));
    FX_CUDA (e, cudaStreamSynchronize (e->stream));
    FX_CUDA (e, cudaEventSynchronize (e->ev_last));
    return FX_OK;
}

// ---- OSC wire output ----------------------------------------------------------------------------------------------
namespace {
// OSCFeatureAnalysisOutput.h:107
const int kOscCode12[12]   = { FX_ONSET, FX_RMS, FX_F0, FX_CENTROID, FX_SLOPE, FX_SPREAD, FX_FLATNESS, FX_LER, FX_FLUX, FX_HER, FX_OER, FX_INHARM };
// README.md:55-57
const int kOscReadme10[10] = { FX_ONSET, FX_RMS, FX_F0, FX_CENTROID, FX_SLOPE, FX_SPREAD, FX_FLATNESS, FX_FLUX, FX_HER, FX_INHARM };
}

fx_status fx_osc_order (const float in12[FX_NUM_FEATURES], float* out, int n_out)
{
    if (! in12 || ! out) return FX_ERR_INVALID_ARG;
    if (n_out == 12) { for (int i = 0; i < 12; ++i) out[i] = in12[kOscCode12[i]]; return FX_OK; }
    if (n_out == 10) { for (int i = 0; i < 10; ++i) out[i] = in12[kOscReadme10[i]]; return FX_OK; }
    return FX_ERR_INVALID_ARG;
}

fx_status fx_osc_encode_tracks (fx_engine* e, const int* tracks, int n_tracks, const char* const* addresses, int n_floats,
                                unsigned char* out, int datagram_stride, int* sizes)
{
    if (! e || ! tracks || ! addresses || ! out || ! sizes || n_tracks < 0 || datagram_stride < 0) return FX_ERR_INVALID_ARG;
    if (n_floats != FX_OSC_FLOATS_CODE && n_floats != FX_OSC_FLOATS_README) return FX_ERR_INVALID_ARG;
    const int* order = n_floats == 12 ? kOscCode12 : kOscReadme10;
    const int tag_len = (1 + n_floats + 1 + 3) & ~3;                 // "," + n x "f" + NUL, padded to 4
    for (int i = 0; i < n_tracks; ++i)
    {
        sizes[i] = 0;
        if (tracks[i] < 0 || tracks[i] >= e->cfg.n_tracks || ! addresses[i]) return FX_ERR_INVALID_ARG;
        const int alen = (int) strlen (addresses[i]);
        const int apad = (alen + 1 + 3) & ~3;
        const int total = apad + tag_len + 4 * n_floats;
        if (total > datagram_stride) continue;
        float v[FX_NUM_FEATURES];
        fx_status st = fx_poll_block (e, tracks[i], 1, v, nullptr);
        if (st != FX_OK) return st;
        unsigned char* m = out + (size_t) i * (size_t) datagram_stride;
        memset (m, 0, (size_t) (apad + tag_len));
        memcpy (m, addresses[i], (size_t) alen);
        m[apad] = ',';
        memset (m + apad + 1, 'f', (size_t) n_floats);
        unsigned char* f = m + apad + tag_len;
        for (int k = 0; k < n_floats; ++k)
        {
            uint32_t bits;
            memcpy (&bits, &v[order[k]], 4);
            bits = htonl (bits);
            memcpy (f + 4 * k, &bits, 4);
        }
        sizes[i] = total;
    }
    return FX_OK;
}

// ---- measurement support ----------------------------------------------------------------------------------------------
fx_status fx_synth_device_at (fx_engine* e, float* d_audio, long track_stride, long n_samples,
                              long first_track, long first_sample, uint64_t seed, void* stream)
{
    if (! e || ! d_audio || first_sample < 0 || (first_sample & 3)) return FX_ERR_INVALID_ARG;
    FX_CUDA (e, cudaSetDevice (e->cfg.device));
    FX_CUDA (e, launch_synth (d_audio, track_stride, n_samples, e->cfg.n_tracks, first_track, first_sample, e->cfg.sample_rate, seed,
                              stream ? (cudaStream_t) stream : e->stream));
    e->launches += 1;
    return FX_OK;
}

fx_status fx_synth_device (fx_engine* e, float* d_audio, long track_stride, long n_samples,
                           long first_track, uint64_t seed, void* stream)
{
    return fx_synth_device_at (e, d_audio, track_stride, n_samples, first_track, 0, seed, stream);
}

uint64_t fx_kernel_launches (const fx_engine* e) { return e ? e->launches.load() : 0; }

fx_status fx_profile_enable (fx_engine* e, int on)
{
    if (! e) return FX_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> api (e->api_mutex);
    e->profiling = on != 0;
    return FX_OK;
}

fx_status fx_profile_read (fx_engine* e, double* ms_analyse, double* ms_post, long* n_calls)
{
    if (! e) return FX_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> api (e->api_mutex);
    FX_CUDA (e, cudaSetDevice (e->cfg.device));
    double ka = 0.0, kp = 0.0;
    long n = 0;
    for (auto& pr : e->prof_pending)
    {
        FX_CUDA (e, cudaEventSynchronize (pr.c));
        float m1 = 0.0f, m2 = 0.0f;
        FX_CUDA (e, cudaEventElapsedTime (&m1, pr.a, pr.b));
        FX_CUDA (e, cudaEventElapsedTime (&m2, pr.b, pr.c));
        ka += m1; kp += m2; ++n;
        e->prof_free.push_back (pr);
    }
    e->prof_pending.clear();
    if (ms_analyse) *ms_analyse = ka;
    if (ms_post) *ms_post = kp;
    if (n_calls) *n_calls = n;
    return FX_OK;
}

fx_status fx_measure_fp32_peak (int device, double* tflops)
{
    if (! tflops) return FX_ERR_INVALID_ARG;
    if (cudaSetDevice (device) != cudaSuccess) return FX_ERR_NO_DEVICE;
    return fx::measure_fp32_peak (tflops) == cudaSuccess ? FX_OK : FX_ERR_CUDA;
}

// Host -> device link probe: `reps` copies of `bytes` from a pinned buffer (write-combined if asked) to the device on one
// stream, timed with CUDA events.  bench.py runs it on all ranks at once to measure the box's concurrent upload ceiling next
// to the end-to-end figure.
fx_status fx_h2d_probe (int device, long bytes, int reps, int write_combined, double* gbs)
{
    if (! gbs || bytes <= 0 || reps <= 0) return FX_ERR_INVALID_ARG;
    if (cudaSetDevice (device) != cudaSuccess) return FX_ERR_NO_DEVICE;
    void *h = nullptr, *d = nullptr;
    cudaStream_t s = nullptr;
    cudaEvent_t a = nullptr, b = nullptr;
    fx_status st = FX_ERR_CUDA;
    float ms = 0.0f;
    if (cudaHostAlloc (&h, (size_t) bytes, write_combined ? cudaHostAllocWriteCombined : cudaHostAllocDefault) != cudaSuccess) goto done;
    memset (h, 1, (size_t) bytes);
    if (cudaMalloc (&d, (size_t) bytes) != cudaSuccess) goto done;
    if (cudaStreamCreateWithFlags (&s, cudaStreamNonBlocking) != cudaSuccess) goto done;
    if (cudaEventCreate (&a) != cudaSuccess || cudaEventCreate (&b) != cudaSuccess) goto done;
    if (cudaMemcpyAsync (d, h, (size_t) bytes, cudaMemcpyHostToDevice, s) != cudaSuccess) goto done;      // warm-up
    cudaEventRecord (a, s);
    for (int i = 0; i < reps; ++i) if (cudaMemcpyAsync (d, h, (size_t) bytes, cudaMemcpyHostToDevice, s) != cudaSuccess) goto done;
    cudaEventRecord (b, s);
    if (cudaEventSynchronize (b) != cudaSuccess) goto done;
    cudaEventElapsedTime (&ms, a, b);
    *gbs = (double) bytes * reps / (ms * 1e-3) / 1e9;
    st = FX_OK;
done:
    if (a) cudaEventDestroy (a);
    if (b) cudaEventDestroy (b);
    if (s) cudaStreamDestroy (s);
    if (d) cudaFree (d);
    if (h) cudaFreeHost (h);
    return st;
}

} // extern "C"
