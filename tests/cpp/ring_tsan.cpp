// ring_tsan.cpp -- the host-side primitives of the real-time path (feature-extractor_b200/csrc/fx_rt_host.h) under
// ThreadSanitizer: the code that replaces AudioDataCollector's non-atomic writeIndex / readIndex / busy flag
// (AudioDataCollector.h:36-94) and the unsynchronised AudioFeatures reads (OSCFeatureAnalysisOutput.h:91-104).
// Built by tests/test_rt_host.py with -fsanitize=thread; exit code 0 and no "ThreadSanitizer" line = pass.
//
// Threads: one producer per half of the tracks (audio threads: push only), one consumer per track group (the engine's
// workers: verify every sample, release, publish under the seqlock), two pollers (OSC / GUI timers: the published block
// must never be torn), one control thread (clear requests, a track deactivated and re-activated while blocks flow).
#include "../../feature-extractor_b200/csrc/fx_rt_host.h"

#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <thread>
#include <vector>

using namespace fx;

static float sample_of (long track, long index) { return (float) ((track * 1000003L + index * 7L) % 65521L); }

int main (int argc, char** argv)
{
    const long T = 8, per = 4, H = 64, ring_hops = 8, L = ring_hops * H;
    const long total_hops = argc > 1 ? atol (argv[1]) : 4000;
    const long block = 24;
    std::vector<float> memory ((size_t) (T * L), 0.0f);
    TrackRings rings;
    rings.init (memory.data(), T, L, per);
    const long G = rings.G;
    std::vector<WakeWord> wake ((size_t) G);
    std::vector<SeqBlock> latest ((size_t) G);
    for (auto& s : latest) s.init ((size_t) per * 14);
    std::atomic<bool> stop { false };
    std::atomic<long> errors { 0 }, overruns { 0 }, cleared_seen { 0 };
    std::atomic<long> hops_done[2];
    hops_done[0].store (0); hops_done[1].store (0);
    // the controlled track carries a constant (its stream restarts at an arbitrary position after the re-activation)
    const long special = 6;
    const float special_value = 12345.0f;
    std::atomic<int>  special_phase { 0 };       // 0 active from the start, 1 inactive, 2 active again
    std::atomic<long> reactivated_at { 0 };      // hops_done[1] when the special track became active again
    std::mutex batch_mutex[2];                   // the engine's per-group batch mutex: consumer batches vs life-cycle calls

    auto producer = [&] (long first, long n)
    {
        std::vector<std::vector<float>> buf ((size_t) n, std::vector<float> ((size_t) block));
        std::vector<const float*> ch ((size_t) n);
        std::vector<long> pos ((size_t) n, 0);
        while (! stop.load (std::memory_order_acquire))
        {
            for (long i = 0; i < n; ++i)
            {
                const long t = first + i;
                // the producer of an inactive track keeps offering blocks (they are dropped); its stream position follows wpos
                pos[(size_t) i] = rings.wpos[(size_t) t].load (std::memory_order_relaxed);
                for (long k = 0; k < block; ++k) buf[(size_t) i][(size_t) k] = t == special ? special_value : sample_of (t, pos[(size_t) i] + k);
                ch[(size_t) i] = buf[(size_t) i].data();
            }
            unsigned char crossed[8] = { 0 };
            if (! rings.push (first, n, ch.data(), block, H, crossed)) { overruns.fetch_add (1); std::this_thread::yield(); continue; }
            for (long g = 0; g < G; ++g) if (crossed[g]) wake[(size_t) g].signal();
        }
    };

    auto consumer = [&] (long g)
    {
        const long t0 = g * per;
        while (! stop.load (std::memory_order_acquire))
        {
            const uint32_t ticket = wake[(size_t) g].observe();
            std::unique_lock<std::mutex> lk (batch_mutex[g]);
            long hops = rings.hops_available (g, t0, per, H);
            if (hops > ring_hops) hops = ring_hops;
            if (hops == 0) { lk.unlock(); wake[(size_t) g].wait (ticket, 5); continue; }
            const long r = rings.read_pos (g), n = hops * H;
            for (long t = t0; t < t0 + per; ++t)
            {
                rings.apply_clear (t, r, n);
                const bool act = rings.active[(size_t) t].load (std::memory_order_acquire) != 0u;
                const float* row = rings.row (t);
                for (long a = r; a < r + n; ++a)
                {
                    const float v = row[a % L];
                    if (v == 0.0f && (! act || t == 1)) { if (t == 1) cleared_seen.fetch_add (1); continue; }   // silence: inactive or cleared
                    if (act && v != (t == special ? special_value : sample_of (t, a))) errors.fetch_add (1);
                }
            }
            rings.consumed (g, n);
            const long done = hops_done[g].fetch_add (hops) + hops;
            latest[(size_t) g].write_begin();
            for (size_t i = 0; i < latest[(size_t) g].size(); ++i) latest[(size_t) g].put (i, (uint32_t) done);
            latest[(size_t) g].write_end();
        }
    };

    auto poller = [&] ()
    {
        std::vector<uint32_t> w ((size_t) per * 14);
        while (! stop.load (std::memory_order_acquire))
            for (long g = 0; g < G; ++g)
            {
                latest[(size_t) g].read (0, w.size(), w.data());
                for (uint32_t x : w) if (x != w[0]) { errors.fetch_add (1); break; }
            }
    };

    auto control = [&] ()
    {
        while (! stop.load (std::memory_order_acquire))
        {
            std::this_thread::sleep_for (std::chrono::milliseconds (2));
            rings.request_clear (1);                                   // track 1: transport events while audio flows
            const int ph = special_phase.load();
            if (ph == 0 && hops_done[1].load() > total_hops / 4)
            {
                std::lock_guard<std::mutex> lk (batch_mutex[rings.group_of (special)]);      // as fx_set_track_active does
                rings.deactivate (special);
                special_phase.store (1);
            }
            else if (ph == 1 && hops_done[1].load() > total_hops / 2)
            {
                std::lock_guard<std::mutex> lk (batch_mutex[rings.group_of (special)]);
                rings.activate (special);
                reactivated_at.store (hops_done[1].load());
                special_phase.store (2);
            }
        }
    };

    std::vector<std::thread> th;
    th.emplace_back (producer, 0L, 4L);
    th.emplace_back (producer, 4L, 4L);
    for (long g = 0; g < G; ++g) th.emplace_back (consumer, g);
    th.emplace_back (poller);
    th.emplace_back (poller);
    th.emplace_back (control);
    // the control thread advances one phase per tick: a fast box can reach total_hops before it has re-activated the special
    // track, so the run also lasts until the re-activated track has been checked for total_hops / 4 more hops
    while (hops_done[0].load() < total_hops || hops_done[1].load() < total_hops || special_phase.load() != 2 ||
           hops_done[1].load() < reactivated_at.load() + total_hops / 4)
        std::this_thread::sleep_for (std::chrono::milliseconds (1));
    stop.store (true, std::memory_order_release);
    for (long g = 0; g < G; ++g) wake[(size_t) g].signal();
    for (auto& t : th) t.join();
    printf ("hops %ld %ld overruns %ld cleared_samples %ld phase %d errors %ld\n", hops_done[0].load(), hops_done[1].load(), overruns.load(),
            cleared_seen.load(), special_phase.load(), errors.load());
    return errors.load() == 0 && special_phase.load() == 2 ? 0 : 1;
}
