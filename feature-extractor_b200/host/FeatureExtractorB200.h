// FeatureExtractorB200.h -- C++ host facade: the reference's per-track analyser surface, rebuilt over the C ABI
// of libfxb200.so (include/fx_engine.h).  Header-only; link with -lfxb200.
//
// Same class names, method names and argument meaning as the reference (all citations relative to
// /root/reference/Source/), so code written against
//     AudioDataCollector / RealTimeAnalyser / RealTimeSpectralAnalyser / RealTimeHarmonicAnalyser /
//     AudioFeatures / OSCFeatureAnalysisOutput / AnalyserTrackController
// keeps compiling when it switches `#include "include.h"` for this header and `juce::` device plumbing for
// fxb200::AudioDeviceManager.  What changed underneath:
//   * AudioDataCollector's 4096-float ring + spinning consumer (AudioDataCollector.h:24,72-94) is the engine's
//     pinned host ring (fx_push_block on the audio thread: copy + publish + wake, nothing else);
//   * the two analyser threads per track (AnalyserTrackController.h:184-185) are the engine's worker threads, one
//     per track group: startThread / stopThread start and stop the analysis of the track, the wake-up that
//     Thread::notify() gave is part of fx_push_block, and no CPU thread spins;
//   * AudioFeatures::getValue reads the engine's latest published smoothed vector (fx_poll_features, a seqlock);
//   * the 60 Hz timers of OSCFeatureAnalysisOutput (OSCFeatureAnalysisOutput.h:84-87,133) share one timer thread
//     (as juce::Timer objects do) that encodes every sender's datagram in one pass and ships them with sendmmsg.
// Everything lives in namespace fxb200 so that it can coexist with JUCE.
#pragma once

#include "../../include/fx_engine.h"

#include <arpa/inet.h>
#include <netdb.h>
#include <sys/socket.h>
#include <sys/uio.h>
#include <unistd.h>

#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <utility>
#include <vector>

namespace fxb200 {

using String = std::string;

// ------------------------------------------------------------------------------------------------------
// The slice of juce::AudioSampleBuffer the scope callback of AudioDataCollector hands out (one channel).
class AudioSampleBuffer
{
public:
    AudioSampleBuffer() = default;
    AudioSampleBuffer (int numChannels, int numSamples) : data ((size_t) (numChannels > 0 ? numSamples : 0), 0.0f) {}
    int getNumChannels() const noexcept { return 1; }
    int getNumSamples() const noexcept  { return (int) data.size(); }
    const float* getReadPointer (int) const noexcept { return data.data(); }
    float* getWritePointer (int) noexcept            { return data.data(); }
    float getSample (int, int i) const noexcept      { return data[(size_t) i]; }
    void setSample (int, int i, float v) noexcept    { data[(size_t) i] = v; }
private:
    std::vector<float> data;
};

// juce::AudioIODeviceCallback, as far as AudioDataCollector uses it (AudioDataCollector.h:18,28-38)
class AudioIODevice;
class AudioIODeviceCallback
{
public:
    virtual ~AudioIODeviceCallback() = default;
    virtual void audioDeviceIOCallback (const float** inputChannelData, int numInputChannels,
                                        float** outputChannelData, int numOutputChannels, int numSamples) = 0;
    virtual void audioDeviceAboutToStart (AudioIODevice*) {}
    virtual void audioDeviceStopped() {}
};

// ------------------------------------------------------------------------------------------------------
// AudioDeviceManager: stands where juce::AudioDeviceManager stood in AnalyserTrackController's constructor
// (AnalyserTrackController.h:17,35,41).  It owns the GPU engine for all its input channels.
//
// Threads, as in the reference (AudioDataCollector.h:36-70 copies and notifies; the analysis runs on its own threads,
// RealTimeAnalyser.h:97-127):
//   audio thread     processBlock(): every registered collector stages its channel pointer, then ONE fx_push_block per run
//                    of staged channels copies the block into the pinned ring and wakes the engine's group workers.
//                    No CUDA call, no lock, no allocation, no exception.
//   engine workers   analyse the complete hops (started by the first RealTimeAnalyser::startThread, stopped by the last
//                    stopThread) and then run the after-analysis hooks on the worker thread -- where
//                    RealTimeSpectralAnalyser::run fires its onset callback (RealTimeAnalyser.h:228-229).
//   message thread   everything else (construction, parameters, transport events).
class AudioDeviceManager
{
public:
    struct AudioDeviceSetup { int bufferSize = 512; double sampleRate = 48000.0; };

    AudioDeviceManager (int numInputChannels, double sampleRate = 48000.0, int bufferSize = 512,
                        int windowSize = 2048, int device = 0, int tracksPerGroup = 0,
                        int spectrum = FX_SPECTRUM_RE_SQUARED)       // FX_SPECTRUM_POWER: |X|^2 per bin (fx_engine.h)
    {
        fx_config cfg;
        fx_default_config (&cfg);
        cfg.spectrum = spectrum;
        cfg.n_tracks = numInputChannels;
        cfg.window = windowSize;                 // AnalyserTrackController.h:20-21
        cfg.hop = windowSize / 2;                // RealTimeAudioAnalysis.h:207
        cfg.sample_rate = sampleRate;
        cfg.device = device;
        cfg.tracks_per_group = tracksPerGroup > 0 ? tracksPerGroup : (numInputChannels > 128 ? 128 : numInputChannels);
        cfg.ring_hops = 16;
        setup.bufferSize = bufferSize;
        setup.sampleRate = sampleRate;
        numChannels = numInputChannels;
        hopSize = cfg.hop;
        if (fx_engine_create (&cfg, &engine) != FX_OK)
            throw std::runtime_error (String ("fx_engine_create: ") + fx_last_error (nullptr));   // no CPU fallback
        staged.assign ((size_t) numChannels, nullptr);
        owners.assign ((size_t) numChannels, nullptr);
        running.assign ((size_t) numChannels, 0);
        fresh.assign ((size_t) numChannels, 1);
        // a channel is analysed once an AnalyserTrackController has claimed it and started its analysers
        fx_set_track_active (engine, -1, 0, 0);
        fx_set_features_callback (engine, &AudioDeviceManager::featuresThunk, this);
    }

    ~AudioDeviceManager()
    {
        if (engine) { fx_rt_stop (engine); fx_engine_destroy (engine); }
    }
    AudioDeviceManager (const AudioDeviceManager&) = delete;
    AudioDeviceManager& operator= (const AudioDeviceManager&) = delete;

    void addAudioCallback (AudioIODeviceCallback* cb)    { callbacks.push_back (cb); }
    void removeAudioCallback (AudioIODeviceCallback* cb)
    {
        for (size_t i = 0; i < callbacks.size(); ++i)
            if (callbacks[i] == cb) { callbacks.erase (callbacks.begin() + (long) i); break; }
    }
    void getAudioDeviceSetup (AudioDeviceSetup& s) const { s = setup; }

    // The audio thread's entry point: one device block for every channel (what JUCE's device manager does when it calls each
    // AudioIODeviceCallback).  Only copies: the analysis happens on the engine's workers.
    void processBlock (const float** inputChannelData, int numInputChannels, int numSamples,
                       float** outputChannelData = nullptr, int numOutputChannels = 0) noexcept
    {
        inBlock = true;
        for (auto* cb : callbacks)
            cb->audioDeviceIOCallback (inputChannelData, numInputChannels, outputChannelData, numOutputChannels, numSamples);
        inBlock = false;
        for (int c = 0; c < numChannels;)
        {
            if (staged[(size_t) c] == nullptr) { ++c; continue; }
            int end = c;
            while (end < numChannels && staged[(size_t) end] != nullptr) ++end;
            const fx_status st = fx_push_block (engine, c, end - c, staged.data() + c, numSamples);
            if (st != FX_OK) { lastPushStatus = st; ++pushErrors; }
            for (int k = c; k < end; ++k) staged[(size_t) k] = nullptr;
            c = end;
        }
    }
    // collectors (audio thread): inside processBlock the pointer is staged for the block's one push
    void pushFromCollector (int track, const float* src, int numSamples) noexcept
    {
        if (track < 0 || track >= numChannels) return;
        if (inBlock) { staged[(size_t) track] = src; return; }
        const float* one[1] = { src };
        const fx_status st = fx_push_block (engine, track, 1, one, numSamples);
        if (st != FX_OK) { lastPushStatus = st; ++pushErrors; }
    }
    int  getLastPushStatus() const noexcept { return lastPushStatus; }     // FX_ERR_OVERRUN: the analysis fell a whole ring behind
    long getPushErrorCount() const noexcept { return pushErrors; }

    // hooks run on an engine worker thread after the hops of their track were analysed
    void addAfterAnalysisHook (const void* owner, int track, std::function<void()> f)
    {
        std::lock_guard<std::mutex> lk (hooksMutex);
        afterAnalysis.push_back (Hook { owner, track, std::move (f) });
    }
    void removeAfterAnalysisHooks (const void* owner)
    {
        std::lock_guard<std::mutex> lk (hooksMutex);
        for (size_t i = afterAnalysis.size(); i-- > 0;)
            if (afterAnalysis[i].owner == owner) afterAnalysis.erase (afterAnalysis.begin() + (long) i);
    }

    fx_engine* getEngine() const noexcept { return engine; }
    int getNumInputChannels() const noexcept { return numChannels; }
    long getHopSize() const noexcept { return hopSize; }

    // RealTimeAnalyser::startThread / stopThread (AnalyserTrackController.h:184-185,190-194)
    void analyserStarted (int track)
    {
        if (track < 0 || track >= numChannels) return;
        std::lock_guard<std::mutex> lk (stateMutex);
        if (running[(size_t) track]++ == 0)
        {
            fx_set_track_active (engine, track, 1, fresh[(size_t) track]);      // a new controller starts from empty histories
            fresh[(size_t) track] = 0;
        }
        if (totalRunning++ == 0) fx_rt_start (engine);
    }
    void analyserStopped (int track)
    {
        if (track < 0 || track >= numChannels) return;
        std::lock_guard<std::mutex> lk (stateMutex);
        if (running[(size_t) track] == 0) return;
        if (--running[(size_t) track] == 0) fx_set_track_active (engine, track, 0, 0);
        if (--totalRunning == 0) fx_rt_stop (engine);
    }

    // one collector per track feeds the ring; the reference's second collector per track carries the same samples
    bool claimTrack (int track, const void* owner)
    {
        if (track < 0 || track >= numChannels) return false;
        std::lock_guard<std::mutex> lk (stateMutex);
        if (owners[(size_t) track] == nullptr) { owners[(size_t) track] = owner; fresh[(size_t) track] = 1; }
        return owners[(size_t) track] == owner;
    }
    void releaseTrack (int track, const void* owner)
    {
        if (track < 0 || track >= numChannels) return;
        std::lock_guard<std::mutex> lk (stateMutex);
        if (owners[(size_t) track] == owner) owners[(size_t) track] = nullptr;
    }

    // blocks until `track` has analysed at least `hop` hops (tests and offline drivers; never the audio thread)
    bool waitForHop (int track, uint64_t hop, int timeoutMs = 5000) const
    {
        float v[FX_NUM_FEATURES];
        uint64_t idx = 0;
        for (int waited = 0; waited <= timeoutMs * 20; ++waited)
        {
            if (fx_poll_features (engine, track, v, &idx) == FX_OK && idx >= hop) return true;
            ::usleep (50);
        }
        return false;
    }

private:
    struct Hook { const void* owner; int track; std::function<void()> fn; };

    static void featuresThunk (void* user, int firstTrack, int nTracks, uint64_t /*frameIndex*/, int /*nNew*/)
    {
        auto* self = static_cast<AudioDeviceManager*> (user);
        std::lock_guard<std::mutex> lk (self->hooksMutex);
        for (auto& h : self->afterAnalysis)
            if (h.track >= firstTrack && h.track < firstTrack + nTracks) h.fn();
    }

    fx_engine* engine = nullptr;
    AudioDeviceSetup setup;
    int numChannels = 0;
    long hopSize = 0;
    bool inBlock = false;
    int lastPushStatus = FX_OK;
    long pushErrors = 0;
    int totalRunning = 0;
    std::mutex stateMutex, hooksMutex;
    std::vector<Hook> afterAnalysis;
    std::vector<AudioIODeviceCallback*> callbacks;
    std::vector<const float*> staged;
    std::vector<const void*> owners;
    std::vector<int> running;
    std::vector<int> fresh;
};

// ------------------------------------------------------------------------------------------------------
// AudioFeatures (RealTimeAnalyser.h:14-92): same enum, same accessors.  Bound to an engine track it reads the
// GPU's smoothed vector; unbound it is the reference's host-side store of ValueHistory moving averages.
struct AudioFeatures
{
    enum eAudioFeature
    {
        enOnset = 0, enRMS, enF0, enCentroid, enSpread, enFlatness, enLER, enFlux, enSlope,
        enHarmonicEnergyRatio, enOddEvenHarmonicRatio, enInharmonicity, numFeatures
    };

    static String getFeatureName (eAudioFeature f)
    {
        static const char* names[] = { "Onset", "Amp.", "Pitch", "Centroid", "Spread", "Flatness", "L.E.R", "Flux",
                                       "Slope", "H.E.R", "O.E.R", "Inharm." };
        return f >= 0 && f < numFeatures ? names[f] : "";
    }
    static float getMaxValueForFeature (eAudioFeature) { return 1.0f; }

    AudioFeatures()
    {
        for (int f = 0; f < numFeatures; ++f)
            local.emplace_back ((f == enOnset || f == enFlux) ? 1 : 10);      // RealTimeAnalyser.h:72-73
    }
    AudioFeatures (fx_engine* e, int trackIndex) : AudioFeatures() { engine = e; track = trackIndex; }

    void bind (fx_engine* e, int trackIndex) { engine = e; track = trackIndex; }
    fx_engine* getEngine() const noexcept { return engine; }
    int getTrack() const noexcept { return track; }

    void updateFeature (eAudioFeature f, float v)                              // RealTimeAnalyser.h:76-82
    {
        History& h = local[(size_t) f];
        for (size_t i = 0; i + 1 < h.v.size(); ++i) h.v[i] = h.v[i + 1];
        h.v.back() = v;
        if (h.recorded < (int) h.v.size()) h.recorded++;
    }

    float getValue (eAudioFeature f) const                                     // RealTimeAnalyser.h:84-88
    {
        if (engine != nullptr)
        {
            float v[FX_NUM_FEATURES];
            if (fx_poll_features (engine, track, v, nullptr) == FX_OK) return v[(int) f];
            return NAN;
        }
        const History& h = local[(size_t) f];
        float total = 0.0f;
        for (float x : h.v) total += x;
        return total / (float) h.recorded;
    }

    // all 12 at once + the index of the hop they belong to
    bool snapshot (float out12[FX_NUM_FEATURES], uint64_t* frameIndex = nullptr) const
    {
        return engine != nullptr && fx_poll_features (engine, track, out12, frameIndex) == FX_OK;
    }

private:
    struct History { explicit History (int n) : v ((size_t) n, 0.0f) {} std::vector<float> v; int recorded = 0; };
    std::vector<History> local;
    fx_engine* engine = nullptr;
    int track = -1;
};

// ------------------------------------------------------------------------------------------------------
// AudioDataCollector (AudioDataCollector.h:18-138)
class AudioDataCollector : public AudioIODeviceCallback
{
public:
    explicit AudioDataCollector (int audioChannelToCollect) : channelToCollect (audioChannelToCollect) {}
    ~AudioDataCollector() override { if (manager) manager->releaseTrack (channelToCollect, this); }
    AudioDataCollector (const AudioDataCollector&) = delete;
    AudioDataCollector& operator= (const AudioDataCollector&) = delete;

    void attach (AudioDeviceManager& m) { manager = &m; primary = m.claimTrack (channelToCollect, this); }

    // Audio thread.  Wait-free: the block is staged for the manager's one fx_push_block (memcpy into the pinned ring + publish).
    void audioDeviceIOCallback (const float** inputChannelData, int numInputChannels,
                                float** outputChannelData, int numOutputChannels, int numberOfSamples) override
    {
        const float* const* channelData = collectInput ? inputChannelData : (const float* const*) outputChannelData;   // :42
        const int available = collectInput ? numInputChannels : numOutputChannels;
        if (channelData == nullptr || channelToCollect < 0 || channelToCollect >= available || manager == nullptr) return;
        const float* src = channelData[channelToCollect];
        if (primary) manager->pushFromCollector (channelToCollect, src, numberOfSamples);
        if (bufferToDrawUpdated)                                                                       // :96-102
        {
            AudioSampleBuffer b (1, numberOfSamples);
            for (int i = 0; i < numberOfSamples; ++i) b.setSample (0, i, src[i] * gain);
            bufferToDrawUpdated (b);
        }
        if (notifyAnalysisThread) notifyAnalysisThread();                                              // :68-69
    }

    void setBufferToDrawUpdatedCallback  (std::function<void (AudioSampleBuffer&)> f) { bufferToDrawUpdated = std::move (f); }
    void setNotifyAnalysisThreadCallback (std::function<void()> f)                    { notifyAnalysisThread = std::move (f); }

    void toggleCollectInput (bool shouldCollectInput) { clearBuffer(); collectInput = shouldCollectInput; }         // :119
    void setExpectedSamplesPerBlock (int spb) noexcept         { expectedSamplesPerBlock = spb; }                    // :120
    // :122 circleBuffer.clear(): what was collected but not analysed yet becomes silence, positions stay
    void clearBuffer() { if (manager && primary) fx_clear_buffer (manager->getEngine(), channelToCollect); }
    void setChannelToCollect (int c)
    {
        if (manager) manager->releaseTrack (channelToCollect, this);
        channelToCollect = c;
        if (manager) primary = manager->claimTrack (c, this);
    }
    void setGain (float g)                                                                             // :124
    {
        gain = g;
        if (manager) fx_set_gain (manager->getEngine(), channelToCollect, g);
    }
    int  getChannel() const noexcept   { return channelToCollect; }
    int  getLastStatus() const noexcept { return manager ? manager->getLastPushStatus() : FX_OK; }   // FX_ERR_OVERRUN when the analysis fell behind the producer
    bool isPrimary() const noexcept { return primary; }
    AudioDeviceManager* getManager() const noexcept { return manager; }

private:
    AudioDeviceManager* manager = nullptr;
    std::function<void (AudioSampleBuffer&)> bufferToDrawUpdated;
    std::function<void()> notifyAnalysisThread;
    float gain = 1.0f;
    int expectedSamplesPerBlock = 512;
    int channelToCollect = 0;
    bool collectInput = true;
    bool primary = false;
};

// ------------------------------------------------------------------------------------------------------
struct OnsetDetector
{
    enum eOnsetDetectionType { enSpectral = 0, enAmplitude, enCombination, enNumTypes };     // SpectralCharacteristics.h:213-219
    static String getStringForDetectionType (eOnsetDetectionType t)
    {
        switch (t) { case enSpectral: return "Spectral"; case enAmplitude: return "Amplitude"; case enCombination: return "Combination"; default: return "UNKNOWN"; }
    }
};

// RealTimeAnalyser (RealTimeAnalyser.h:97-127): the juce::Thread surface is kept, the thread is the GPU.
class RealTimeAnalyser
{
public:
    RealTimeAnalyser (AudioDataCollector& adc, AudioFeatures& featuresRef, int windowSize, double sampleRate = 48000.0)
        : audioDataCollector (adc), features (featuresRef), window (windowSize), rate (sampleRate) {}
    virtual ~RealTimeAnalyser() { stopThread (0); }
    RealTimeAnalyser (const RealTimeAnalyser&) = delete;
    RealTimeAnalyser& operator= (const RealTimeAnalyser&) = delete;

    // :111-114 fft.setNyquistValue: every frequency-dependent quantity follows from the next analysed hop on (one rate per
    // device manager, as one audio device has)
    void sampleRateChanged (double newSampleRate)
    {
        rate = newSampleRate;
        if (fx_engine* e = engineOrNull()) fx_set_sample_rate (e, newSampleRate);
    }
    void startThread (int /*priority*/ = 5)
    {
        if (running) return;
        running = true;
        if (auto* m = audioDataCollector.getManager()) m->analyserStarted (audioDataCollector.getChannel());
    }
    bool stopThread (int /*timeoutMs*/)
    {
        if (! running) return true;
        running = false;
        if (auto* m = audioDataCollector.getManager()) m->analyserStopped (audioDataCollector.getChannel());
        return true;
    }
    bool isThreadRunning() const noexcept         { return running; }
    // Thread::notify(): the wake-up is part of fx_push_block (a futex wake of the group's worker when a hop completed)
    void notify() {}
    AudioFeatures& getFeatures() { return features; }
    int getWindowSize() const noexcept { return window; }
    double getSampleRate() const noexcept { return rate; }

protected:
    fx_engine* engineOrNull() const { return audioDataCollector.getManager() ? audioDataCollector.getManager()->getEngine() : nullptr; }
    AudioDataCollector& audioDataCollector;
    AudioFeatures& features;
    int window;
    double rate;
    bool running = false;
};

class RealTimeHarmonicAnalyser : public RealTimeAnalyser       // RealTimeAnalyser.h:133-188
{
public:
    using RealTimeAnalyser::RealTimeAnalyser;
};

class RealTimeSpectralAnalyser : public RealTimeAnalyser       // RealTimeAnalyser.h:193-269
{
public:
    using RealTimeAnalyser::RealTimeAnalyser;

    void setOnsetDetectionSensitivity (float s)                                  // :244-248
    {
        multiplier = 1.0f + s;
        apply();
    }
    void setOnsetWindowLength (int length)                                       // :250-254
    {
        histLen = length;
        apply();
    }
    void setOnsetDetectionType (OnsetDetector::eOnsetDetectionType t)            // :258
    {
        type = t;
        apply();
    }
    void setOnsetDetectedCallback (std::function<void()> f) { onsetDetectedCallback = std::move (f); }     // :256

    // runs on the engine's worker thread after this track's hops were analysed: fires the callback when the newest hop
    // carries an onset (:228-229)
    void dispatchOnsetCallback()
    {
        if (onsetDetectedCallback && features.getValue (AudioFeatures::enOnset) > 0.0f) onsetDetectedCallback();
    }

private:
    void apply()
    {
        if (fx_engine* e = engineOrNull())
            fx_set_onset (e, audioDataCollector.getChannel(), (int) type, histLen, multiplier);
    }
    OnsetDetector::eOnsetDetectionType type = OnsetDetector::enAmplitude;        // SpectralCharacteristics.h:240
    int histLen = 5;                                                             // :238-239
    float multiplier = 1.7f;                                                     // :311
    std::function<void()> onsetDetectedCallback;
};

// ------------------------------------------------------------------------------------------------------
// OSCFeatureAnalysisOutput (OSCFeatureAnalysisOutput.h:25-145): OSC 1.0 message over UDP,
// address pattern = bundleAddress, type tags ",ffffffffffff", twelve big-endian floats in the order of :107.
// connectToAddress starts the 60 Hz timer as the reference does (:133).  All timers share one thread (OSCTimerThread, as
// juce::Timer objects share JUCE's timer thread): per tick it encodes the datagrams of every running sender in one pass over
// the engine's published feature block (fx_osc_encode_tracks) and ships them with one sendmmsg per 1024 datagrams.
class OSCFeatureAnalysisOutput;

class OSCTimerThread
{
public:
    static OSCTimerThread& instance() { static OSCTimerThread t; return t; }

    void add (OSCFeatureAnalysisOutput* o, int hz)
    {
        std::lock_guard<std::mutex> lk (mutex);
        for (auto* x : outputs) if (x == o) return;
        outputs.push_back (o);
        rateHz = hz > 0 ? hz : 60;
        if (! thread.joinable()) { quit = false; thread = std::thread ([this] { run(); }); }
    }
    void remove (OSCFeatureAnalysisOutput* o)
    {
        std::unique_lock<std::mutex> lk (mutex);
        for (size_t i = 0; i < outputs.size(); ++i)
            if (outputs[i] == o) { outputs.erase (outputs.begin() + (long) i); break; }
        if (outputs.empty() && thread.joinable())
        {
            quit = true;
            lk.unlock();
            thread.join();
        }
    }
    // one timer tick for every registered sender, on the calling thread; returns the number of datagrams handed to the kernel
    long tick();
    unsigned long ticks() const noexcept { return tickCount; }
    unsigned long datagramsSent() const noexcept { return sentCount; }

    ~OSCTimerThread() { if (thread.joinable()) { quit = true; thread.join(); } }

private:
    OSCTimerThread() = default;
    void run()
    {
        auto next = std::chrono::steady_clock::now();
        while (! quit)
        {
            next += std::chrono::nanoseconds (1000000000L / rateHz);
            tick();
            std::this_thread::sleep_until (next);
        }
    }

    std::mutex mutex;
    std::vector<OSCFeatureAnalysisOutput*> outputs;
    std::thread thread;
    std::atomic<bool> quit { false };
    int rateHz = 60;
    int sock = -1;
    std::atomic<unsigned long> tickCount { 0 }, sentCount { 0 };
    // per-tick scratch (only the ticking thread touches it, under `mutex`)
    std::vector<int> tracks;
    std::vector<const char*> addrs;
    std::vector<unsigned char> wire;
    std::vector<int> sizes;
    std::vector<mmsghdr> msgs;
    std::vector<iovec> iov;
    std::vector<OSCFeatureAnalysisOutput*> batch;
};

class OSCFeatureAnalysisOutput
{
public:
    static constexpr int kDatagramStride = 256;

    OSCFeatureAnalysisOutput (AudioFeatures& rta, String ip, String bundle)
        : realTimeAudioFeatures (rta), address (std::move (ip)), bundleAddress (std::move (bundle))
    {
        if (! bundleAddress.empty()) connectToAddress (address);                  // :80-81
    }
    ~OSCFeatureAnalysisOutput() { stopTimer(); if (sock >= 0) ::close (sock); }
    OSCFeatureAnalysisOutput (const OSCFeatureAnalysisOutput&) = delete;
    OSCFeatureAnalysisOutput& operator= (const OSCFeatureAnalysisOutput&) = delete;

    // drivers that step the sender by hand switch the automatic 60 Hz timer off before constructing senders
    static bool& timerAutoStart() { static bool on = true; return on; }

    void startTimerHz (int hz) { timerRunning = true; OSCTimerThread::instance().add (this, hz); }          // juce::Timer
    void stopTimer()           { if (timerRunning) { timerRunning = false; OSCTimerThread::instance().remove (this); } }
    bool isTimerRunning() const noexcept { return timerRunning; }

    void timerCallback() { sendSpectralFeaturesViaOSC (true); }                   // :84-87

    // builds the message; returns the bytes that went (or would go) on the wire
    std::vector<uint8_t> encode() const
    {
        std::vector<uint8_t> m ((size_t) kDatagramStride);
        int size = 0;
        if (fx_engine* e = realTimeAudioFeatures.getEngine())
        {
            const int track = realTimeAudioFeatures.getTrack();
            const char* a = bundleAddress.c_str();
            fx_osc_encode_tracks (e, &track, 1, &a, FX_OSC_FLOATS_CODE, m.data(), kDatagramStride, &size);
            m.resize ((size_t) size);
            return m;
        }
        // unbound feature store: the same message from the host-side histories
        float v[FX_NUM_FEATURES], o[FX_OSC_FLOATS_CODE];
        for (int f = 0; f < FX_NUM_FEATURES; ++f) v[f] = realTimeAudioFeatures.getValue ((AudioFeatures::eAudioFeature) f);
        fx_osc_order (v, o, FX_OSC_FLOATS_CODE);
        m.clear();
        auto padded = [&m] (const String& s)
        {
            m.insert (m.end(), s.begin(), s.end());
            m.push_back (0);
            while (m.size() % 4) m.push_back (0);
        };
        padded (bundleAddress);
        padded (String (",") + String ((size_t) FX_OSC_FLOATS_CODE, 'f'));
        for (int i = 0; i < FX_OSC_FLOATS_CODE; ++i)
        {
            uint32_t bits;
            std::memcpy (&bits, &o[i], 4);
            bits = htonl (bits);
            const uint8_t* b = reinterpret_cast<const uint8_t*> (&bits);
            m.insert (m.end(), b, b + 4);
        }
        return m;
    }

    void sendSpectralFeaturesViaOSC (bool updateHarmonicFeatures)                 // :89-113
    {
        if (! updateHarmonicFeatures) return;                                     // the reference sends nothing in that branch (:109-112)
        const std::vector<uint8_t> m = encode();
        if (sock >= 0) ::send (sock, m.data(), m.size(), 0);
    }

    bool connectToAddress (String newAddress)                                     // :115-136
    {
        int port = 9000;
        const size_t sep = newAddress.find_last_of (':');
        if (sep != String::npos) port = std::atoi (newAddress.substr (sep + 1).c_str());
        address = newAddress.substr (0, newAddress.find (':'));
        stopTimer();
        if (sock >= 0) { ::close (sock); sock = -1; }
        connected = false;
        addrinfo hints{}; hints.ai_family = AF_INET; hints.ai_socktype = SOCK_DGRAM;
        addrinfo* res = nullptr;
        if (getaddrinfo (address.c_str(), std::to_string (port).c_str(), &hints, &res) != 0 || res == nullptr) return false;
        sock = ::socket (res->ai_family, res->ai_socktype, res->ai_protocol);
        const bool ok = sock >= 0 && ::connect (sock, res->ai_addr, res->ai_addrlen) == 0;
        if (ok && res->ai_addrlen <= sizeof (destination)) { std::memcpy (&destination, res->ai_addr, res->ai_addrlen); destinationLen = res->ai_addrlen; connected = true; }
        freeaddrinfo (res);
        if (! ok && sock >= 0) { ::close (sock); sock = -1; }
        if (ok && timerAutoStart()) startTimerHz (60);                            // :133
        return ok;
    }

    float getAudioFeature (AudioFeatures::eAudioFeature f) const { return realTimeAudioFeatures.getValue (f); }

    AudioFeatures& realTimeAudioFeatures;
    String address;
    String bundleAddress { "/Audio/Features" };

private:
    friend class OSCTimerThread;
    int sock = -1;
    bool connected = false, timerRunning = false;
    sockaddr_storage destination{};
    socklen_t destinationLen = 0;
};

inline long OSCTimerThread::tick()
{
    std::lock_guard<std::mutex> lk (mutex);
    ++tickCount;
    if (outputs.empty()) return 0;
    if (sock < 0) sock = ::socket (AF_INET, SOCK_DGRAM, 0);
    const size_t stride = (size_t) OSCFeatureAnalysisOutput::kDatagramStride;
    long sent = 0;
    // senders bound to an engine, engine by engine: one encode pass each
    std::vector<OSCFeatureAnalysisOutput*> pending (outputs);
    while (! pending.empty())
    {
        fx_engine* e = pending.front()->realTimeAudioFeatures.getEngine();
        batch.clear(); tracks.clear(); addrs.clear();
        for (size_t i = 0; i < pending.size();)
        {
            OSCFeatureAnalysisOutput* o = pending[i];
            if (o->realTimeAudioFeatures.getEngine() != e) { ++i; continue; }
            if (o->connected) { batch.push_back (o); tracks.push_back (o->realTimeAudioFeatures.getTrack()); addrs.push_back (o->bundleAddress.c_str()); }
            pending.erase (pending.begin() + (long) i);
        }
        if (batch.empty()) continue;
        const size_t n = batch.size();
        wire.resize (n * stride); sizes.assign (n, 0);
        if (e != nullptr)
        {
            if (fx_osc_encode_tracks (e, tracks.data(), (int) n, addrs.data(), FX_OSC_FLOATS_CODE, wire.data(), (int) stride, sizes.data()) != FX_OK) continue;
        }
        else
            for (size_t i = 0; i < n; ++i)
            {
                const std::vector<uint8_t> m = batch[i]->encode();
                sizes[i] = (int) (m.size() <= stride ? m.size() : 0);
                std::memcpy (wire.data() + i * stride, m.data(), (size_t) sizes[i]);
            }
        msgs.assign (n, mmsghdr{}); iov.resize (n);
        size_t count = 0;
        for (size_t i = 0; i < n; ++i)
        {
            if (sizes[i] <= 0) continue;
            iov[count].iov_base = wire.data() + i * stride;
            iov[count].iov_len = (size_t) sizes[i];
            msgs[count].msg_hdr.msg_name = &batch[i]->destination;
            msgs[count].msg_hdr.msg_namelen = batch[i]->destinationLen;
            msgs[count].msg_hdr.msg_iov = &iov[count];
            msgs[count].msg_hdr.msg_iovlen = 1;
            ++count;
        }
        for (size_t at = 0; at < count;)
        {
            const size_t chunk = count - at < 1024 ? count - at : 1024;         // UIO_MAXIOV
            const int r = ::sendmmsg (sock, msgs.data() + at, (unsigned) chunk, 0);
            if (r <= 0) break;
            sent += r;
            at += (size_t) r;
        }
    }
    sentCount += (unsigned long) sent;
    return sent;
}

// ------------------------------------------------------------------------------------------------------
// AudioFormatReader: what AudioFormatManager::createReaderFor (AudioFilePlayer.h:47, after registerBasicFormats :17) yields
// for the two basic formats the reference can open -- WAV (RIFF/WAVE: PCM, IEEE float, WAVE_FORMAT_EXTENSIBLE) and AIFF /
// AIFF-C ('NONE', 'sowt', 'fl32').  Only the container is parsed on the host; the sample data stays as it lies in the file
// and is converted on the GPU (kernel k_pcm_decode behind fx_analyse_host_pcm).
class AudioFormatReader
{
public:
    double  sampleRate = 0.0;
    int     numChannels = 0;
    int     bitsPerSample = 0;
    bool    usesFloatingPointData = false;
    long    lengthInSamples = 0;                  // sample frames
    int     pcmFormat = 0;                        // FX_PCM_*
    String  formatName;                           // "WAV file" / "AIFF file" as JUCE names them

    const uint8_t* data() const noexcept { return file.data() + dataOffset; }
    size_t dataBytes() const noexcept { return (size_t) lengthInSamples * (size_t) numChannels * (size_t) fx_pcm_bytes_per_sample (pcmFormat); }

    // nullptr when the file cannot be opened or is not a WAV / AIFF this reader understands (as createReaderFor does)
    static std::unique_ptr<AudioFormatReader> createReaderFor (const String& path)
    {
        FILE* f = fopen (path.c_str(), "rb");
        if (! f) return nullptr;
        std::unique_ptr<AudioFormatReader> r (new AudioFormatReader);
        fseek (f, 0, SEEK_END);
        const long size = ftell (f);
        fseek (f, 0, SEEK_SET);
        if (size < 12) { fclose (f); return nullptr; }
        r->file.resize ((size_t) size);
        const bool ok = fread (r->file.data(), 1, (size_t) size, f) == (size_t) size;
        fclose (f);
        if (! ok) return nullptr;
        return (r->parseWav() || r->parseAiff()) ? std::move (r) : nullptr;
    }
    static std::unique_ptr<AudioFormatReader> createReaderFor (std::vector<uint8_t> bytes)
    {
        std::unique_ptr<AudioFormatReader> r (new AudioFormatReader);
        r->file = std::move (bytes);
        return (r->file.size() >= 12 && (r->parseWav() || r->parseAiff())) ? std::move (r) : nullptr;
    }

private:
    std::vector<uint8_t> file;
    size_t dataOffset = 0;

    bool tag (size_t at, const char* four) const { return at + 4 <= file.size() && memcmp (file.data() + at, four, 4) == 0; }
    uint32_t le32 (size_t at) const { return (uint32_t) file[at] | ((uint32_t) file[at + 1] << 8) | ((uint32_t) file[at + 2] << 16) | ((uint32_t) file[at + 3] << 24); }
    uint16_t le16 (size_t at) const { return (uint16_t) (file[at] | (file[at + 1] << 8)); }
    uint32_t be32 (size_t at) const { return (uint32_t) file[at + 3] | ((uint32_t) file[at + 2] << 8) | ((uint32_t) file[at + 1] << 16) | ((uint32_t) file[at] << 24); }
    uint16_t be16 (size_t at) const { return (uint16_t) (file[at + 1] | (file[at] << 8)); }

    bool finish (size_t offset, size_t bytes, int bits, bool isFloat, bool bigEndian, bool eightBitSigned)
    {
        int fmt = 0;
        if (isFloat)        fmt = bits == 32 ? (bigEndian ? FX_PCM_F32BE : FX_PCM_F32LE) : 0;
        else if (bits == 8) fmt = eightBitSigned ? FX_PCM_S8 : FX_PCM_U8;
        else if (bits == 16) fmt = bigEndian ? FX_PCM_S16BE : FX_PCM_S16LE;
        else if (bits == 24) fmt = bigEndian ? FX_PCM_S24BE : FX_PCM_S24LE;
        else if (bits == 32) fmt = bigEndian ? FX_PCM_S32BE : FX_PCM_S32LE;
        if (fmt == 0 || numChannels < 1 || sampleRate <= 0.0 || offset > file.size()) return false;
        if (bytes > file.size() - offset) bytes = file.size() - offset;           // truncated file: read what is there
        pcmFormat = fmt; bitsPerSample = bits; usesFloatingPointData = isFloat; dataOffset = offset;
        lengthInSamples = (long) (bytes / ((size_t) numChannels * (size_t) fx_pcm_bytes_per_sample (fmt)));
        return true;
    }

    bool parseWav()
    {
        if (! (tag (0, "RIFF") && tag (8, "WAVE"))) return false;
        size_t at = 12;
        int formatTag = 0, bits = 0;
        bool haveFmt = false;
        while (at + 8 <= file.size())
        {
            const size_t len = le32 (at + 4), body = at + 8;
            if (tag (at, "fmt ") && body + 16 <= file.size())
            {
                formatTag = le16 (body); numChannels = le16 (body + 2); sampleRate = (double) le32 (body + 4); bits = le16 (body + 14);
                if (formatTag == 0xFFFE && len >= 40 && body + 26 <= file.size()) formatTag = le16 (body + 24);      // sub-format GUID, first two bytes
                haveFmt = true;
            }
            else if (tag (at, "data") && haveFmt)
            {
                formatName = "WAV file";
                return (formatTag == 1 || formatTag == 3) && finish (body, len, bits, formatTag == 3, false, false);
            }
            at = body + len + (len & 1u);                                         // chunks are word aligned
        }
        return false;
    }

    static double extended80 (const uint8_t* b)                                    // the AIFF sample rate
    {
        const int exponent = ((b[0] & 0x7f) << 8) | b[1];
        uint64_t mant = 0;
        for (int i = 0; i < 8; ++i) mant = (mant << 8) | b[2 + i];
        if (exponent == 0 && mant == 0) return 0.0;
        return std::ldexp ((double) mant, exponent - 16383 - 63) * ((b[0] & 0x80) ? -1.0 : 1.0);
    }

    bool parseAiff()
    {
        if (! (tag (0, "FORM") && (tag (8, "AIFF") || tag (8, "AIFC")))) return false;
        const bool aifc = tag (8, "AIFC");
        size_t at = 12;
        int bits = 0; uint32_t frames = 0; bool haveComm = false, littleEndian = false, isFloat = false;
        while (at + 8 <= file.size())
        {
            const size_t len = be32 (at + 4), body = at + 8;
            if (tag (at, "COMM") && body + 18 <= file.size())
            {
                numChannels = be16 (body); frames = be32 (body + 2); bits = be16 (body + 6); sampleRate = extended80 (file.data() + body + 8);
                if (aifc && len >= 22 && body + 22 <= file.size())
                {
                    if (tag (body + 18, "sowt")) littleEndian = true;
                    else if (tag (body + 18, "fl32") || tag (body + 18, "FL32")) isFloat = true;
                    else if (! tag (body + 18, "NONE")) return false;             // compressed AIFF-C
                }
                haveComm = true;
            }
            else if (tag (at, "SSND") && haveComm && body + 8 <= file.size())
            {
                const size_t offset = be32 (body);
                formatName = "AIFF file";
                const size_t bps = (size_t) ((bits + 7) / 8);
                return finish (body + 8 + offset, (size_t) frames * (size_t) numChannels * bps, (int) bps * 8, isFloat, ! littleEndian, true);
            }
            at = body + len + (len & 1u);
        }
        return false;
    }
};

// ------------------------------------------------------------------------------------------------------
// AudioFilePlayer (AudioFilePlayer.h:14-78).  The reference plays the file through the device output and the collectors
// re-capture one output channel per track (AudioDataCollector.h:42-43); here the loaded file is analysed in one call:
// track t of the engine takes channel t % numChannels of the file, the PCM goes to the GPU at its file width.
// The transport surface (play / pause / stop / restart / hasFile) is kept; it selects what analyseLoadedFile() covers.
class AudioFilePlayer
{
public:
    AudioFilePlayer() = default;
    AudioFilePlayer (const AudioFilePlayer&) = delete;
    AudioFilePlayer& operator= (const AudioFilePlayer&) = delete;

    void setupAudioCallback (AudioDeviceManager& deviceManager) { manager = &deviceManager; }           // :29-33

    void loadFileIntoTransport (const String& audioFile)                                              // :41-60
    {
        playing = false; position = 0;
        currentAudioFileSource = AudioFormatReader::createReaderFor (audioFile);
    }
    void play()    { playing = true; }                                                                  // :62
    void pause()   { playing = false; }                                                                 // :63
    void stop()    { pause(); position = 0; }                                                           // :64
    void restart() { position = 0; }                                                                    // :65
    bool hasFile() const { return currentAudioFileSource != nullptr; }                                  // :67
    bool isPlaying() const noexcept { return playing; }
    const AudioFormatReader* getReader() const noexcept { return currentAudioFileSource.get(); }
    void setPosition (long sampleFrame) { position = sampleFrame < 0 ? 0 : sampleFrame; }

    // Analyse the loaded file from the transport position to its end (complete hops only) on the manager's engine.
    // smoothed receives [tracks][frames][12] in AudioFeatures order; returns the number of frames per track, -1 on error.
    long analyseLoadedFile (std::vector<float>& smoothed, std::vector<float>* raw = nullptr)
    {
        if (! manager || ! currentAudioFileSource) return -1;
        const AudioFormatReader& r = *currentAudioFileSource;
        fx_engine* e = manager->getEngine();
        const long remaining = r.lengthInSamples - position;
        if (remaining <= 0) return 0;
        const size_t frameBytes = (size_t) r.numChannels * (size_t) fx_pcm_bytes_per_sample (r.pcmFormat);
        const int T = manager->getNumInputChannels();
        const long hop = manager->getHopSize();
        const long frames = remaining / hop;
        smoothed.assign ((size_t) T * (size_t) frames * FX_NUM_FEATURES, 0.0f);
        if (raw) raw->assign (smoothed.size(), 0.0f);
        if (frames == 0) return 0;
        long got = 0;
        const fx_status st = fx_analyse_host_pcm (e, r.data() + (size_t) position * frameBytes, r.pcmFormat, r.numChannels, -1, 0, remaining,
                                                  raw ? raw->data() : nullptr, smoothed.data(), nullptr, &got);
        if (st != FX_OK || got != frames) return -1;
        position += frames * hop;
        return frames;
    }

private:
    AudioDeviceManager* manager = nullptr;
    std::unique_ptr<AudioFormatReader> currentAudioFileSource;
    bool playing = false;
    long position = 0;
};

// ------------------------------------------------------------------------------------------------------
// AnalyserTrackController (AnalyserTrackController.h:14-212) without the GUI link and the file player.
class AnalyserTrackController
{
public:
    AnalyserTrackController (AudioDeviceManager& deviceManagerRef, int channelToAnalyse, String nameOfInputChannel,
                             String ip, String secondaryIP, String bundle)
        : features (channelToAnalyse >= 0 ? deviceManagerRef.getEngine() : nullptr, channelToAnalyse),
          audioDataCollectorHarm (channelToAnalyse), audioDataCollectorSpec (channelToAnalyse),
          audioAnalyserHarm (audioDataCollectorHarm, features, 2048), audioAnalyserSpec (audioDataCollectorSpec, features, 2048),
          oscFeatureSender (features, std::move (ip), bundle), secondaryOSCFeatureSender (features, std::move (secondaryIP), bundle),
          deviceManager (deviceManagerRef), channelName (std::move (nameOfInputChannel))
    {
        enabled = channelToAnalyse >= 0;                                          // :27
        if (enabled)
        {
            audioDataCollectorSpec.attach (deviceManager);                        // feeds the ring
            audioDataCollectorHarm.attach (deviceManager);                        // same samples: second collector of the reference (:35)
            audioDataCollectorHarm.setNotifyAnalysisThreadCallback ([this]() { audioAnalyserHarm.notify(); });
            deviceManager.addAudioCallback (&audioDataCollectorHarm);
            audioDataCollectorSpec.setNotifyAnalysisThreadCallback ([this]() { audioAnalyserSpec.notify(); });
            deviceManager.addAudioCallback (&audioDataCollectorSpec);
            deviceManager.addAfterAnalysisHook (this, channelToAnalyse, [this]() { audioAnalyserSpec.dispatchOnsetCallback(); });      // RealTimeAnalyser.h:228-229
        }
    }

    ~AnalyserTrackController()
    {
        if (enabled)
        {
            deviceManager.removeAudioCallback (&audioDataCollectorHarm);
            deviceManager.removeAudioCallback (&audioDataCollectorSpec);
            deviceManager.removeAfterAnalysisHooks (this);
        }
        stopAnalysis();
        audioDataCollectorHarm.setNotifyAnalysisThreadCallback (nullptr);
        audioDataCollectorSpec.setNotifyAnalysisThreadCallback (nullptr);
    }
    AnalyserTrackController (const AnalyserTrackController&) = delete;
    AnalyserTrackController& operator= (const AnalyserTrackController&) = delete;

    void clearAnalysisBuffers() { audioDataCollectorHarm.clearBuffer(); audioDataCollectorSpec.clearBuffer(); }    // :167-171
    float getAudioFeature (AudioFeatures::eAudioFeature f) const { return features.getValue (f); }                 // :173

    void prepareToPlay (int samplesPerBlockExpected, double sampleRate)           // :175-188
    {
        stopAnalysis();
        audioAnalyserHarm.sampleRateChanged (sampleRate);
        audioAnalyserSpec.sampleRateChanged (sampleRate);
        audioAnalyserHarm.startThread (4);
        audioAnalyserSpec.startThread (4);
        audioDataCollectorHarm.setExpectedSamplesPerBlock (samplesPerBlockExpected);
        audioDataCollectorSpec.setExpectedSamplesPerBlock (samplesPerBlockExpected);
    }
    void stopAnalysis() { audioAnalyserHarm.stopThread (100); audioAnalyserSpec.stopThread (100); }                // :190-194

    // the setters AnalyserTrack's GUI callbacks reach (:126-134)
    void setGain (float g)                       { audioDataCollectorHarm.setGain (g); audioDataCollectorSpec.setGain (g); }
    void setOnsetDetectionSensitivity (float s)  { audioAnalyserSpec.setOnsetDetectionSensitivity (s); }
    void setOnsetWindowLength (int n)            { audioAnalyserSpec.setOnsetWindowLength (n); }
    void setOnsetDetectionType (OnsetDetector::eOnsetDetectionType t) { audioAnalyserSpec.setOnsetDetectionType (t); }
    void setOnsetDetectedCallback (std::function<void()> f) { audioAnalyserSpec.setOnsetDetectedCallback (std::move (f)); }

    String getChannelName() const noexcept { return channelName; }
    bool isEnabled() const noexcept { return enabled; }
    AudioFeatures& getFeatures() { return features; }
    OSCFeatureAnalysisOutput& getOSCSender() { return oscFeatureSender; }
    OSCFeatureAnalysisOutput& getSecondaryOSCSender() { return secondaryOSCFeatureSender; }

private:
    AudioFeatures            features;
    AudioDataCollector       audioDataCollectorHarm;
    AudioDataCollector       audioDataCollectorSpec;
    RealTimeHarmonicAnalyser audioAnalyserHarm;
    RealTimeSpectralAnalyser audioAnalyserSpec;
    OSCFeatureAnalysisOutput oscFeatureSender;
    OSCFeatureAnalysisOutput secondaryOSCFeatureSender;
    AudioDeviceManager&      deviceManager;
    String                   channelName;
    bool                     enabled { true };
};

} // namespace fxb200
