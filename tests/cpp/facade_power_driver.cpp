// facade_power_driver.cpp -- test driver for the power-spectrum mode of the C++ host facade: AudioDeviceManager constructed with
// FX_SPECTRUM_POWER (its trailing constructor argument), one AnalyserTrackController per channel, audio in device blocks.
// Usage: facade_power_driver <audio.f32> <n_tracks> <n_samples> <block> <sample_rate> <out.f32>
// Reads [n_tracks][n_samples] fp32 and after every block that completed a hop appends the 12 smoothed features x n_tracks.
#include "../../feature-extractor_b200/host/FeatureExtractorB200.h"

#include <cstdio>
#include <cstdlib>
#include <memory>

using namespace fxb200;

int main (int argc, char** argv)
{
    if (argc < 7) { fprintf (stderr, "usage\n"); return 2; }
    const int T = atoi (argv[2]);
    const long S = atol (argv[3]);
    const int block = atoi (argv[4]);
    const double sr = atof (argv[5]);
    std::vector<float> audio ((size_t) T * (size_t) S);
    FILE* f = fopen (argv[1], "rb");
    if (! f || fread (audio.data(), sizeof (float), audio.size(), f) != audio.size()) { fprintf (stderr, "read failed\n"); return 2; }
    fclose (f);
    FILE* out = fopen (argv[6], "wb");

    OSCFeatureAnalysisOutput::timerAutoStart() = false;
    AudioDeviceManager deviceManager (T, sr, block, 2048, 0, 0, FX_SPECTRUM_POWER);
    std::vector<std::unique_ptr<AnalyserTrackController>> tracks;
    for (int ch = 0; ch < T; ++ch)
        tracks.emplace_back (new AnalyserTrackController (deviceManager, ch, "Input " + std::to_string (ch), "127.0.0.1:9000",
                                                          "127.0.0.1:9000", "/Audio/A" + std::to_string (ch)));
    AudioDeviceManager::AudioDeviceSetup setup;
    deviceManager.getAudioDeviceSetup (setup);
    for (auto& t : tracks) t->prepareToPlay (setup.bufferSize, setup.sampleRate);

    std::vector<const float*> chans ((size_t) T);
    uint64_t lastHop = 0;
    const long hopSize = deviceManager.getHopSize();
    for (long pos = 0; pos + block <= S; pos += block)
    {
        for (int ch = 0; ch < T; ++ch) chans[(size_t) ch] = audio.data() + (size_t) ch * (size_t) S + pos;
        deviceManager.processBlock (chans.data(), T, block);
        const uint64_t due = (uint64_t) ((pos + block) / hopSize);
        if (due == lastHop) continue;
        for (int ch = 0; ch < T; ++ch)
            if (! deviceManager.waitForHop (ch, due)) { fprintf (stderr, "hop %llu of track %d never arrived\n", (unsigned long long) due, ch); return 4; }
        lastHop = due;
        for (int ch = 0; ch < T; ++ch)
        {
            float v[FX_NUM_FEATURES];
            uint64_t hop = 0;
            tracks[(size_t) ch]->getFeatures().snapshot (v, &hop);
            fwrite (v, sizeof (float), FX_NUM_FEATURES, out);
        }
    }
    fclose (out);
    for (auto& t : tracks) t->stopAnalysis();
    printf ("hops %llu push_errors %ld\n", (unsigned long long) lastHop, deviceManager.getPushErrorCount());
    return 0;
}
