// A client of include/habdec_b200/Decoder.hpp that hands channel 1 to a new payload: a batch file of N channels
// ([N][n] cf32) pushed in 65 536-sample calls, channel 1 reset before call K_RESET.
//   reset_channels FILE N n FS K_RESET   ->   "PRE <hex of channel 1's characters polled before the reset>", then
//                                              "CH<c> <hex of polled characters> <hex of getRTTY>" per channel
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <string>
#include <vector>

#include "habdec_b200/Decoder.hpp"

static std::string hex(const std::string& s)
{
    std::string out;
    char b[3];
    for (unsigned char c : s) { snprintf(b, sizeof(b), "%02x", c); out += b; }
    return out;
}

int main(int argc, char** argv)
{
    if (argc != 6) { fprintf(stderr, "usage: reset_channels FILE N n FS K_RESET\n"); return 2; }
    const int n_ch = atoi(argv[2]);
    const size_t n = size_t(atol(argv[3])), chunk = 65536;
    const double fs = atof(argv[4]);
    const size_t k_reset = size_t(atol(argv[5]));
    std::vector<std::complex<float>> iq(size_t(n_ch) * n);
    std::ifstream in(argv[1], std::ios::binary);
    in.read(reinterpret_cast<char*>(iq.data()), std::streamsize(iq.size() * sizeof(iq[0])));
    if (size_t(in.gcount()) != iq.size() * sizeof(iq[0])) { fprintf(stderr, "short file\n"); return 1; }

    habdec_b200::BatchDecoder dec(n_ch);
    // the Python BatchDecoder's defaults
    dec.baud(300.0); dec.rtty_bits(size_t(8)); dec.rtty_stops(2.0f); dec.dc_remove(false); dec.lowpass_bw(1500.0f); dec.lowpass_trans(0.025f);
    if (dec.setupDecimationStagesFactor(256) != 256) { fprintf(stderr, "factor\n"); return 1; }
    for (size_t k = 0; k * chunk < n; ++k) {
        if (k == k_reset) {
            printf("PRE %s\n", hex(dec.pollChars(1)).c_str());
            if (dec.resetChannel(1) != HBD_OK) { fprintf(stderr, "reset: %s\n", dec.lastError().c_str()); return 1; }
        }
        if (!dec.pushSamples(iq.data() + k * chunk, chunk, n, fs)) { fprintf(stderr, "push: %s\n", dec.lastError().c_str()); return 1; }
        if (dec.process() != HBD_OK) { fprintf(stderr, "process: %s\n", dec.lastError().c_str()); return 1; }
    }
    if (dec.resetChannels({}) != HBD_OK || dec.resetChannels({0, 0}) != HBD_ERR_ARG) { fprintf(stderr, "errors\n"); return 1; }
    for (int c = 0; c < n_ch; ++c) printf("CH%d %s %s\n", c, hex(dec.pollChars(c)).c_str(), hex(dec.getRTTY(c)).c_str());
    return 0;
}
