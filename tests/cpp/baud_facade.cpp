// A client of the baud-rate estimation members of include/habdec_b200/Decoder.hpp: N channels of a batch file ([N][n] cf32)
// pushed in 65 536-sample calls with estimation on, then the estimates and one apply.
//   baud_facade FILE N n FS   ->   "EST<c> <baud> <nominal> <confidence> <runs> <long_runs>" per channel,
//                                  "APPLIED <count>" and "BAUD<c> <rate>" per channel
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <stdexcept>
#include <vector>

#include "habdec_b200/Decoder.hpp"

int main(int argc, char** argv)
{
    if (argc != 5) { fprintf(stderr, "usage: baud_facade FILE N n FS\n"); return 2; }
    const int n_ch = atoi(argv[2]);
    const size_t n = size_t(atol(argv[3])), chunk = 65536;
    const double fs = atof(argv[4]);
    std::vector<std::complex<float>> iq(size_t(n_ch) * n);
    std::ifstream in(argv[1], std::ios::binary);
    in.read(reinterpret_cast<char*>(iq.data()), std::streamsize(iq.size() * sizeof(iq[0])));
    if (size_t(in.gcount()) != iq.size() * sizeof(iq[0])) { fprintf(stderr, "short file\n"); return 1; }
    try {
        habdec_b200::BatchDecoder dec(n_ch);
        dec.baud(45.45); dec.rtty_bits(size_t(8)); dec.rtty_stops(2.0f);
        if (dec.setupDecimationStagesFactor(256) != 256) { fprintf(stderr, "factor\n"); return 1; }
        if (dec.applyBaudEstimates() != HBD_ERR_STATE || !dec.getBaudEstimates().empty()) { fprintf(stderr, "off: no error\n"); return 1; }
        if (dec.setBaudEstimation(true) != HBD_OK) { fprintf(stderr, "on: %s\n", dec.lastError().c_str()); return 1; }
        for (size_t k = 0; (k + 1) * chunk <= n; ++k) {
            if (!dec.pushSamples(iq.data() + k * chunk, chunk, n, fs) || dec.process() != HBD_OK) { fprintf(stderr, "call: %s\n", dec.lastError().c_str()); return 1; }
        }
        const std::vector<hbd_baud_estimate> est = dec.getBaudEstimates();
        if (int(est.size()) != n_ch) { fprintf(stderr, "estimates: %s\n", dec.lastError().c_str()); return 1; }
        for (int c = 0; c < n_ch; ++c)
            printf("EST%d %.17g %.17g %.17g %u %u\n", c, est[c].baud, est[c].nominal, est[c].confidence, est[c].runs, est[c].long_runs);
        std::vector<double> applied(static_cast<size_t>(n_ch));
        const int count = dec.applyBaudEstimates(0.8, 50, applied.data());
        printf("APPLIED %d\n", count);
        for (int c = 0; c < n_ch; ++c) printf("BAUD%d %.17g\n", c, hbd_get_baud(dec.handle(), c));
    } catch (const std::runtime_error& e) {
        fprintf(stderr, "%s\n", e.what());
        return 1;
    }
    return 0;
}
