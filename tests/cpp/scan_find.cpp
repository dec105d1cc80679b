// A client of include/habdec_b200/Scanner.hpp: scan a cf32 file in pushes of `chunk` samples and print the signals found.
//   scan_find FILE FS N_FFT CHUNK   ->   "NSEG s" then one "SIG center shift snr bin_lo bin_hi" line per signal
#include <cstdio>
#include <cstdlib>
#include <fstream>

#include "habdec_b200/Scanner.hpp"

int main(int argc, char** argv)
{
    if (argc != 5) { fprintf(stderr, "usage: scan_find FILE FS N_FFT CHUNK\n"); return 2; }
    const double fs = atof(argv[2]);
    const size_t chunk = size_t(atol(argv[4]));
    habdec_b200::Scanner scan(size_t(atol(argv[3])));
    std::ifstream in(argv[1], std::ios::binary);
    habdec_b200::IQVector v;
    v.samplingRate(fs);
    for (;;) {
        v.resize(chunk);
        in.read(reinterpret_cast<char*>(v.data()), std::streamsize(chunk * sizeof(v[0])));
        v.resize(size_t(in.gcount()) / sizeof(v[0]));
        if (v.empty()) break;
        if (!scan.push(v)) { fprintf(stderr, "push: %s\n", scan.lastError()); return 1; }
    }
    unsigned long long n_seg = 0;
    if (scan.psd(&n_seg).size() != scan.size()) { fprintf(stderr, "psd: %s\n", scan.lastError()); return 1; }
    printf("NSEG %llu\n", n_seg);
    for (const hbd_scan_signal& s : scan.find()) printf("SIG %.17g %.17g %.17g %d %d\n", s.center_hz, s.shift_hz, s.snr_db, s.bin_lo, s.bin_hi);
    return 0;
}
