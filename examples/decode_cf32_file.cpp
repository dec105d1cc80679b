// Minimal drop-in check of the C++ facade: decode a raw interleaved IQ file the way the reference's
// DECODER_THREAD does (code/websocketServer/main.cpp:235-245: 65536-sample pushes, process after each).
//   g++ -std=c++17 -I include examples/decode_cf32_file.cpp -L habdec_b200 -lhabdec_b200 -Wl,-rpath,$PWD/habdec_b200 -o decode_cf32
//   ./decode_cf32 capture.cf32 2048000 300 8 2 256
//   ./decode_cf32 capture.cu8 2048000 300 8 2 256 cu8      (an rtl_sdr capture; cs16 / cs8 likewise)
// Integer files are pushed as integers: the library dequantises them on the GPU (include/habdec_b200.h, hbd_push_iq).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <vector>
#include "habdec_b200/Decoder.hpp"

int main(int argc, char** argv)
{
    if (argc < 3) { std::cerr << "usage: " << argv[0] << " file sampling_rate [baud bits stops dec_factor [cf32|cs16|cs8|cu8]]\n"; return 2; }
    const double fs = atof(argv[2]);
    const char* fmt_name = argc > 7 ? argv[7] : "cf32";
    hbd_iq_format fmt;
    size_t bytes;
    if (!strcmp(fmt_name, "cf32")) { fmt = HBD_IQ_CF32; bytes = 8; }
    else if (!strcmp(fmt_name, "cs16")) { fmt = HBD_IQ_CS16; bytes = 4; }
    else if (!strcmp(fmt_name, "cs8")) { fmt = HBD_IQ_CS8; bytes = 2; }
    else if (!strcmp(fmt_name, "cu8")) { fmt = HBD_IQ_CU8; bytes = 2; }
    else { std::cerr << "unknown sample format " << fmt_name << "\n"; return 2; }
    habdec_b200::Decoder D;
    D.baud(argc > 3 ? atof(argv[3]) : 300);
    D.rtty_bits(argc > 4 ? atoi(argv[4]) : 8);
    D.rtty_stops(argc > 5 ? atof(argv[5]) : 2);
    D.lowpass_bw(1500); D.lowpass_trans(0.025f);
    D.setupDecimationStagesFactor(argc > 6 ? atoi(argv[6]) : 256);
    D.sentence_callback_ = [](std::string cs, std::string data, std::string crc) { std::cout << "\nSENTENCE " << cs << "," << data << "*" << crc << std::endl; };
    D.character_callback_ = [](std::string s) { std::cout << s << std::flush; };
    FILE* f = fopen(argv[1], "rb");
    if (!f) { perror("open"); return 1; }
    habdec_b200::IQVector v; v.samplingRate(fs);
    std::vector<unsigned char> raw(256 * 256 * bytes);
    for (;;) {
        const size_t n = fread(raw.data(), bytes, 256 * 256, f);
        if (!n) break;
        if (fmt == HBD_IQ_CF32) {
            v.assign(reinterpret_cast<const std::complex<float>*>(raw.data()), reinterpret_cast<const std::complex<float>*>(raw.data()) + n);
            D.pushSamples(v);
        } else {
            D.pushSamples(raw.data(), fmt, n, fs);
        }
        D();
    }
    fclose(f);
    std::cout << "\nlast sentence: " << D.getLastSentence() << std::endl;
    return 0;
}
