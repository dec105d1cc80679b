// Host-side, non data-parallel pieces of the path (see host_tail.cpp)
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <algorithm>
#include <deque>
#include <functional>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "../../include/habdec_b200.h"

namespace hbd {

// FirFilter::LP_BlackmanHarris; returns the (possibly unchanged) tap count, fills `taps` only on a redesign
size_t design_lowpass(float rel_width, float trans, size_t input_size, size_t current_taps, std::vector<float>& taps);

std::string crc16_hex(const std::string& s);

struct SentenceMatch {
    bool ok = false;
    std::string callsign, data, crc;
    size_t rest_offset = 0;
};
bool extract_sentence(const std::string& stream, SentenceMatch& m);

using SentenceSink = std::function<void(int ch, const std::string& callsign, const std::string& data, const std::string& crc)>;

// text side of one channel (Decoder.h:188-200: rtty_char_stream_, last_sentence_, chr_callback_stream_).
// What waits to be polled / gathered -- printable characters and CRC-valid sentences since the last poll -- lives in the
// channel's slot of ONE array of hbd_result_record (hbd_decoder::pend): hbd_pack_results is then a sequential copy of that
// array, and the drain loop touches one cache line of it per channel instead of two scattered heap strings.  What does
// not fit a slot (88 characters / 128 sentence bytes) spills into the strings below and moves up when the slot is emptied.
struct TextChannel {
    std::string text_stream;        // getRTTY()
    std::string last_sentence;      // getLastSentence()
    std::string chars_spill, sent_spill;
    std::vector<unsigned char> raw_pending; // raw chars since the last poll (SSDV consumers)
    bool scan_clean = true;         // text_stream is known to hold no extractable sentence (see feed)
    bool latent = false;            // ... except one that only waits for a '*' to appear in the stream (see feed)
    void feed(const unsigned char* raw, size_t n, int ch, const SentenceSink& sink, bool keep_raw, hbd_result_record& pend);
    // the text state of a new Decoder (hbd_reset_channels); what waits to be polled (the pending record, the spills,
    // raw_pending) is output, not state, and stays
    void restart() { text_stream.clear(); last_sentence.clear(); scan_clean = true; latent = false; }
    // pull the end of the string feed() appends to into the cache (the drain loop knows its next channels)
    void prefetch_tails() const { __builtin_prefetch(text_stream.data() + text_stream.size()); }

    static void append(char* slot, uint16_t& used, size_t cap, std::string& spill, const char* p, size_t n)
    {
        if (spill.empty()) {
            const size_t k = std::min(n, cap - used);
            memcpy(slot + used, p, k);
            used = uint16_t(used + k); p += k; n -= k;
        }
        if (n) spill.append(p, n);
    }
    static void refill(char* slot, uint16_t& used, size_t cap, std::string& spill)   // the slot has just been emptied
    {
        const size_t k = std::min(cap, spill.size());
        if (k) { memcpy(slot, spill.data(), k); spill.erase(0, k); }
        used = uint16_t(k);
    }
    size_t chars_size(const hbd_result_record& r) const { return r.n_chars + chars_spill.size(); }
    size_t sent_size(const hbd_result_record& r) const { return r.sentence_bytes + sent_spill.size(); }
    std::string chars_from(const hbd_result_record& r, size_t from) const   // pending characters [from, end)
    {
        std::string out;
        if (from < r.n_chars) out.assign(r.chars + from, r.n_chars - from);
        const size_t sf = from > r.n_chars ? from - r.n_chars : 0;
        if (sf < chars_spill.size()) out.append(chars_spill, sf, std::string::npos);
        return out;
    }
    std::string sentences_all(const hbd_result_record& r) const { return std::string(r.sentences, r.sentence_bytes) + sent_spill; }
    void clear_chars(hbd_result_record& r) { r.n_chars = 0; chars_spill.clear(); }
    void clear_sentences(hbd_result_record& r) { r.sentence_bytes = 0; sent_spill.clear(); }
};

// ---- SSDV packet sync: the buffer automaton and image bookkeeping of SSDV_wraper_t (ssdv_wrapper.cpp:37-148) -------
// The packet test (ssdv_dec_is_packet, :66) is not evaluated here: the GPU tests every window of 256 consecutive
// characters that starts at a 0x55 and reports the accepted ones by stream position (ssdv.cu).  That is enough because
// every window the automaton can ask about is such a window:
//   * `buff` is always [junk | contiguous stream bytes]: junk (bytes left in front of an extracted packet, :91) holds
//     no 0x55, since the packet started at the FIRST 0x55 of the buffer (:54) or at offset 0 (:82-83);
//   * packet_begin always points into the contiguous part, and the 256 bytes from it are contiguous too.
// The automaton itself -- one packet test per push, the `size < 256` early outs that depend on the junk length, the
// buffer clears -- is replayed byte for byte, so accepted packets surface on the same call as in the reference.
struct SsdvHeader {                  // what ssdv_dec_header (fsphil/ssdv, published layout) extracts, :92
    char callsign[8] = {0};
    uint16_t image_id = 0, packet_id = 0, width = 0, height = 0;
};
SsdvHeader ssdv_decode_header(const unsigned char* pkt);

struct SsdvVerdict { uint32_t pos; int errors; std::array<unsigned char, 256> data; };
struct SsdvEvent { SsdvHeader header; int errors = 0; int set_size = 0; std::array<unsigned char, 256> data; };

struct SsdvChannel {
    std::vector<unsigned char> buff;                 // ssdv_wrapper.h:38
    long packet_begin = -1;                          // :39
    uint32_t stream_end = 0;                         // stream index one past the last byte of buff (mod 2^32)
    std::deque<SsdvVerdict> verdicts;                // accepted windows reported by the GPU, ascending position
    using ImageKey = std::pair<std::string, uint16_t>;
    struct Filed { SsdvHeader header; std::array<unsigned char, 256> data; };
    std::map<ImageKey, std::map<uint16_t, Filed>> packets;   // :62; the inner map is the set ordered by packet id (:53-57)
    ImageKey last_key{"", 0};                        // last_img_k_, :82
    std::vector<SsdvEvent> events_pending;           // accepted packets since the last poll

    // one SSDV_wraper_t::push(); true (and `ev` filled) when a packet was filed
    bool push(const unsigned char* chars, size_t n, SsdvEvent& ev);
    // a new SSDV_wraper_t (hbd_reset_channels); packets not polled yet (events_pending) stay
    void restart() { buff.clear(); packet_begin = -1; stream_end = 0; verdicts.clear(); packets.clear(); last_key = ImageKey("", 0); }
    size_t image(const std::string& callsign, int image_id, unsigned char* out, size_t cap) const;
};

} // namespace hbd
