// C ABI of the telemetry layer (include/habdec_b200.h, "telemetry" section): stateless parse / distance functions and
// hbd_tracker, the host object that plays the role of SentenceCallback + GLOBALS::STATS for many channels at once.
// Host-only: usable on rank 0 over sentences gathered from every rank, or attached to a decoder handle.
#include <algorithm>
#include <chrono>
#include <cstring>
#include <mutex>
#include <unordered_map>

#include "../../include/habdec_b200.h"
#include "telemetry.h"
#include "telemetry_abi.h"

using namespace hbd;

struct hbd_tracker {
    std::mutex mtx;
    std::unordered_map<int, TelemetryChannel> chans;
    float st_lat = 0, st_lon = 0, st_alt = 0;       // GLOBALS::PARAMS station_lat_/lon_/alt_ (floats, GLOBALS.h:83-85)
    long long frozen_now = -1;
    double t_create = 0;
    hbd_telemetry_cb cb = nullptr; void* cb_user = nullptr;
};

namespace {
double mono_now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

size_t copy_str(const std::string& s, char* out, size_t cap)
{
    if (out && cap) { const size_t k = std::min(s.size(), cap - 1); memcpy(out, s.data(), k); out[k] = 0; }
    return s.size();
}

void fill(hbd_telemetry& o, const Telemetry& t)
{
    memset(&o, 0, sizeof o);
    strncpy(o.payload_callsign, t.payload_callsign.c_str(), sizeof o.payload_callsign - 1);
    strncpy(o.datetime, t.datetime.c_str(), sizeof o.datetime - 1);
    o.frame = t.frame; o.lat = t.lat; o.lon = t.lon; o.alt = t.alt;
}

void fill(hbd_gps_distance& o, const GpsDistance& g)
{
    o.dist_line_ = g.dist_line_; o.dist_circle_ = g.dist_circle_; o.dist_radians_ = g.dist_radians_;
    o.elevation_ = g.elevation_; o.bearing_ = g.bearing_;
}
} // namespace

int hbd::tracker_feed(hbd_tracker* t, int ch, const std::string& callsign, const std::string& data, const std::string& crc)
{
    hbd_telemetry rec; hbd_telemetry_cb cb = nullptr; void* user = nullptr; std::string sentence;
    {
        std::lock_guard<std::mutex> l(t->mtx);
        TelemetryChannel& tc = t->chans[ch];
        const ParseStatus r = tc.on_sentence(callsign, data, crc, t->st_lat, t->st_lon, t->st_alt, t->frozen_now, mono_now());
        if (r != PARSE_OK) return int(r);
        if (!t->cb) return 1;
        fill(rec, tc.pending.back()); cb = t->cb; user = t->cb_user;
        sentence = callsign + "," + data + "*" + crc;
    }
    cb(user, ch, &rec, sentence.c_str());
    return 1;
}

extern "C" {

int hbd_parse_sentence(const char* s, long long now_unix, hbd_telemetry* out)
{
    if (!s || !out) return HBD_PARSE_BADARG;
    Telemetry t;
    const ParseStatus r = parse_sentence(s, now_unix, t);
    if (r == PARSE_OK) fill(*out, t);
    return int(r);
}

int hbd_parse_sentence_time(const char* s, int* hour, int* minute, float* second)
{
    if (!s || !hour || !minute || !second) return HBD_PARSE_BADARG;
    return int(parse_sentence_time(s, *hour, *minute, *second));
}

int hbd_parse_gps_pos(const char* s, float* out)
{
    if (!s || !out) return HBD_PARSE_BADARG;
    return int(parse_gps_pos(s, *out));
}

size_t hbd_timestamp_from_hms(int hour, int minute, float second, long long now_unix, char* out, size_t cap)
{
    return copy_str(timestamp_from_hms(hour, minute, second, now_unix), out, cap);
}

void hbd_calc_gps_distance(double lat1, double lon1, double alt1, double lat2, double lon2, double alt2, hbd_gps_distance* out)
{
    if (out) fill(*out, calc_gps_distance(lat1, lon1, alt1, lat2, lon2, alt2));
}

size_t hbd_tracking_telemetry_payload(const hbd_telemetry* t, char* out, size_t cap)
{
    if (!t) return 0;
    Telemetry x; x.payload_callsign = t->payload_callsign; x.datetime = t->datetime; x.frame = t->frame; x.lat = t->lat; x.lon = t->lon; x.alt = t->alt;
    return copy_str(tracking_payload(x), out, cap);
}

hbd_tracker* hbd_tracker_create(void) { hbd_tracker* t = new hbd_tracker; t->t_create = mono_now(); return t; }
void hbd_tracker_destroy(hbd_tracker* t) { delete t; }

int hbd_tracker_set_station(hbd_tracker* t, float lat, float lon, float alt)
{
    if (!t) return HBD_ERR_ARG;
    std::lock_guard<std::mutex> l(t->mtx); t->st_lat = lat; t->st_lon = lon; t->st_alt = alt; return HBD_OK;
}

int hbd_tracker_set_clock(hbd_tracker* t, long long now_unix)
{
    if (!t) return HBD_ERR_ARG;
    std::lock_guard<std::mutex> l(t->mtx); t->frozen_now = now_unix; return HBD_OK;
}

int hbd_tracker_set_callback(hbd_tracker* t, hbd_telemetry_cb cb, void* user)
{
    if (!t) return HBD_ERR_ARG;
    std::lock_guard<std::mutex> l(t->mtx); t->cb = cb; t->cb_user = user; return HBD_OK;
}

int hbd_tracker_push(hbd_tracker* t, int ch, const char* callsign, const char* data, const char* crc)
{
    if (!t || !callsign || !data || !crc) return HBD_PARSE_BADARG;
    return tracker_feed(t, ch, callsign, data, crc);
}

int hbd_tracker_push_sentence(hbd_tracker* t, int ch, const char* sentence)
{
    if (!t || !sentence) return HBD_PARSE_BADARG;
    std::string s(sentence);
    while (!s.empty() && (s.back() == '\n' || s.back() == '\r')) s.pop_back();
    const size_t comma = s.find(','), star = s.rfind('*');
    if (comma == std::string::npos || star == std::string::npos || star < comma) return HBD_PARSE_BADARG;
    return tracker_feed(t, ch, s.substr(0, comma), s.substr(comma + 1, star - comma - 1), s.substr(star + 1));
}

int hbd_tracker_reset(hbd_tracker* t, int ch)
{
    if (!t) return HBD_ERR_ARG;
    std::lock_guard<std::mutex> l(t->mtx); t->chans.erase(ch); return HBD_OK;
}

size_t hbd_tracker_poll(hbd_tracker* t, int ch, hbd_telemetry* out, size_t cap)
{
    if (!t) return 0;
    std::lock_guard<std::mutex> l(t->mtx);
    auto it = t->chans.find(ch);
    if (it == t->chans.end()) return 0;
    std::vector<Telemetry>& p = it->second.pending;
    const size_t n = p.size();
    if (!out) return n;
    const size_t k = std::min(n, cap);
    for (size_t i = 0; i < k; ++i) fill(out[i], p[i]);
    p.erase(p.begin(), p.begin() + long(k));
    return n;
}

int hbd_tracker_stats(hbd_tracker* t, int ch, hbd_channel_stats* out)
{
    if (!t || !out) return HBD_ERR_ARG;
    std::lock_guard<std::mutex> l(t->mtx);
    auto it = t->chans.find(ch);
    TelemetryChannel none;
    const TelemetryChannel& tc = it == t->chans.end() ? none : it->second;
    out->num_ok_ = tc.num_ok_; fill(out->D_, tc.D_); out->dist_max_ = tc.dist_max_; out->elev_min_ = tc.elev_min_;
    out->age_s = mono_now() - (tc.last_sentence_mono >= 0 ? tc.last_sentence_mono : t->t_create);
    return HBD_OK;
}

size_t hbd_tracker_stats_payload(hbd_tracker* t, int ch, int with_age, char* out, size_t cap)
{
    if (!t) return 0;
    std::lock_guard<std::mutex> l(t->mtx);
    auto it = t->chans.find(ch);
    TelemetryChannel none;
    const TelemetryChannel& tc = it == t->chans.end() ? none : it->second;
    // age: whole seconds since the last sentence (duration_cast<seconds> truncates; the int(round()) after it is a no-op)
    const long long age = with_age ? (long long)(mono_now() - (tc.last_sentence_mono >= 0 ? tc.last_sentence_mono : t->t_create)) : -1;
    return copy_str(tc.stats_payload(t->st_lat, t->st_lon, t->st_alt, age), out, cap);
}

size_t hbd_tracker_get_sentence(hbd_tracker* t, int ch, int frame, char* out, size_t cap)
{
    if (!t) return 0;
    std::lock_guard<std::mutex> l(t->mtx);
    auto it = t->chans.find(ch);
    if (it == t->chans.end()) return 0;
    auto s = it->second.sentences_map.find(frame);
    return s == it->second.sentences_map.end() ? 0 : copy_str(s->second, out, cap);
}

} // extern "C"
