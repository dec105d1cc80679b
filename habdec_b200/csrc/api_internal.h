// internal hooks between the translation units of libhabdec_b200.so (not part of the ABI)
#pragma once
#include <memory>
#include <string>
struct hbd_decoder;
struct hbd_result_sink;
struct hbd_result_record;
namespace hbd {
int internal_device(hbd_decoder* h);
void internal_set_error(hbd_decoder* h, const std::string& what);
void internal_free_dist(void* ctx);            // implemented in dist.cu
struct DistFree { void operator()(void* ctx) const { internal_free_dist(ctx); } };
using DistSlot = std::unique_ptr<void, DistFree>;
DistSlot& internal_dist_slot(hbd_decoder* h);  // opaque per-handle context of dist.cu
// gather.cpp: feed a sink without copying; `recs` must stay valid and unchanged until sink_flush(s) has returned
int sink_feed_borrowed(hbd_result_sink* s, const hbd_result_record* recs, size_t n);
void sink_flush(hbd_result_sink* s);
}
