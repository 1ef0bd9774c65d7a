// libsrcnn.cpp -- ProcessSRCNN (include/libsrcnn.h): the reference's implied library API
// (src/test.cpp:347-361) on top of the C ABI.  Host-side glue only; all arithmetic runs in the CUDA
// kernels behind srcnn_process_host().  No CPU fallback.
#include "../../include/libsrcnn.h"

#include <cstring>
#include <mutex>
#include <new>

#include "../../include/srcnn_b200.h"

namespace {
std::mutex g_mu;
srcnn_ctx* g_ctx = nullptr;  // one lazily created context on device 0, like the reference's process-wide state
}  // namespace

int ProcessSRCNN(const unsigned char* refbuff, unsigned w, unsigned h, unsigned d, float muliply,
                 unsigned char*& outbuff, unsigned& outbuffsz) {
    outbuff = nullptr;
    outbuffsz = 0;
    if (!refbuff || w == 0 || h == 0 || d < 1 || d > 4) return SRCNN_E_ARG;
    int ow = 0, oh = 0;
    int rc = srcnn_out_dims((int)w, (int)h, muliply, &ow, &oh);
    if (rc) return rc;
    std::lock_guard<std::mutex> lock(g_mu);
    if (!g_ctx) {
        rc = srcnn_create(&g_ctx, 0, SRCNN_VARIANT_TC);
        if (rc) return rc;
    }
    const size_t onpx = (size_t)ow * oh;
    unsigned char* out = new (std::nothrow) unsigned char[onpx * d];
    if (!out) return SRCNN_E_NOMEM;
    // every d is one call straight into `out`: grey, grey + alpha, RGB, RGBA (alpha through the plain bicubic resize of the path,
    // resize(..., CV_INTER_CUBIC) src/srcnn.cpp:577-582, no CNN)
    static const int kOrder[5] = {-1, SRCNN_ORDER_GRAY, SRCNN_ORDER_GRAYA, SRCNN_ORDER_RGB, SRCNN_ORDER_RGBA};
    rc = srcnn_process_host(g_ctx, refbuff, (int)w, (int)h, (size_t)w * d, kOrder[d], muliply, out, (size_t)ow * d);
    if (rc) { delete[] out; return rc; }
    outbuff = out;
    outbuffsz = (unsigned)(onpx * d);
    return 0;
}
