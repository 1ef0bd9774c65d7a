// libsrcnn.cpp -- ProcessSRCNN (include/libsrcnn.h): the reference's implied library API
// (src/test.cpp:347-361) on top of the C ABI.  Host-side glue only; all arithmetic runs in the CUDA
// kernels behind srcnn_process_host().  No CPU fallback.
#include "../../include/libsrcnn.h"

#include <cstring>
#include <mutex>
#include <new>
#include <vector>

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
    const size_t npx = (size_t)w * h, onpx = (size_t)ow * oh;
    const bool has_alpha = d == 2, gray = d <= 2;
    unsigned char* out = new (std::nothrow) unsigned char[onpx * d];
    if (!out) return SRCNN_E_NOMEM;
    // grey (d = 1) and RGBA (d = 4): one call straight into `out` (RGBA: the colour path plus alpha through the plain bicubic
    // resize, on the device); grey + alpha (d = 2): the one-plane path and the alpha plane apart, interleaved here
    std::vector<unsigned char> pix, pix_out, alpha, alpha_out;
    const size_t ch = gray ? 1 : 3;
    if (d == 1) {
        rc = srcnn_process_host(g_ctx, refbuff, (int)w, (int)h, (size_t)w, SRCNN_ORDER_GRAY, muliply, out, (size_t)ow);
    } else if (d == 4) {
        rc = srcnn_process_host(g_ctx, refbuff, (int)w, (int)h, (size_t)w * 4, SRCNN_ORDER_RGBA, muliply, out, (size_t)ow * 4);
    } else {
        pix.resize(npx * ch); pix_out.resize(onpx * ch);
        if (has_alpha) { alpha.resize(npx); alpha_out.resize(onpx); }
        for (size_t i = 0; i < npx; i++) {
            const unsigned char* p = refbuff + i * d;
            for (size_t k = 0; k < ch; k++) pix[ch * i + k] = p[k];
            if (has_alpha) alpha[i] = p[d - 1];
        }
        rc = srcnn_process_host(g_ctx, pix.data(), (int)w, (int)h, (size_t)w * ch, gray ? SRCNN_ORDER_GRAY : SRCNN_ORDER_RGB, muliply,
                                pix_out.data(), (size_t)ow * ch);
    }
    if (rc) { delete[] out; return rc; }
    if (has_alpha) {
        // alpha: the plain bicubic resize of the path (resize(..., CV_INTER_CUBIC), src/srcnn.cpp:577-582), no CNN
        rc = srcnn_resize_plane_host(g_ctx, alpha.data(), (int)w, (int)h, (size_t)w, muliply, alpha_out.data(), (size_t)ow);
        if (rc) { delete[] out; return rc; }
    }
    if (d == 2 || d == 3)
        for (size_t i = 0; i < onpx; i++) {
            unsigned char* q = out + i * d;
            for (size_t k = 0; k < ch; k++) q[k] = pix_out[ch * i + k];
            if (has_alpha) q[d - 1] = alpha_out[i];
        }
    outbuff = out;
    outbuffsz = (unsigned)(onpx * d);
    return 0;
}
