// libsrcnn.h -- the library entry point the reference's own smoke test binds (src/test.cpp:347-353;
// the header `libsrcnn.h` it includes is absent from the reference repo, so the signature is taken
// from that call site).  C++ (reference-compatible references); a thin wrapper over the C ABI in
// srcnn_b200.h, implemented in srcnn_cpp_b200/cli/libsrcnn.cpp and exported by libsrcnn_b200.so.
//
//   refbuff   packed 8-bit pixels, `d` bytes per pixel: 3 = RGB, 4 = RGBA (one SRCNN_ORDER_RGBA call: colour goes through the
//             SRCNN path, straight alpha takes the path's plain bicubic resize, no CNN), 1 = grey (SRCNN_ORDER_GRAY), 2 =
//             grey+alpha (one SRCNN_ORDER_GRAYA call: grey through the one-plane path, alpha as for d = 4) -- the inputs
//             src/test.cpp:34-134 (convImage) can produce
//   w, h, d   geometry
//   muliply   scale ratio (sic, the reference's spelling)
//   outbuff   callee-allocated with new[] (caller delete[]s it, src/test.cpp:365-369)
//   outbuffsz (unsigned)((float)w*muliply) * (unsigned)((float)h*muliply) * d   (src/test.cpp:357-361)
// returns 0 on success, a negative srcnn status otherwise.
#ifndef LIBSRCNN_H
#define LIBSRCNN_H

#if defined(__GNUC__)
#define LIBSRCNN_API __attribute__((visibility("default")))
#else
#define LIBSRCNN_API
#endif

LIBSRCNN_API int ProcessSRCNN(const unsigned char* refbuff, unsigned w, unsigned h, unsigned d, float muliply,
                              unsigned char*& outbuff, unsigned& outbuffsz);

#endif
