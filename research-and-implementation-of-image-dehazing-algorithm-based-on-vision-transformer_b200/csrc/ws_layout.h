// Bump layout of one call's workspace: regions of 256-byte-rounded sizes, in the order the call asks for them.  Without a
// base it only counts (the *_workspace_bytes query); with the caller's workspace it hands out the same offsets (the launch),
// so the query and the launch run one layout function and cannot disagree.
#pragma once
#include <stddef.h>

namespace lewin {

struct WsLayout {
    unsigned char* base = nullptr;
    size_t bytes = 0;
    template <typename P>
    P* take(size_t n) {
        P* p = base ? reinterpret_cast<P*>(base + bytes) : nullptr;
        bytes += (n + 255) / 256 * 256;
        return p;
    }
};

}  // namespace lewin
