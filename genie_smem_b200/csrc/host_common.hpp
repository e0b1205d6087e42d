// Shared host-side helpers of libgenie_smem (error text, status codes).
#pragma once
#include <stdint.h>

#include <string>

namespace gsm {
extern thread_local std::string g_last_error;
int fail(int code, const std::string& msg);

// kernels.cu: device counts (n uint32) -> exclusive offsets (n + 1 uint64, off[n] = total) on `stream`, through the
// record scan of gsm_smem_select; tmp holds scan_tmp_bytes(n) bytes of device scratch.
uint64_t scan_tmp_bytes(uint64_t n);
int scan_counts(const uint32_t* cnt, uint64_t n, uint64_t* off, void* tmp, uint64_t tmp_bytes, void* stream);
}  // namespace gsm
