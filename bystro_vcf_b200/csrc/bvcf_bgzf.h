// bvcf_bgzf.h -- inside libbvcf: the bgzf header rule of bvcf_bgzf.cpp, shared with bgzf_walk (bvcf_api.cu).
#ifndef BVCF_BGZF_H
#define BVCF_BGZF_H

#include <cstddef>
#include <cstdint>

// The size BSIZE of the bgzf block whose header starts at p: 0 when the header is not complete in p[0, n), -1 with a
// static reason in *why (when why is not null) when it is not a bgzf header.
__attribute__((visibility("hidden"))) long long bgzf_header(const uint8_t *p, size_t n, const char **why);

#endif
