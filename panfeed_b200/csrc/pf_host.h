// Host-side helpers shared by the host-only translation units (pf_format.cu, pf_feeder.cu, pf_tsv.cu).
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <thread>

// Threads a host-side entry point uses when its caller passes n_threads = 0: every core, or
// PF_HOST_THREADS when that is set (several ranks of one box share the host's cores; the CLI
// under torchrun sets it to cores / ranks, as the staging-copy threads of pf_upload read it).
inline uint32_t pf_host_threads() {
  static const uint32_t n = []() {
    const char* e = getenv("PF_HOST_THREADS");
    const int v = e ? atoi(e) : 0;
    return v > 0 ? (uint32_t)v : std::max(1u, std::thread::hardware_concurrency());
  }();
  return n;
}
