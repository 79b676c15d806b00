// libpanfeed_b200.so — C-ABI entry points (include/panfeed_b200.h) and the host
// side of the pipeline: batch validation and planning, buffer management,
// kernel sequencing, result staging.  One translation unit; the parts, in order:
//   kernels      k1_*.cuh k2_*.cuh k3_*.cuh k4_dedup.cuh k5_md5.cuh k6_assoc.cuh synth.cuh
//   host side    pf_ctx.cuh pf_lifetime.cuh pf_upload.cuh pf_execute.cuh pf_pipeline.cuh
//                pf_synth_api.cuh pf_exchange.cuh pf_exchange_run.cuh pf_assoc.cuh
// (pf_format.cu, the native text formatter, is a second, host-only translation unit.)
#include <cuda.h>            // driver types for the virtual-memory pool (entry points are fetched at run time)
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <unistd.h>
#include <unordered_map>
#include <vector>

#include "../../include/panfeed_b200.h"
#include "k1_extract.cuh"
#include "k1_fused.cuh"
#include "k2_onesweep.cuh"
#include "k3_reduce.cuh"
#include "k3_local.cuh"
#include "k3_block.cuh"
#include "k4_dedup.cuh"
#include "k5_md5.cuh"
#include "k6_assoc.cuh"
#include "synth.cuh"

using namespace pf;

#include "pf_ctx.cuh"
#include "pf_lifetime.cuh"
#include "pf_upload.cuh"
#include "pf_execute.cuh"
#include "pf_pipeline.cuh"
#include "pf_synth_api.cuh"
#include "pf_exchange.cuh"
#include "pf_exchange_run.cuh"
#include "pf_assoc.cuh"
