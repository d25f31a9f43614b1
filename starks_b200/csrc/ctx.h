// ctx.h -- library context shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <string>
#include <vector>
#include "../../include/starks_b200.h"
#include "field.cuh"
#include "hostmath.h"

struct stk_table {
  stk::fe root;     // canonical root the table was built for
  uint64_t n;       // number of entries (w^0 .. w^(n-1)), twiddle form
  int mont;         // built for the Montgomery field currently set?
  stk::fe* d;
};

// validated (root, n, direction) -> derived constants; repeated transforms skip the host
// exponentiations (an inverse costs two 256-bit modular inversions otherwise)
struct stk_ntt_consts {
  stk::fe root;
  uint64_t n;
  int inverse;
  stk::fe w;          // root or root^-1
  stk::fe scale_tw;   // n^-1 in twiddle form (inverse only)
  const stk::fe* W = nullptr;  // resolved table (valid while table_gen is unchanged)
  uint64_t wstride = 1;
  uint64_t table_gen = ~0ull;
};

// (G2^i - 1)^-1 table of the pointwise boundary quotient (stark.cu); per context like `tables`
struct stk_invtable {
  stk::fe root;
  uint64_t n;
  stk::fe* d;
};

// Byte budgets of the two table caches (a 2^26 twiddle table is 2 GiB, a 2^23 inverse table
// 256 MiB): least recently used entries are dropped once a cache would exceed its budget.
static const uint64_t kTableCacheBytes = 6ull << 30;
static const uint64_t kInvTableCacheBytes = 2ull << 30;

struct stk_ctx {
  int device = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_streams[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev[8] = {};
  int sm_count = 148;
  bool is_stark = true;
  stk::fe p;
  stk::MontField mont;
  std::vector<stk_table> tables;       // least recently used first
  std::vector<stk_invtable> invtables; // least recently used first
  std::vector<stk_ntt_consts> ntt_consts;
  uint64_t table_gen = 0;  // bumped whenever a table is freed
  static const int kScratchSlots = 14;
  void* scratch[kScratchSlots] = {};   // 0-1 transforms, 2-3 small staging, 4-7 host pipeline, 8-9 FRI,
  uint64_t scratch_bytes[kScratchSlots] = {};  // 10 device-side counters, 11 host-trace staging,
                                               // 12-13 polynomial product / division (poly.cu)
  std::string err;
};

static inline int stk_fail(stk_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  return code;
}

#define STK_CUDA(c, call)                                                                     \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return stk_fail((c), STK_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                      __FILE__, __LINE__);                                                    \
  } while (0)

#define STK_TRY(expr)            \
  do {                           \
    int rc_ = (expr);            \
    if (rc_ != STK_OK) return rc_; \
  } while (0)

// internal helpers (ntt_api.cu)
int stk_scratch(stk_ctx* c, int slot, uint64_t bytes, void** out);
int stk_get_table(stk_ctx* c, const stk::fe& root, uint64_t n, const stk::fe** d_table);
// Same, but may return a longer cached table T (order n*stride, T.root^stride == root) to be
// indexed as T[e*stride]: sub-transforms (G1 = G2^ext, FRI layers' roots w^4, w^16, ...)
// reuse the big table instead of building and caching their own.
int stk_get_table_strided(stk_ctx* c, const stk::fe& root, uint64_t n, const stk::fe** d_table, uint64_t* stride);
stk::fe stk_load_fe(const uint32_t* w);
// optional peer scatter of a transform's final pass (sharded commit, see ntt.cuh peer_on = 2)
struct stk_peer_leaf {
  int g;                      // log2 of the rank count
  uint32_t col0;              // global index of this rank's first column
  const uint64_t* ptrs;       // nranks exchange buffers (columns_total x N/G elements each)
};
int stk_ntt_dev_peer(stk_ctx* c, const stk::fe* d_in, uint64_t n_in, uint64_t in_stride, uint64_t n, uint64_t batch,
                     const stk::fe& root, const stk_peer_leaf& peer);
// branch gather with the query indices already on the device; asynchronous (merkle.cu)
int stk_merkle_paths_dev(stk_ctx* c, const stk::fe* d_cols, uint64_t n, uint64_t ncols, uint64_t col_stride,
                         const uint8_t* d_nodes, const uint64_t* d_idx, uint64_t k, uint32_t* d_out, uint64_t rec_bytes);
int stk_ntt_dev(stk_ctx* c, const stk::fe* d_in, uint64_t n_in, uint64_t in_stride, stk::fe* d_out,
                uint64_t out_stride, uint64_t n, uint64_t batch, const stk::fe& root, int inverse, int scale);
int stk_ntt_dev_r0(stk_ctx* c, const stk::fe* d_in, uint64_t n_in, uint64_t in_stride, stk::fe* d_out,
                   uint64_t out_stride, uint64_t n, uint64_t batch, const stk::fe& root, const stk::fe* r0,
                   uint64_t r0_stride);
// field-generic host helpers
stk::fe stk_h_mul(stk_ctx* c, const stk::fe& a, const stk::fe& b);
stk::fe stk_h_pow(stk_ctx* c, const stk::fe& a, uint64_t e);
stk::fe stk_h_inv(stk_ctx* c, const stk::fe& a);
stk::fe stk_h_to_tw(stk_ctx* c, const stk::fe& a);
