// ctx.h -- library context shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <initializer_list>
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

// Scratch slots: context-owned device buffers that grow on demand (stk_scratch), one owner each.
// A slot's contents live until its owner's next call.
enum stk_slot {
  kSlotNtt,           // transforms on the context stream: pass ping-pong, in-place staging (ntt_api.cu)
  kSlotLdeCoeffs,     // stk_lde / stk_lde_p2p: the coefficients when the caller keeps none
  kSlotStage,         // one call's small buffers: staged host arrays, counters, branch records
  kSlotHostNtt,       // stk_ntt_host: each copy stream's transform temporaries (3 slots) ...
  kSlotHostNttBufs = kSlotHostNtt + 3,  // ... and the three streams' input and output buffers
  kSlotFriLayers,     // stk_fri_prove: folded columns and their trees
  kSlotFriStage,      // stk_fri_prove: query indices and branch records
  kSlotCounter,       // stk_count_noncanonical: its counter outlives the call when sync = 0
  kSlotLdeHost,       // stk_lde_commit_host: the two upload slots
  kSlotPolyEvals,     // mul_low's evaluations (poly.cu).  Every mul_low call writes here, so nothing
                      // that must survive a mul_low call may live in this slot.
  kSlotPolyDiv,       // stk_poly_divmod: f, g, rev(a) and a product
  kSlotPolyA,         // composition and multivariate evaluation (poly.cu): two buffers
  kSlotPolyB,
  kScratchSlots
};

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
  void* scratch[kScratchSlots] = {};
  uint64_t scratch_bytes[kScratchSlots] = {};
  std::string err;
};

#define STK_API extern "C" __attribute__((visibility("default")))

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

// Launches for the context's field: fn(f) receives StarkField() or the run-time MontField, so a
// kernel template launched as k<<<...>>>(..., f) is instantiated for both; the launch is checked.
template <class Fn>
int stk_with_field(stk_ctx* c, Fn&& fn) {
  if (c->is_stark) fn(stk::StarkField());
  else fn(c->mont);
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

// ceil(log2(x)): the least l with 2^l >= x
static inline int stk_ilog2(uint64_t x) {
  int l = 0;
  while ((1ull << l) < x) ++l;
  return l;
}

// internal helpers (ntt_api.cu)
int stk_scratch(stk_ctx* c, int slot, uint64_t bytes, void** out);
// One host-to-device copy into a scratch slot: `bytes` from h to byte offset `off`.
struct stk_upload {
  uint64_t off;
  const void* h;
  uint64_t bytes;
};
// Grows `slot` to `bytes`, copies the host arrays into it and waits for the copies: the arrays
// belong to the caller's frame, which ends before the device reads them.
int stk_stage(stk_ctx* c, int slot, uint64_t bytes, std::initializer_list<stk_upload> ups, void** out);
int stk_get_table(stk_ctx* c, const stk::fe& root, uint64_t n, const stk::fe** d_table);
// Same, but may return a longer cached table T (order n*stride, T.root^stride == root) to be
// indexed as T[e*stride]: sub-transforms (G1 = G2^ext, FRI layers' roots w^4, w^16, ...)
// reuse the big table instead of building and caching their own.
int stk_get_table_strided(stk_ctx* c, const stk::fe& root, uint64_t n, const stk::fe** d_table, uint64_t* stride);
// Same for kernels that index T[e << shift]: a longer table at a stride that is not a power of
// two is passed over for one of order n.
int stk_get_table_shift(stk_ctx* c, const stk::fe& root, uint64_t n, const stk::fe** d_table, int* shift);
stk::fe stk_load_fe(const uint32_t* w);
// forward transform whose final pass scatters every row to the rank owning its Merkle leaf
// (sharded commit, see ntt.cuh peer_on = 2): ptrs holds the nranks exchange buffers
// (columns_total x n/nranks elements each), col_base the global index of the first column
int stk_ntt_dev_peer(stk_ctx* c, const stk::fe* d_in, uint64_t n_in, uint64_t in_stride, uint64_t n, uint64_t batch,
                     const stk::fe& root, uint64_t nranks, uint64_t col_base, const uint64_t* ptrs);
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
stk::fe stk_h_one(stk_ctx* c);
// root^n == 1 and root^(n/2) != 1: for n a power of two, root has order exactly n
bool stk_h_primitive(stk_ctx* c, const stk::fe& root, uint64_t n);
