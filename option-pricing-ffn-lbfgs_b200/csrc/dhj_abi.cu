// dhj_abi.cu — host side of libdhj.so: contexts, device/pinned buffers, option books, and the extern "C"
// entry points declared in include/dhj.h.  No torch, no Python: plain CUDA runtime.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>
#include <omp.h>

#include "dhj.h"
#include "dhj_kernels.cuh"
#include "dhj_greeks.cuh"
#include "dhj_jac.cuh"
#include "dhj_generate.cuh"
#include "dhj_iv.cuh"
#include "dhj_ivloss.cuh"
#include "dhj_mc.cuh"

using namespace dhj;

extern "C" int dhj_host_threads();      // dhj_lbfgs.cpp: threads of the host-side parallel loops
extern "C" int dhj_lbfgs_shape(const dhj_lbfgs* opt, int64_t* n, int32_t* dim);   // dhj_lbfgs.cpp: states, dimension

namespace {

char g_init_error[512] = "";

// A growable buffer of device (DevBuf) or pinned host (PinBuf) memory
template <cudaError_t (*Alloc)(void**, size_t), cudaError_t (*Free)(void*)>
struct Buf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) Free(p);
    p = nullptr; cap = 0;
    size_t want = std::max(bytes, (size_t)256);
    cudaError_t e = Alloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) Free(p); p = nullptr; cap = 0; }
};
using DevBuf = Buf<cudaMalloc, cudaFree>;
using PinBuf = Buf<cudaMallocHost, cudaFreeHost>;

// Host description of the option slices (options grouped by maturity, first-appearance order).
struct BookHost {
  int M = 0, n_slices = 0, max_slice = 0;
  std::vector<double> slice_T;
  std::vector<int> slice_off, pos;
  std::vector<unsigned char> call;
  void group(const double* maturity, const int32_t* is_call, int m) {
    M = m;
    slice_T.clear();
    std::vector<int> slice_of(m);
    for (int o = 0; o < m; ++o) {
      int s = -1;
      for (size_t t = 0; t < slice_T.size(); ++t)
        if (slice_T[t] == maturity[o] || (std::isnan(slice_T[t]) && std::isnan(maturity[o]))) { s = (int)t; break; }
      if (s < 0) { s = (int)slice_T.size(); slice_T.push_back(maturity[o]); }
      slice_of[o] = s;
    }
    n_slices = (int)slice_T.size();
    slice_off.assign(n_slices + 1, 0);
    for (int o = 0; o < m; ++o) slice_off[slice_of[o] + 1]++;
    max_slice = 0;
    for (int s = 0; s < n_slices; ++s) { max_slice = std::max(max_slice, slice_off[s + 1]); slice_off[s + 1] += slice_off[s]; }
    pos.assign(m, 0); call.assign(m, 0);
    std::vector<int> fill(slice_off.begin(), slice_off.end() - 1);
    for (int o = 0; o < m; ++o) {
      int d = fill[slice_of[o]]++;
      pos[d] = o;
      call[d] = is_call[o] ? 1 : 0;
    }
  }
  void grid(const double* maturities, int nT, int nK, int is_call_flag) {
    M = nT * nK; n_slices = nT; max_slice = nK;
    slice_T.assign(maturities, maturities + nT);
    slice_off.resize(nT + 1);
    for (int t = 0; t <= nT; ++t) slice_off[t] = t * nK;
    pos.resize(M); call.assign(M, is_call_flag ? 1 : 0);
    for (int o = 0; o < M; ++o) pos[o] = o;
  }
  // bytes of the packed device image: slice_T | slice_off | pos | call (8-byte aligned segments)
  size_t packed_bytes() const {
    return align8(n_slices * sizeof(double)) + align8((n_slices + 1) * sizeof(int)) + align8(M * sizeof(int)) +
           align8(M);
  }
  static size_t align8(size_t b) { return (b + 7) & ~(size_t)7; }
  void pack(unsigned char* dst) const {
    size_t o = 0;
    memcpy(dst + o, slice_T.data(), n_slices * sizeof(double)); o += align8(n_slices * sizeof(double));
    memcpy(dst + o, slice_off.data(), (n_slices + 1) * sizeof(int)); o += align8((n_slices + 1) * sizeof(int));
    memcpy(dst + o, pos.data(), M * sizeof(int)); o += align8(M * sizeof(int));
    memcpy(dst + o, call.data(), M);
  }
  void view(SliceView* v, const unsigned char* dbase) const {
    size_t o = 0;
    v->n_slices = n_slices; v->n_options = M;
    v->slice_T = (const double*)(dbase + o); o += align8(n_slices * sizeof(double));
    v->slice_off = (const int*)(dbase + o); o += align8((n_slices + 1) * sizeof(int));
    v->pos = (const int*)(dbase + o); o += align8(M * sizeof(int));
    v->call = dbase + o;
  }
};

// Option books (packed slice tables + shared strike row) live in a small ring of device slots, so that a call
// with a new (K, T) table neither waits for the device nor disturbs launches that still read an older table
// (DoubleHeston(...).pricing() changes the book on every call; the previous design synchronised the whole device).
constexpr int kBookSlots = 8;
struct BookSlot {
  DevBuf d;
  PinBuf h;
  std::vector<unsigned char> image;     // what the slot holds (empty: nothing)
  cudaEvent_t uploaded = nullptr;        // the H2D copy of `image`
  cudaEvent_t last_use = nullptr;        // the last launch that reads the slot
  cudaStream_t upload_stream = nullptr;
};

// Chunks of a host-buffer call rotate through three slots (stream + device buffers + pinned staging each): a slot's
// upload, kernel and download are serialised by its stream, so with two slots a chunk every (H2D + kernel + D2H) / 2
// is the best the pipeline can do — slower than the kernel as soon as the host link gives a rank less than ~20 GB/s
// (eight ranks copying at once on one host: 11.5 GB/s down per GPU, measured; profiles/README.md r02).
constexpr int kSlots = 3;
struct Slot {
  cudaStream_t stream = nullptr;
  cudaEvent_t done = nullptr;
  DevBuf d_in, d_out;
  PinBuf h_in, h_out;
  // deferred copy-out of a staged chunk
  double* user_out = nullptr;
  size_t out_bytes = 0;
  bool pending = false;
  // generator path: several destination arrays per chunk
  struct Piece { void* dst; size_t off, bytes; };
  std::vector<Piece> pieces;
  void drain_pieces(void (*copy)(void*, const void*, size_t)) {
    for (const Piece& pc : pieces) copy(pc.dst, (const unsigned char*)h_out.p + pc.off, pc.bytes);
    pieces.clear();
  }
};

}  // namespace

struct dhj_ctx {
  int device = 0;
  int sm_count = 0;
  int loss_blocks_per_sm = 1;
  cudaStream_t stream = nullptr;
  int64_t launches = 0;
  char err[512] = "";
  // cached option books for the pricing entry points
  BookSlot books[kBookSlots];
  int book_next = 0;                          // ring position of the next slot to overwrite
  int book_cur = 0;                           // slot of the last upload_book call
  Slot slots[kSlots];
  // loss path
  DevBuf d_x, d_xv, d_idx, d_f, d_fg, d_counters, d_prices, d_jac;
  DevBuf d_ivres;                             // IV objective: model vols | 1 / vega per unit and option
  PinBuf h_x, h_res;
  size_t counters_zeroed = 0;
  DevBuf d_peak;
  DevBuf d_mc_in, d_mc_part, d_mc_out;          // dhj_mc_price: inputs, chunk partials + carried sums, outputs
  // device buffers of destroyed markets, kept for the next dhj_market_create: cudaMalloc / cudaFree synchronise the
  // whole device, which stalls the other lock-step pipelines of a calibrate_many call every time a market comes or goes
  std::vector<DevBuf> pool;
  cudaError_t pool_take(DevBuf* out, size_t bytes) {
    int best = -1;
    for (size_t i = 0; i < pool.size(); ++i)
      if (pool[i].cap >= bytes && (best < 0 || pool[i].cap < pool[(size_t)best].cap)) best = (int)i;
    if (best >= 0 && pool[(size_t)best].cap <= 4 * std::max(bytes, (size_t)4096)) {
      *out = pool[(size_t)best];
      pool.erase(pool.begin() + best);
      return cudaSuccess;
    }
    *out = DevBuf();
    return out->reserve(bytes);
  }
  void pool_give(DevBuf* b) {
    if (b->p && pool.size() < 32 && b->cap <= ((size_t)256 << 20)) pool.push_back(*b);
    else b->release();
    b->p = nullptr; b->cap = 0;
  }
};

struct dhj_market {
  dhj_ctx* ctx = nullptr;
  int n_markets = 0, M = 0, N = 128;
  double r = 0.0;
  BookHost book;
  DevBuf d_book, d_strike, d_S0, d_price;
  long long strike_stride = 0;
  SliceView view{};
  // implied-volatility objective (dhj_market_set_objective): market vols [n_markets][M] (NaN: left out) and the
  // option tables in the caller's order, maturity[M] | is_call[M] (made on first use)
  int objective = DHJ_OBJECTIVE_PRICE;
  DevBuf d_mvol, d_ivtab;
};

namespace {

int fail(dhj_ctx* ctx, int code, const char* fmt, ...) {
  char* dst = ctx ? ctx->err : g_init_error;
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(dst, 512, fmt, ap);
  va_end(ap);
  return code;
}

#define DHJ_CUDA(ctx, call)                                                                          \
  do {                                                                                               \
    cudaError_t e__ = (call);                                                                        \
    if (e__ != cudaSuccess)                                                                          \
      return fail((ctx), e__ == cudaErrorMemoryAllocation ? DHJ_ERR_NOMEM : DHJ_ERR_CUDA,            \
                  "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__);     \
  } while (0)

// after every kernel launch: the launch's own error, and the count of dhj_launch_count
#define DHJ_LAUNCHED(ctx)                    \
  do {                                       \
    DHJ_CUDA((ctx), cudaGetLastError());     \
    (ctx)->launches++;                       \
  } while (0)

// a 1-D grid of `blocks` blocks, clamped to what one launch takes
int grid_1d(long long blocks) { return (int)std::max<long long>(1, std::min(blocks, 2147483647LL)); }

// the grid of the grid-stride elementwise kernels (implied vol, Black-Scholes price, IV residual) over n elements
int grid_stride_blocks(const dhj_ctx* ctx, long long n) {
  return (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, 32LL * ctx->sm_count));
}

// staging copies between the caller's pageable memory and the pinned slots: a single thread moves ~10 GB/s, less
// than the kernel consumes per chunk, so large copies are split over eight host threads (four: 14.75 ms per
// 1 Mi-set grid from pageable memory, eight: 14.28)
int copy_threads() { return std::max(1, std::min(8, dhj_host_threads())); }

void host_copy(void* dst, const void* src, size_t bytes) {
  constexpr size_t kPiece = (size_t)1 << 18;
  if (bytes < 4 * kPiece) { memcpy(dst, src, bytes); return; }
  const long long pieces = (long long)((bytes + kPiece - 1) / kPiece);
#pragma omp parallel for schedule(static) num_threads(copy_threads())
  for (long long i = 0; i < pieces; ++i) {
    const size_t off = (size_t)i * kPiece;
    memcpy((char*)dst + off, (const char*)src + off, std::min(kPiece, bytes - off));
  }
}

bool is_pinned_host(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeHost;
}

// Batch size of the batch engine for a launch of `n_units` units of `items_per_unit` items each (pricing: unit = item).
// A block's time is its phase 1 (one warp, ~0.9 item times) plus that of its busiest warp (items are dealt to the four
// warps in turn); a launch's time is the number of waves of resident blocks times that.  Minimise
// waves x (0.9 + ceil(items per batch / 4)) over whole units per batch; ties go to the larger batch.  E.g. 7 000 loss
// evaluations of a 3-slice market: 10 units per batch = 700 blocks = 2 waves (the second nearly empty) of 8 items per
// warp, 4 units per batch = 3 waves of 3.  Large launches end at full batches, a single calibration at one unit per
// block (every unit on its own SM: latency).
int pick_units_per_batch(long long n_units, int items_per_unit, int max_items, long long resident_blocks) {
  const int upb_max = std::max(1, max_items / std::max(1, items_per_unit));
  long long best_cost = -1;
  int best = 1;
  for (int upb = upb_max; upb >= 1; --upb) {
    const long long blocks = (n_units + upb - 1) / upb;
    const long long waves = (blocks + resident_blocks - 1) / resident_blocks;
    const long long cost = waves * (9 + 10 * (((long long)upb * items_per_unit + kBatchWarps - 1) / kBatchWarps));
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = upb; }
  }
  return best;
}

// k_price_batch handles slices of <= 8 strikes (warp per item, lane per k, <= 32 items per block); k_price_dense the rest
int launch_price(dhj_ctx* ctx, const SliceView& v, PriceArgs a, int max_slice, cudaStream_t st);

int launch_price(dhj_ctx* ctx, const SliceView& v, PriceArgs a, int max_slice, cudaStream_t st) {
  const long long items = a.P * (long long)v.n_slices;
  if (max_slice <= kBatchMaxStrikes) {
    // full batches of 32 items unless the launch is only a few waves long (mid-size loss rounds through the split path)
    const long long resident = (long long)ctx->sm_count * ctx->loss_blocks_per_sm;
    a.items_per_batch = (items > 64 * resident * kPriceItems) ? kPriceItems
                                                              : pick_units_per_batch(items, 1, kPriceItems, resident);
    const long long batches = (items + a.items_per_batch - 1) / a.items_per_batch;
    // one block per batch: the hardware block scheduler balances the SMs dynamically (a persistent grid with a
    // static batch -> block map measured ~3 % slower: the slowest SM sets the time)
    // DHJ_DEBUG_EXTRA_SMEM (bytes): developer knob that pads the launch with unused dynamic shared memory to
    // lower the resident block count (occupancy experiments, profiles/README.md); never set in production
    static const size_t extra = [] {
      const char* e = getenv("DHJ_DEBUG_EXTRA_SMEM");
      size_t b = e ? (size_t)atol(e) : 0;
      if (b) cudaFuncSetAttribute(k_price_batch<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b);
      return b;
    }();
    const int grid = grid_1d(batches);
    if (a.items_per_batch == kPriceItems) k_price_batch<true><<<grid, kBatchThreads, extra, st>>>(v, a);
    else k_price_batch<false><<<grid, kBatchThreads, 0, st>>>(v, a);
  } else {
    // a warp per item, four items per block; the block's shared memory (four private strike tables) exceeds the
    // 48 KB static limit: opt in once
    static const cudaError_t attr = cudaFuncSetAttribute(k_price_dense, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                         (int)sizeof(DenseSmem));
    DHJ_CUDA(ctx, attr);
    const long long blocks = (items + kDenseWarps - 1) / kDenseWarps;
    k_price_dense<<<grid_1d(blocks), 32 * kDenseWarps, sizeof(DenseSmem), st>>>(v, a);
  }
  DHJ_LAUNCHED(ctx);
  return DHJ_OK;
}

// Find (or upload into the ring) a packed table image (an option book + shared strike table for a pricing call, or
// the option tables of an implied-vol call) on `stream`; *d_image is its device copy.
// No device-wide synchronisation: a new table goes to the least recently filled slot (after the last launch that
// read that slot has finished — normally long ago), its copy is ordered before the caller's launches by stream
// order or an event wait, and launches that still read other slots are not disturbed.
int upload_image(dhj_ctx* ctx, std::vector<unsigned char>& image, cudaStream_t stream, const unsigned char** d_image) {
  int hit = -1;
  for (int i = 0; i < kBookSlots && hit < 0; ++i)
    if (ctx->books[i].image == image) hit = i;
  if (hit < 0) {
    hit = ctx->book_next;
    ctx->book_next = (ctx->book_next + 1) % kBookSlots;
    BookSlot& b = ctx->books[hit];
    b.image.clear();
    // the slot's device table may still be read, its pinned staging may still feed the previous upload
    DHJ_CUDA(ctx, cudaEventSynchronize(b.last_use));
    DHJ_CUDA(ctx, cudaEventSynchronize(b.uploaded));
    DHJ_CUDA(ctx, b.d.reserve(image.size()));
    DHJ_CUDA(ctx, b.h.reserve(image.size()));
    memcpy(b.h.p, image.data(), image.size());
    DHJ_CUDA(ctx, cudaMemcpyAsync(b.d.p, b.h.p, image.size(), cudaMemcpyHostToDevice, stream));
    DHJ_CUDA(ctx, cudaEventRecord(b.uploaded, stream));
    b.upload_stream = stream;
    b.image.swap(image);
  } else if (ctx->books[hit].upload_stream != stream) {
    DHJ_CUDA(ctx, cudaStreamWaitEvent(stream, ctx->books[hit].uploaded, 0));
  }
  ctx->book_cur = hit;
  *d_image = (const unsigned char*)ctx->books[hit].d.p;
  return DHJ_OK;
}

int upload_book(dhj_ctx* ctx, const BookHost& book, const double* shared_strikes, int n_shared,
                cudaStream_t stream, SliceView* v) {
  const size_t bb = book.packed_bytes();
  const size_t sb = BookHost::align8((size_t)n_shared * sizeof(double));
  std::vector<unsigned char> image(bb + sb);
  book.pack(image.data());
  if (n_shared) memcpy(image.data() + bb, shared_strikes, (size_t)n_shared * sizeof(double));
  const unsigned char* d_image;
  int rc = upload_image(ctx, image, stream, &d_image);
  if (rc) return rc;
  book.view(v, d_image);
  v->strike = n_shared ? (const double*)(d_image + bb) : nullptr;
  v->strike_stride = 0;
  return DHJ_OK;
}

// the launches of the current call on `stream` read the current book slot
int book_used(dhj_ctx* ctx, cudaStream_t stream) {
  DHJ_CUDA(ctx, cudaEventRecord(ctx->books[ctx->book_cur].last_use, stream));
  return DHJ_OK;
}

int check_arrays(dhj_ctx* ctx, const void* in, int64_t P, const void* S0, const void* out) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (!in || !S0 || !out) return fail(ctx, DHJ_ERR_ARG, "null array argument");
  if (P < 0) return fail(ctx, DHJ_ERR_ARG, "P must be >= 0 (got %lld)", (long long)P);
  return DHJ_OK;
}

int check_common(dhj_ctx* ctx, const void* params, int64_t P, const void* S0, int32_t N, double L, const void* out) {
  int rc = check_arrays(ctx, params, P, S0, out);
  if (rc) return rc;
  if (N < 1) return fail(ctx, DHJ_ERR_ARG, "N must be >= 1 (got %d)", N);
  if (!(L == L)) return fail(ctx, DHJ_ERR_ARG, "L is NaN");
  return DHJ_OK;
}

// The option tables and strides of an option list (dhj_price_list's layout).  *empty: M == 0 or P == 0, nothing to
// compute; the tables are not looked at then.
int check_list(dhj_ctx* ctx, int64_t P, int64_t s0_stride, const double* strike, int64_t strike_stride,
               const double* maturity, const int32_t* is_call, int32_t M, bool* empty) {
  if (M < 0) return fail(ctx, DHJ_ERR_ARG, "M must be >= 0");
  *empty = M == 0 || P == 0;
  if (*empty) return DHJ_OK;
  if (!strike || !maturity || !is_call) return fail(ctx, DHJ_ERR_ARG, "null option table");
  if (s0_stride != 0 && s0_stride != 1) return fail(ctx, DHJ_ERR_ARG, "s0_stride must be 0 or 1");
  if (strike_stride != 0 && strike_stride != M) return fail(ctx, DHJ_ERR_ARG, "strike_stride must be 0 or M");
  return DHJ_OK;
}

// An option list priced by dhj_price_list, dhj_price_jacobian and dhj_price_greeks: the maturity book (and a shared
// strike row) in the book ring and the view over it.  A per-set strike row (strike_stride = M) is the caller's to
// point the view at.
struct OptionList {
  bool empty = true;
  SliceView v{};
  int max_slice = 0;
};

// out_der: the call's second output (dhj_price_list, which has none, passes out again)
int option_list(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride, double r,
                double q, const double* strike, int64_t strike_stride, const double* maturity, const int32_t* is_call,
                int32_t M, int32_t N, double L, const void* out, const void* out_der, OptionList* ol) {
  int rc = check_common(ctx, params, P, S0, N, L, out);
  if (rc) return rc;
  if (!out_der) return fail(ctx, DHJ_ERR_ARG, "null array argument");
  rc = check_list(ctx, P, s0_stride, strike, strike_stride, maturity, is_call, M, &ol->empty);
  if (rc || ol->empty) return rc;
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  BookHost book;
  book.group(maturity, is_call, M);
  rc = upload_book(ctx, book, strike_stride ? nullptr : strike, strike_stride ? 0 : M, ctx->stream, &ol->v);
  if (rc) return rc;
  ol->v.scale_by_spot = 0; ol->v.n_cos = N; ol->v.r = r; ol->v.q = q; ol->v.L = L;
  ol->max_slice = book.max_slice;
  return DHJ_OK;
}

// Chunked, double-buffered host-to-host pricing: params/S0/strike rows in, price rows out.
int run_price_host(dhj_ctx* ctx, SliceView v, int max_slice, const double* params, int64_t P, const double* S0,
                   int64_t s0_stride, const double* strike, int64_t strike_stride, double* out) {
  const int M = v.n_options;
  if (P == 0 || M == 0) return DHJ_OK;
  const size_t in_row = (size_t)kNumParams + (s0_stride ? 1 : 0) + (strike_stride ? (size_t)M : 0);
  const size_t row_doubles = in_row + (size_t)M;
  int64_t chunk = (int64_t)std::max<size_t>(256, std::min<size_t>(131072, ((size_t)1 << 23) / row_doubles));
  // a call that moves more than 16 MB is cut into at least 8 chunks so that transfers overlap kernels even when
  // one set is large (the 200 x 20 surface: 32 KB of prices per set, 1 024 sets -> 8 chunks of 128)
  if ((size_t)P * row_doubles * sizeof(double) > ((size_t)16 << 20))
    chunk = std::min<int64_t>(chunk, std::max<int64_t>(32, (P + 7) / 8));
  const bool pin_in = is_pinned_host(params) && (!s0_stride || is_pinned_host(S0)) &&
                      (!strike_stride || is_pinned_host(strike));
  const bool pin_out = is_pinned_host(out);
  // Chunk schedule: the first chunk's upload and the last chunk's download cannot overlap any kernel, so with
  // pinned buffers the schedule ramps up from chunk/8 and down to chunk/8 again (exposed transfer 0.54 -> 0.07 ms
  // on the 1 Mi-set grid: 13.87 -> 13.23 ms).  Pageable buffers keep uniform chunks: their staging copies make
  // the host the bottleneck while the chunks are small (14.3 vs 14.9 ms).
  std::vector<int64_t> sizes;
  {
    std::vector<int64_t> head, tail;
    int64_t left = P;
    if (pin_in && pin_out && chunk >= 1024)
      for (int64_t s = chunk / 8; s < chunk && left > 2 * s + chunk; s *= 2) {
        head.push_back(s); tail.push_back(s);
        left -= 2 * s;
      }
    sizes = head;
    for (; left > 0; left -= chunk) sizes.push_back(std::min(chunk, left));
    sizes.insert(sizes.end(), tail.rbegin(), tail.rend());
  }
  // A previous call on this context may have failed half-way (DHJ_ERR_NOMEM is recoverable) and left a staged
  // chunk behind: its caller's buffer is gone, so nothing of it may be copied out now.  Drain and forget.
  for (int i = 0; i < kSlots; ++i) {
    Slot& sl = ctx->slots[i];
    DHJ_CUDA(ctx, cudaEventSynchronize(sl.done));
    sl.pending = false; sl.user_out = nullptr; sl.out_bytes = 0; sl.pieces.clear();
    // the option book was uploaded on another stream
    DHJ_CUDA(ctx, cudaStreamWaitEvent(sl.stream, ctx->books[ctx->book_cur].uploaded, 0));
  }
  // DHJ_DEBUG_FAIL_AT_CHUNK (test hook, tests/test_gpu_dropin.py): return DHJ_ERR_NOMEM before that chunk is staged,
  // as a failed allocation would, with earlier chunks still in flight
  const char* fail_env = getenv("DHJ_DEBUG_FAIL_AT_CHUNK");
  const long fail_at = fail_env ? atol(fail_env) : -1;
  int slot_i = 0;
  int64_t lo = 0;
  for (size_t ci = 0; ci < sizes.size(); lo += sizes[ci], ++ci, slot_i = (slot_i + 1) % kSlots) {
    const int64_t n = sizes[ci];
    Slot& sl = ctx->slots[slot_i];
    if ((long)ci == fail_at) return fail(ctx, DHJ_ERR_NOMEM, "injected failure at chunk %ld (DHJ_DEBUG_FAIL_AT_CHUNK)", fail_at);
    // the slot's previous chunk must have left its buffers
    DHJ_CUDA(ctx, cudaEventSynchronize(sl.done));
    if (sl.pending) { host_copy(sl.user_out, sl.h_out.p, sl.out_bytes); sl.pending = false; }
    const size_t pb = (size_t)n * kNumParams * sizeof(double);
    const size_t s0b = s0_stride ? (size_t)n * sizeof(double) : sizeof(double);
    const size_t kb = strike_stride ? (size_t)n * M * sizeof(double) : 0;
    const size_t ob = (size_t)n * M * sizeof(double);
    DHJ_CUDA(ctx, sl.d_in.reserve(pb + s0b + kb));
    DHJ_CUDA(ctx, sl.d_out.reserve(ob));
    unsigned char* din = (unsigned char*)sl.d_in.p;
    const double* src_params = params + lo * kNumParams;
    const double* src_s0 = s0_stride ? S0 + lo : S0;
    const double* src_strike = strike_stride ? strike + lo * (int64_t)M : nullptr;
    if (pin_in) {
      DHJ_CUDA(ctx, cudaMemcpyAsync(din, src_params, pb, cudaMemcpyHostToDevice, sl.stream));
      DHJ_CUDA(ctx, cudaMemcpyAsync(din + pb, src_s0, s0b, cudaMemcpyHostToDevice, sl.stream));
      if (kb) DHJ_CUDA(ctx, cudaMemcpyAsync(din + pb + s0b, src_strike, kb, cudaMemcpyHostToDevice, sl.stream));
    } else {
      DHJ_CUDA(ctx, sl.h_in.reserve(pb + s0b + kb));
      unsigned char* hin = (unsigned char*)sl.h_in.p;
      host_copy(hin, src_params, pb);
      host_copy(hin + pb, src_s0, s0b);
      if (kb) host_copy(hin + pb + s0b, src_strike, kb);
      DHJ_CUDA(ctx, cudaMemcpyAsync(din, hin, pb + s0b + kb, cudaMemcpyHostToDevice, sl.stream));
    }
    SliceView vv = v;
    if (strike_stride) { vv.strike = (const double*)(din + pb + s0b); vv.strike_stride = M; }
    PriceArgs a;
    a.params = (const double*)din; a.S0 = (const double*)(din + pb); a.s0_stride = s0_stride ? 1 : 0;
    a.row_index = nullptr; a.P = n; a.transform = 0; a.out = (double*)sl.d_out.p;
    int rc = launch_price(ctx, vv, a, max_slice, sl.stream);
    if (rc) return rc;
    double* dst = out + lo * (int64_t)M;
    if (pin_out) {
      DHJ_CUDA(ctx, cudaMemcpyAsync(dst, sl.d_out.p, ob, cudaMemcpyDeviceToHost, sl.stream));
    } else {
      DHJ_CUDA(ctx, sl.h_out.reserve(ob));
      DHJ_CUDA(ctx, cudaMemcpyAsync(sl.h_out.p, sl.d_out.p, ob, cudaMemcpyDeviceToHost, sl.stream));
      sl.user_out = dst; sl.out_bytes = ob; sl.pending = true;
    }
    DHJ_CUDA(ctx, cudaEventRecord(sl.done, sl.stream));
  }
  for (int i = 0; i < kSlots; ++i) {
    Slot& sl = ctx->slots[i];
    DHJ_CUDA(ctx, cudaEventSynchronize(sl.done));
    if (sl.pending) { host_copy(sl.user_out, sl.h_out.p, sl.out_bytes); sl.pending = false; }
  }
  return DHJ_OK;
}

int stage_x(dhj_ctx* ctx, const dhj_market* mk, const double* x, const int32_t* market_index, int64_t B,
            const int** d_index) {
  if (!ctx || !mk) return fail(ctx, DHJ_ERR_ARG, "null context or market");
  if (mk->ctx != ctx) return fail(ctx, DHJ_ERR_ARG, "market belongs to another context");
  if (!x) return fail(ctx, DHJ_ERR_ARG, "null x");
  if (B < 0 || B > (int64_t)100000000) return fail(ctx, DHJ_ERR_ARG, "bad batch size %lld", (long long)B);
  const size_t xb = (size_t)B * kNumParams * sizeof(double);
  const size_t ib = market_index ? (size_t)B * sizeof(int) : 0;
  if (market_index)
    for (int64_t i = 0; i < B; ++i)
      if (market_index[i] < 0 || market_index[i] >= mk->n_markets)
        return fail(ctx, DHJ_ERR_ARG, "market_index[%lld] = %d out of range [0,%d)", (long long)i,
                    market_index[i], mk->n_markets);
  DHJ_CUDA(ctx, ctx->h_x.reserve(xb + ib));
  DHJ_CUDA(ctx, ctx->d_x.reserve(xb + ib));
  host_copy(ctx->h_x.p, x, xb);
  if (ib) memcpy((unsigned char*)ctx->h_x.p + xb, market_index, ib);
  DHJ_CUDA(ctx, cudaMemcpyAsync(ctx->d_x.p, ctx->h_x.p, xb + ib, cudaMemcpyHostToDevice, ctx->stream));
  *d_index = ib ? (const int*)((unsigned char*)ctx->d_x.p + xb) : nullptr;
  return DHJ_OK;
}

// The B x staged by stage_x, transformed by k_fd_expand (fd: into the kFdPoints stencil points of each) into d_xv /
// d_idx, and the arguments of the market's pricing launch over those points (out is the caller's to set).
int expand_x(dhj_ctx* ctx, const dhj_market* mk, const int* d_index, int64_t B, int fd, double h, PriceArgs* pa) {
  const int64_t n = B * (fd ? kFdPoints : 1);
  DHJ_CUDA(ctx, ctx->d_xv.reserve((size_t)n * kNumParams * sizeof(double)));
  DHJ_CUDA(ctx, ctx->d_idx.reserve((size_t)n * sizeof(int)));
  k_fd_expand<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((const double*)ctx->d_x.p, d_index, B, fd, h,
                                                                   (double*)ctx->d_xv.p, (int*)ctx->d_idx.p);
  DHJ_LAUNCHED(ctx);
  pa->params = (const double*)ctx->d_xv.p; pa->S0 = (const double*)mk->d_S0.p; pa->s0_stride = 1;
  pa->row_index = (const int*)ctx->d_idx.p; pa->P = n; pa->transform = 0; pa->out = nullptr;
  return DHJ_OK;
}

// (f, g) of B evaluations from d_fg (kFdPoints doubles each: f, then g) into out_f[B] and out_g[B][13]; out_f_all
// (may be null) receives the kFdPoints losses per evaluation in d_f
int download_fg(dhj_ctx* ctx, int64_t B, double* out_f, double* out_g, double* out_f_all) {
  const size_t bytes = (size_t)B * kFdPoints * sizeof(double);
  DHJ_CUDA(ctx, ctx->h_res.reserve(bytes * (out_f_all ? 2 : 1)));
  DHJ_CUDA(ctx, cudaMemcpyAsync(ctx->h_res.p, ctx->d_fg.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (out_f_all)
    DHJ_CUDA(ctx, cudaMemcpyAsync((unsigned char*)ctx->h_res.p + bytes, ctx->d_f.p, bytes, cudaMemcpyDeviceToHost,
                                  ctx->stream));
  DHJ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  const double* res = (const double*)ctx->h_res.p;
  if (out_f_all) host_copy(out_f_all, res + B * kFdPoints, bytes);
#pragma omp parallel for schedule(static) num_threads(copy_threads()) if (B >= 4096)
  for (int64_t c = 0; c < B; ++c) {
    out_f[c] = res[c * kFdPoints];
    memcpy(out_g + c * kNumParams, res + c * kFdPoints + 1, kNumParams * sizeof(double));
  }
  return DHJ_OK;
}

// One host array of a synchronous staged call (stage_sync): an input (`in`) or an output (`out`) of `row` bytes per
// row, or an input of `fixed` bytes that every chunk shares (a shared table, a scalar S0).  A segment without a host
// array is not staged and its device pointer is null, but its row still counts towards the chunk size.
struct Seg {
  const void* in;
  void* out;
  size_t row, fixed;
};
Seg rows_in(const void* p, size_t row) { return {p, nullptr, row, 0}; }
Seg rows_out(void* p, size_t row) { return {nullptr, p, row, 0}; }
Seg table_in(const void* p, size_t bytes) { return {p, nullptr, 0, bytes}; }
Seg s0_in(const double* S0, int64_t s0_stride) {
  return s0_stride ? rows_in(S0, sizeof(double)) : table_in(S0, sizeof(double));
}
// a strike row per row (strike_stride = M); a shared strike row travels in the book ring instead
Seg strike_in(const double* strike, int64_t strike_stride) {
  return rows_in(strike_stride ? strike : nullptr, (size_t)strike_stride * sizeof(double));
}

constexpr size_t kStageChunkBytes = (size_t)32 << 20;
constexpr size_t kOneChunk = SIZE_MAX;   // the whole call in one chunk (one launch)

// Host arrays in -> launch(n, d) -> host arrays out, synchronously through the context's staging buffers, for the
// entry points whose throughput is not a goal.  Rows [0, rows) go in chunks of as many rows as fit in chunk_bytes
// (at least one); per chunk one upload, the launch callback (d[i]: the device copy of segment i's rows of the chunk)
// and one download.
template <size_t N, class Launch>
int stage_sync(dhj_ctx* ctx, int64_t rows, size_t chunk_bytes, const Seg (&segs)[N], Launch launch) {
  size_t row = 0;
  for (const Seg& s : segs) row += s.row;
  const int64_t chunk =
      (int64_t)std::max<size_t>(1, std::min<size_t>((size_t)rows, chunk_bytes / std::max<size_t>(row, 1)));
  // a chunk of n rows: the inputs packed in h_x / d_x, the outputs in d_prices / h_res, 8-byte aligned
  size_t off[N], bytes[N], in_bytes = 0, out_bytes = 0;
  auto layout = [&](int64_t n) {
    in_bytes = out_bytes = 0;
    for (size_t i = 0; i < N; ++i) {
      size_t& end = segs[i].out ? out_bytes : in_bytes;
      off[i] = end;
      bytes[i] = (segs[i].in || segs[i].out) ? (segs[i].row ? (size_t)n * segs[i].row : segs[i].fixed) : 0;
      end += BookHost::align8(bytes[i]);
    }
  };
  layout(chunk);
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  DHJ_CUDA(ctx, ctx->h_x.reserve(in_bytes));
  DHJ_CUDA(ctx, ctx->d_x.reserve(in_bytes));
  DHJ_CUDA(ctx, ctx->d_prices.reserve(out_bytes));
  DHJ_CUDA(ctx, ctx->h_res.reserve(out_bytes));
  unsigned char* hin = (unsigned char*)ctx->h_x.p;
  const unsigned char* hout = (const unsigned char*)ctx->h_res.p;
  for (int64_t lo = 0; lo < rows; lo += chunk) {
    const int64_t n = std::min(chunk, rows - lo);
    layout(n);
    void* d[N];
    for (size_t i = 0; i < N; ++i) {
      const Seg& s = segs[i];
      d[i] = nullptr;
      if (s.in) {
        host_copy(hin + off[i], (const unsigned char*)s.in + (size_t)lo * s.row, bytes[i]);
        d[i] = (unsigned char*)ctx->d_x.p + off[i];
      } else if (s.out) {
        d[i] = (unsigned char*)ctx->d_prices.p + off[i];
      }
    }
    DHJ_CUDA(ctx, cudaMemcpyAsync(ctx->d_x.p, hin, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    int rc = launch(n, (void* const*)d);
    if (rc) return rc;
    DHJ_CUDA(ctx, cudaMemcpyAsync(ctx->h_res.p, ctx->d_prices.p, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    DHJ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < N; ++i)
      if (segs[i].out) host_copy((unsigned char*)segs[i].out + (size_t)lo * segs[i].row, hout + off[i], bytes[i]);
  }
  return DHJ_OK;
}

}  // namespace

// ================================================================================================
extern "C" {

int dhj_abi_version(void) { return DHJ_ABI_VERSION; }

int dhj_device_count(int* count) {
  if (!count) return fail(nullptr, DHJ_ERR_ARG, "null count");
  cudaError_t e = cudaGetDeviceCount(count);
  if (e != cudaSuccess) {
    *count = 0;
    cudaGetLastError();
    return fail(nullptr, DHJ_ERR_CUDA, "cudaGetDeviceCount failed: %s", cudaGetErrorString(e));
  }
  return DHJ_OK;
}

int dhj_init(int device, dhj_ctx** out) {
  if (!out) return fail(nullptr, DHJ_ERR_ARG, "null ctx pointer");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    return fail(nullptr, DHJ_ERR_CUDA, "no CUDA device available (%s); libdhj has no CPU fallback",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
  }
  if (device < 0 || device >= n) return fail(nullptr, DHJ_ERR_ARG, "device %d out of range [0,%d)", device, n);
  cudaDeviceProp prop;
  DHJ_CUDA(nullptr, cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(nullptr, DHJ_ERR_CUDA, "device %d is sm_%d%d; libdhj is built for sm_100a (B200) only", device,
                prop.major, prop.minor);
  DHJ_CUDA(nullptr, cudaSetDevice(device));
  dhj_ctx* ctx = new (std::nothrow) dhj_ctx();
  if (!ctx) return fail(nullptr, DHJ_ERR_NOMEM, "out of host memory");
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  cudaError_t e2 = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  for (int i = 0; i < kBookSlots && e2 == cudaSuccess; ++i) {
    e2 = cudaEventCreateWithFlags(&ctx->books[i].uploaded, cudaEventDisableTiming);
    if (e2 == cudaSuccess) e2 = cudaEventCreateWithFlags(&ctx->books[i].last_use, cudaEventDisableTiming);
  }
  for (int i = 0; i < kSlots && e2 == cudaSuccess; ++i) {
    e2 = cudaStreamCreateWithFlags(&ctx->slots[i].stream, cudaStreamNonBlocking);
    if (e2 == cudaSuccess) e2 = cudaEventCreateWithFlags(&ctx->slots[i].done, cudaEventDisableTiming);
    if (e2 == cudaSuccess) e2 = cudaEventRecord(ctx->slots[i].done, ctx->slots[i].stream);
  }
  int bps = 0;
  if (e2 == cudaSuccess)
    e2 = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_loss_batch, kBatchThreads, 0);
  if (e2 != cudaSuccess) {
    fail(nullptr, DHJ_ERR_CUDA, "context setup failed: %s", cudaGetErrorString(e2));
    dhj_destroy(ctx);
    return DHJ_ERR_CUDA;
  }
  ctx->loss_blocks_per_sm = std::max(1, bps);
  *out = ctx;
  return DHJ_OK;
}

int dhj_destroy(dhj_ctx* ctx) {
  if (!ctx) return DHJ_OK;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (int i = 0; i < kSlots; ++i) {
    Slot& s = ctx->slots[i];
    s.d_in.release(); s.d_out.release(); s.h_in.release(); s.h_out.release();
    if (s.done) cudaEventDestroy(s.done);
    if (s.stream) cudaStreamDestroy(s.stream);
  }
  for (int i = 0; i < kBookSlots; ++i) {
    BookSlot& b = ctx->books[i];
    b.d.release(); b.h.release();
    if (b.uploaded) cudaEventDestroy(b.uploaded);
    if (b.last_use) cudaEventDestroy(b.last_use);
  }
  ctx->d_x.release(); ctx->d_xv.release(); ctx->d_idx.release(); ctx->d_f.release(); ctx->d_fg.release();
  ctx->d_counters.release(); ctx->d_prices.release(); ctx->d_jac.release(); ctx->h_x.release(); ctx->h_res.release();
  ctx->d_peak.release(); ctx->d_ivres.release();
  ctx->d_mc_in.release(); ctx->d_mc_part.release(); ctx->d_mc_out.release();
  for (DevBuf& b : ctx->pool) b.release();
  ctx->pool.clear();
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return DHJ_OK;
}

const char* dhj_last_error(const dhj_ctx* ctx) { return ctx ? ctx->err : g_init_error; }

int dhj_launch_count(const dhj_ctx* ctx, int64_t* count) {
  if (!ctx || !count) return DHJ_ERR_ARG;
  *count = ctx->launches;
  return DHJ_OK;
}

// ---- pricing ---------------------------------------------------------------------------------
int dhj_price_list(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride,
                   double r, double q, const double* strike, int64_t strike_stride, const double* maturity,
                   const int32_t* is_call, int32_t M, int32_t N, double L, double* out) {
  OptionList ol;
  int rc = option_list(ctx, params, P, S0, s0_stride, r, q, strike, strike_stride, maturity, is_call, M, N, L, out,
                       out, &ol);
  if (rc || ol.empty) return rc;
  return run_price_host(ctx, ol.v, ol.max_slice, params, P, S0, s0_stride, strike, strike_stride, out);
}

static int grid_view(dhj_ctx* ctx, const double* strikes, int32_t nK, const double* maturities, int32_t nT,
                     int32_t scale_by_spot, int32_t is_call, int32_t N, double r, double q, double L,
                     cudaStream_t stream, SliceView* v) {
  if (nK < 1 || nT < 1) return fail(ctx, DHJ_ERR_ARG, "nK and nT must be >= 1");
  if (!strikes || !maturities) return fail(ctx, DHJ_ERR_ARG, "null grid table");
  BookHost book;
  book.grid(maturities, nT, nK, is_call);
  std::vector<double> tiled((size_t)nT * nK);
  for (int t = 0; t < nT; ++t) memcpy(tiled.data() + (size_t)t * nK, strikes, (size_t)nK * sizeof(double));
  int rc = upload_book(ctx, book, tiled.data(), nT * nK, stream, v);
  if (rc) return rc;
  v->scale_by_spot = scale_by_spot ? 1 : 0; v->n_cos = N; v->r = r; v->q = q; v->L = L;
  return DHJ_OK;
}

int dhj_price_grid(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride,
                   double r, double q, const double* strikes, int32_t nK, const double* maturities,
                   int32_t nT, int32_t scale_by_spot, int32_t is_call, int32_t N, double L, double* out) {
  int rc = check_common(ctx, params, P, S0, N, L, out);
  if (rc) return rc;
  if (s0_stride != 0 && s0_stride != 1) return fail(ctx, DHJ_ERR_ARG, "s0_stride must be 0 or 1");
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  SliceView v;
  rc = grid_view(ctx, strikes, nK, maturities, nT, scale_by_spot, is_call, N, r, q, L, ctx->stream, &v);
  if (rc) return rc;
  if (P == 0) return DHJ_OK;
  return run_price_host(ctx, v, nK, params, P, S0, s0_stride, nullptr, 0, out);
}

int dhj_price_grid_dev(dhj_ctx* ctx, const double* d_params, int64_t P, const double* d_S0,
                       int64_t s0_stride, double r, double q, const double* strikes, int32_t nK,
                       const double* maturities, int32_t nT, int32_t scale_by_spot, int32_t is_call,
                       int32_t N, double L, double* d_out, void* stream) {
  int rc = check_common(ctx, d_params, P, d_S0, N, L, d_out);
  if (rc) return rc;
  if (s0_stride != 0 && s0_stride != 1) return fail(ctx, DHJ_ERR_ARG, "s0_stride must be 0 or 1");
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;   // NULL = the default stream
  SliceView v;
  rc = grid_view(ctx, strikes, nK, maturities, nT, scale_by_spot, is_call, N, r, q, L, st, &v);
  if (rc) return rc;
  if (P == 0) return DHJ_OK;
  PriceArgs a;
  a.params = d_params; a.S0 = d_S0; a.s0_stride = s0_stride; a.row_index = nullptr; a.P = P; a.transform = 0;
  a.out = d_out;
  rc = launch_price(ctx, v, a, nK, st);
  if (rc) return rc;
  return book_used(ctx, st);
}

// ---- calibration loss ------------------------------------------------------------------------
int dhj_market_create(dhj_ctx* ctx, int32_t n_markets, int32_t M, const double* S0, double r,
                      const double* strike, int64_t strike_stride, const double* maturity,
                      const int32_t* is_call, const double* price, int32_t N, dhj_market** out) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (!out) return fail(ctx, DHJ_ERR_ARG, "null market pointer");
  *out = nullptr;
  if (n_markets < 1 || M < 1) return fail(ctx, DHJ_ERR_ARG, "n_markets and M must be >= 1");
  if (!S0 || !strike || !maturity || !is_call || !price) return fail(ctx, DHJ_ERR_ARG, "null market array");
  if (N < 1) return fail(ctx, DHJ_ERR_ARG, "N must be >= 1");
  if (strike_stride != 0 && strike_stride != M) return fail(ctx, DHJ_ERR_ARG, "strike_stride must be 0 or M");
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  dhj_market* mk = new (std::nothrow) dhj_market();
  if (!mk) return fail(ctx, DHJ_ERR_NOMEM, "out of host memory");
  mk->ctx = ctx; mk->n_markets = n_markets; mk->M = M; mk->N = N; mk->r = r;
  mk->strike_stride = strike_stride;
  mk->book.group(maturity, is_call, M);
  const size_t bb = mk->book.packed_bytes();
  std::vector<unsigned char> image(bb);
  mk->book.pack(image.data());
  const size_t kbytes = (size_t)(strike_stride ? n_markets : 1) * M * sizeof(double);
  const size_t pbytes = (size_t)n_markets * M * sizeof(double);
  cudaError_t e = ctx->pool_take(&mk->d_book, bb);
  if (e == cudaSuccess) e = ctx->pool_take(&mk->d_strike, kbytes);
  if (e == cudaSuccess) e = ctx->pool_take(&mk->d_S0, (size_t)n_markets * sizeof(double));
  if (e == cudaSuccess) e = ctx->pool_take(&mk->d_price, pbytes);
  if (e == cudaSuccess) e = cudaMemcpy(mk->d_book.p, image.data(), bb, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(mk->d_strike.p, strike, kbytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(mk->d_S0.p, S0, (size_t)n_markets * sizeof(double), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(mk->d_price.p, price, pbytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    dhj_market_destroy(mk);
    return fail(ctx, e == cudaErrorMemoryAllocation ? DHJ_ERR_NOMEM : DHJ_ERR_CUDA, "market upload failed: %s",
                cudaGetErrorString(e));
  }
  mk->book.view(&mk->view, (const unsigned char*)mk->d_book.p);
  mk->view.strike = (const double*)mk->d_strike.p;
  mk->view.strike_stride = strike_stride;
  mk->view.scale_by_spot = 0; mk->view.n_cos = N; mk->view.r = r; mk->view.q = 0.0; mk->view.L = 10.0;
  *out = mk;
  return DHJ_OK;
}

int dhj_market_destroy(dhj_market* mk) {
  if (!mk) return DHJ_OK;
  if (mk->ctx) {
    cudaSetDevice(mk->ctx->device);
    // launches that read the market's tables are all on the context's stream: once it has drained the buffers can
    // serve the next market
    cudaStreamSynchronize(mk->ctx->stream);
    mk->ctx->pool_give(&mk->d_book); mk->ctx->pool_give(&mk->d_strike);
    mk->ctx->pool_give(&mk->d_S0); mk->ctx->pool_give(&mk->d_price);
    mk->ctx->pool_give(&mk->d_mvol); mk->ctx->pool_give(&mk->d_ivtab);
  } else {
    mk->d_book.release(); mk->d_strike.release(); mk->d_S0.release(); mk->d_price.release();
    mk->d_mvol.release(); mk->d_ivtab.release();
  }
  delete mk;
  return DHJ_OK;
}

static int launch_iv_residual(dhj_ctx* ctx, const dhj_market* mk, const double* prices, const int* row_index,
                              long long n_units, double* vol, double* inv_vega, int32_t* status);

static int run_loss(dhj_ctx* ctx, const dhj_market* mk, const double* x, const int32_t* market_index, int64_t B,
                    int fd, double h, double* out_f, double* out_g, double* out_f_all) {
  const int* d_index = nullptr;
  DHJ_CUDA(ctx, cudaSetDevice(ctx ? ctx->device : 0));
  int rc = stage_x(ctx, mk, x, market_index, B, &d_index);
  if (rc) return rc;
  if (!out_f || (fd && !out_g)) return fail(ctx, DHJ_ERR_ARG, "null output");
  if (B == 0) return DHJ_OK;
  const int64_t n_units = B * (fd ? kFdPoints : 1);
  if (n_units > 2000000000LL) return fail(ctx, DHJ_ERR_ARG, "batch too large for one launch");
  DHJ_CUDA(ctx, ctx->d_f.reserve((size_t)n_units * sizeof(double)));
  if (fd) DHJ_CUDA(ctx, ctx->d_fg.reserve((size_t)n_units * sizeof(double)));
  const SliceView& v = mk->view;
  // Large batches go through the pricing kernel (expand -> k_price_batch -> reduce): its batches of 32 items keep the
  // four warps balanced whatever the number of slices per loss evaluation, which pays for two extra small launches
  // from a few thousand evaluations on.  Both paths run the same arithmetic and produce the same bits
  // (DHJ_DEBUG_SPLIT_UNITS: developer knob for measuring the crossover).
  static const int64_t kSplitUnits = [] {
    const char* e = getenv("DHJ_DEBUG_SPLIT_UNITS");
    return e ? (int64_t)atoll(e) : (int64_t)8192;
  }();
  const bool iv_objective = mk->objective == DHJ_OBJECTIVE_IV;
  if (!iv_objective && mk->book.max_slice <= kBatchMaxStrikes && v.n_slices <= kPriceItems && n_units < kSplitUnits) {
    // fused path: one launch
    if (fd) {
      const size_t cb = (size_t)B * sizeof(unsigned int);
      if (ctx->d_counters.cap < cb || ctx->counters_zeroed < cb) {
        DHJ_CUDA(ctx, ctx->d_counters.reserve(cb));
        DHJ_CUDA(ctx, cudaMemsetAsync(ctx->d_counters.p, 0, ctx->d_counters.cap, ctx->stream));
        ctx->counters_zeroed = ctx->d_counters.cap;
      }
    }
    LossBatchArgs a;
    a.x = (const double*)ctx->d_x.p; a.market_index = d_index; a.S0 = (const double*)mk->d_S0.p;
    a.market = (const double*)mk->d_price.p; a.fd = fd; a.h = h; a.n_units = n_units;
    a.f_all = (double*)ctx->d_f.p; a.fg = fd ? (double*)ctx->d_fg.p : nullptr;
    a.counters = fd ? (unsigned int*)ctx->d_counters.p : nullptr;
    // whole units per block batch (pick_units_per_batch: waves x block time)
    a.units_per_batch = pick_units_per_batch(n_units, v.n_slices, kPriceItems,
                                             (long long)ctx->sm_count * ctx->loss_blocks_per_sm);
    const long long batches = (n_units + a.units_per_batch - 1) / a.units_per_batch;
    k_loss_batch<<<grid_1d(batches), kBatchThreads, 0, ctx->stream>>>(v, a);
    DHJ_LAUNCHED(ctx);
  } else {
    // general path: stencil points -> pricing kernel (batch or dense by slice size) -> reduction
    DHJ_CUDA(ctx, ctx->d_prices.reserve((size_t)n_units * mk->M * sizeof(double)));
    PriceArgs pa;
    rc = expand_x(ctx, mk, d_index, B, fd, h, &pa);
    if (rc) return rc;
    pa.out = (double*)ctx->d_prices.p;
    rc = launch_price(ctx, v, pa, mk->book.max_slice, ctx->stream);
    if (rc) return rc;
    if (iv_objective) {
      // IV objective (dhj_ivloss.cuh): always this path; model vols per (point, option), then the reduction
      DHJ_CUDA(ctx, ctx->d_ivres.reserve((size_t)n_units * mk->M * sizeof(double)));
      double* vol = (double*)ctx->d_ivres.p;
      rc = launch_iv_residual(ctx, mk, (const double*)ctx->d_prices.p, (const int*)ctx->d_idx.p, n_units, vol,
                              nullptr, nullptr);
      if (rc) return rc;
      k_loss_iv_reduce<<<(unsigned)((B + 127) / 128), 128, 0, ctx->stream>>>(
          vol, (const double*)ctx->d_xv.p, (const int*)ctx->d_idx.p, (const double*)mk->d_mvol.p, v.pos, mk->M, B,
          fd, h, (const double*)ctx->d_x.p, (double*)ctx->d_f.p, fd ? (double*)ctx->d_fg.p : nullptr);
    } else {
      k_loss_reduce<<<(unsigned)((B + 127) / 128), 128, 0, ctx->stream>>>(
          (const double*)ctx->d_prices.p, (const double*)ctx->d_xv.p, (const int*)ctx->d_idx.p,
          (const double*)mk->d_price.p, v.pos, mk->M, B, fd, h, (const double*)ctx->d_x.p, (double*)ctx->d_f.p,
          fd ? (double*)ctx->d_fg.p : nullptr);
    }
    DHJ_LAUNCHED(ctx);
  }
  if (fd) return download_fg(ctx, B, out_f, out_g, out_f_all);
  const size_t res_bytes = (size_t)B * sizeof(double);
  DHJ_CUDA(ctx, ctx->h_res.reserve(res_bytes));
  DHJ_CUDA(ctx, cudaMemcpyAsync(ctx->h_res.p, ctx->d_f.p, res_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  DHJ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  host_copy(out_f, ctx->h_res.p, res_bytes);
  return DHJ_OK;
}

int dhj_loss_batch(dhj_ctx* ctx, const dhj_market* market, const double* x, const int32_t* market_index,
                   int64_t B, double* out_loss) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  return run_loss(ctx, market, x, market_index, B, 0, 0.0, out_loss, nullptr, nullptr);
}

int dhj_loss_fd(dhj_ctx* ctx, const dhj_market* market, const double* x, const int32_t* market_index,
                int64_t C, double h, double* out_f, double* out_g, double* out_f_all) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (!(h > 0.0)) return fail(ctx, DHJ_ERR_ARG, "h must be > 0");
  return run_loss(ctx, market, x, market_index, C, 1, h, out_f, out_g, out_f_all);
}

// The whole lock-step loop of many simultaneous calibrations in one call: ask -> evaluate(x, market index, na, f, g)
// over every state that waits for an evaluation -> tell, until every optimiser has stopped.  (The Python host used
// to drive the three steps itself; with several pipelines per GPU their interpreter work serialised on the GIL — in
// here a pipeline never touches it.)
extern "C++" {
template <class Evaluate>
static int run_lockstep(dhj_lbfgs* opt, dhj_ctx* ctx, const dhj_market* market, const int32_t* state_market,
                        int64_t n_states, int64_t* rounds, int64_t* state_rounds, double* seconds, Evaluate evaluate) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (!opt || !market) return fail(ctx, DHJ_ERR_ARG, "null optimiser or market");
  int64_t n_opt = 0;
  int32_t dim = 0;
  dhj_lbfgs_shape(opt, &n_opt, &dim);
  // an ask writes up to every state of the optimiser into the buffers below, and state_market is read at its indices
  if (n_states != n_opt) return fail(ctx, DHJ_ERR_ARG, "n_states (%lld) != the optimiser's state count (%lld)",
                                     (long long)n_states, (long long)n_opt);
  if (dim != kNumParams) return fail(ctx, DHJ_ERR_ARG, "the optimiser's dimension is %d, not %d", dim, kNumParams);
  std::vector<int64_t> idx((size_t)n_states);
  std::vector<int32_t> mi((size_t)n_states);
  std::vector<double> x((size_t)n_states * kNumParams), f((size_t)n_states), g((size_t)n_states * kNumParams);
  int64_t n_rounds = 0, n_state_rounds = 0;
  double t_ask = 0.0, t_loss = 0.0, t_tell = 0.0;
  for (;;) {
    const double t0 = omp_get_wtime();
    int64_t na = 0;
    int rc = dhj_lbfgs_ask(opt, &na, idx.data(), x.data());
    if (rc) return fail(ctx, rc, "dhj_lbfgs_ask failed (%d)", rc);
    const double t1 = omp_get_wtime();
    t_ask += t1 - t0;
    if (na == 0) break;
    if (state_market)
      for (int64_t a = 0; a < na; ++a) mi[a] = state_market[idx[a]];
    rc = evaluate(x.data(), state_market ? mi.data() : nullptr, na, f.data(), g.data());
    if (rc) return rc;
    const double t2 = omp_get_wtime();
    rc = dhj_lbfgs_tell(opt, na, f.data(), g.data());
    if (rc) return fail(ctx, rc, "dhj_lbfgs_tell failed (%d)", rc);
    t_loss += t2 - t1;
    t_tell += omp_get_wtime() - t2;
    ++n_rounds;
    n_state_rounds += na;
  }
  if (rounds) *rounds = n_rounds;
  if (state_rounds) *state_rounds = n_state_rounds;
  if (seconds) { seconds[0] = t_ask; seconds[1] = t_loss; seconds[2] = t_tell; }
  return DHJ_OK;
}
}  // extern "C++"

int dhj_lbfgs_minimize_fd(dhj_lbfgs* opt, dhj_ctx* ctx, const dhj_market* market, const int32_t* state_market,
                          int64_t n_states, double h, int64_t* rounds, int64_t* state_rounds, double* seconds) {
  if (ctx && !(h > 0.0)) return fail(ctx, DHJ_ERR_ARG, "h must be > 0");
  return run_lockstep(opt, ctx, market, state_market, n_states, rounds, state_rounds, seconds,
                      [&](const double* x, const int32_t* mi, int64_t na, double* f, double* g) {
                        return run_loss(ctx, market, x, mi, na, 1, h, f, g, nullptr);
                      });
}

// ---- analytic parameter gradient (dhj_jac.cuh) -------------------------------------------------------
static int launch_jac(dhj_ctx* ctx, const SliceView& v, const JacArgs& a, cudaStream_t st) {
  const long long blocks = (a.P * (long long)v.n_slices + kJacWarps - 1) / kJacWarps;
  k_price_jac<<<grid_1d(blocks), 32 * kJacWarps, 0, st>>>(v, a);
  DHJ_LAUNCHED(ctx);
  return DHJ_OK;
}

// Prices and derivatives of an option list (dhj_price_jacobian, dhj_price_greeks) come in synchronous chunks through
// the staging buffers, rows = parameter sets: params | S0 | per-set strikes in, prices | derivatives out.  d[2] is
// null for a shared strike row (in the book).
int dhj_price_jacobian(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride, double r,
                       double q, const double* strike, int64_t strike_stride, const double* maturity,
                       const int32_t* is_call, int32_t M, int32_t N, double L, double* out_price, double* out_jac) {
  OptionList ol;
  int rc = option_list(ctx, params, P, S0, s0_stride, r, q, strike, strike_stride, maturity, is_call, M, N, L,
                       out_price, out_jac, &ol);
  if (rc || ol.empty) return rc;
  const size_t row = (size_t)M * sizeof(double);
  rc = stage_sync(ctx, P, kStageChunkBytes,
                  {rows_in(params, kNumParams * sizeof(double)), s0_in(S0, s0_stride), strike_in(strike, strike_stride),
                   rows_out(out_price, row), rows_out(out_jac, row * kNumParams)},
                  [&](int64_t n, void* const* d) {
                    SliceView v = ol.v;
                    if (d[2]) { v.strike = (const double*)d[2]; v.strike_stride = M; }
                    JacArgs a;
                    a.params = (const double*)d[0]; a.S0 = (const double*)d[1]; a.s0_stride = s0_stride ? 1 : 0;
                    a.row_index = nullptr; a.P = n; a.out_price = (double*)d[3]; a.out_jac = (double*)d[4];
                    return launch_jac(ctx, v, a, ctx->stream);
                  });
  return rc ? rc : book_used(ctx, ctx->stream);
}

// ---- Greeks (dhj_greeks.cuh) --------------------------------------------------------------------------
int dhj_price_greeks(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride, double r,
                     double q, const double* strike, int64_t strike_stride, const double* maturity,
                     const int32_t* is_call, int32_t M, int32_t N, double L, double* out_price, double* out_greeks) {
  OptionList ol;
  int rc = option_list(ctx, params, P, S0, s0_stride, r, q, strike, strike_stride, maturity, is_call, M, N, L,
                       out_price, out_greeks, &ol);
  if (rc || ol.empty) return rc;
  const size_t row = (size_t)M * sizeof(double);
  rc = stage_sync(ctx, P, kStageChunkBytes,
                  {rows_in(params, kNumParams * sizeof(double)), s0_in(S0, s0_stride), strike_in(strike, strike_stride),
                   rows_out(out_price, row), rows_out(out_greeks, row * kGreeks)},
                  [&](int64_t n, void* const* d) {
                    SliceView v = ol.v;
                    if (d[2]) { v.strike = (const double*)d[2]; v.strike_stride = M; }
                    GreeksArgs a;
                    a.params = (const double*)d[0]; a.S0 = (const double*)d[1]; a.s0_stride = s0_stride ? 1 : 0;
                    a.row_index = nullptr; a.P = n; a.out_price = (double*)d[3]; a.out_greeks = (double*)d[4];
                    const long long blocks = (n * (long long)v.n_slices + kJacWarps - 1) / kJacWarps;
                    k_price_greeks<<<grid_1d(blocks), 32 * kJacWarps, 0, ctx->stream>>>(v, a);
                    DHJ_LAUNCHED(ctx);
                    return DHJ_OK;
                  });
  return rc ? rc : book_used(ctx, ctx->stream);
}

// ---- implied volatility (dhj_iv.cuh) ----------------------------------------------------------------
namespace {

// The option tables of an implied-vol call as one image in the book ring: maturity[M] | strike[M] (shared strikes
// only) | is_call[M].  Fills the table pointers of *a.
int upload_iv_tables(dhj_ctx* ctx, const double* strike, bool shared_strike, const double* maturity,
                     const int32_t* is_call, int32_t M, cudaStream_t st, iv::IvArgs* a) {
  const size_t db = (size_t)M * sizeof(double);
  const size_t kb = shared_strike ? db : 0;
  std::vector<unsigned char> image(db + kb + (size_t)M * sizeof(int32_t));
  memcpy(image.data(), maturity, db);
  if (kb) memcpy(image.data() + db, strike, kb);
  memcpy(image.data() + db + kb, is_call, (size_t)M * sizeof(int32_t));
  const unsigned char* d;
  int rc = upload_image(ctx, image, st, &d);
  if (rc) return rc;
  a->maturity = (const double*)d;
  if (kb) { a->strike = (const double*)(d + db); a->strike_stride = 0; }
  a->is_call = (const int32_t*)(d + db + kb);
  return DHJ_OK;
}

// one elementwise launch over a.P x a.M options (grid-stride)
int launch_iv(dhj_ctx* ctx, const iv::IvArgs& a, bool inverse, cudaStream_t st) {
  const int blocks = grid_stride_blocks(ctx, a.P * (long long)a.M);
  if (inverse) iv::k_implied_vol<<<blocks, 256, 0, st>>>(a);
  else iv::k_bs_price<<<blocks, 256, 0, st>>>(a);
  DHJ_LAUNCHED(ctx);
  return DHJ_OK;
}

int check_iv(dhj_ctx* ctx, const void* in, int64_t P, const void* S0, int64_t s0_stride, const void* out, int32_t M) {
  int rc = check_arrays(ctx, in, P, S0, out);
  if (rc) return rc;
  if (M < 0) return fail(ctx, DHJ_ERR_ARG, "M must be >= 0");
  if (s0_stride != 0 && s0_stride != 1) return fail(ctx, DHJ_ERR_ARG, "s0_stride must be 0 or 1");
  return DHJ_OK;
}

// dhj_implied_vol (inverse) and dhj_bs_price: host arrays in synchronous chunks through the staging buffers, rows =
// sets: values | S0 | per-set strikes in, results | status out.  The status row counts towards the chunk size
// whether or not it is asked for (dhj_bs_price has none).
int run_iv_list(dhj_ctx* ctx, bool inverse, const double* in, int64_t P, const double* S0, int64_t s0_stride, double r,
                double q, const double* strike, int64_t strike_stride, const double* maturity, const int32_t* is_call,
                int32_t M, double* out, int32_t* status) {
  int rc = check_iv(ctx, in, P, S0, s0_stride, out, M);
  if (rc) return rc;
  bool empty;
  rc = check_list(ctx, P, s0_stride, strike, strike_stride, maturity, is_call, M, &empty);
  if (rc || empty) return rc;
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  iv::IvArgs a{};
  rc = upload_iv_tables(ctx, strike, strike_stride == 0, maturity, is_call, M, ctx->stream, &a);
  if (rc) return rc;
  a.r = r; a.q = q; a.M = M; a.scale_by_spot = 0; a.s0_stride = s0_stride;
  const size_t row = (size_t)M * sizeof(double);
  rc = stage_sync(ctx, P, kStageChunkBytes,
                  {rows_in(in, row), s0_in(S0, s0_stride), strike_in(strike, strike_stride), rows_out(out, row),
                   rows_out(inverse ? status : nullptr, (size_t)M * sizeof(int32_t))},
                  [&](int64_t n, void* const* d) {
                    a.in = (const double*)d[0]; a.S0 = (const double*)d[1]; a.P = n;
                    if (d[2]) { a.strike = (const double*)d[2]; a.strike_stride = M; }
                    a.out = (double*)d[3]; a.status = (int32_t*)d[4];
                    return launch_iv(ctx, a, inverse, ctx->stream);
                  });
  return rc ? rc : book_used(ctx, ctx->stream);
}

}  // namespace

int dhj_implied_vol(dhj_ctx* ctx, const double* price, int64_t P, const double* S0, int64_t s0_stride, double r,
                    double q, const double* strike, int64_t strike_stride, const double* maturity,
                    const int32_t* is_call, int32_t M, double* out_vol, int32_t* out_status) {
  return run_iv_list(ctx, true, price, P, S0, s0_stride, r, q, strike, strike_stride, maturity, is_call, M, out_vol,
                     out_status);
}

int dhj_bs_price(dhj_ctx* ctx, const double* vol, int64_t P, const double* S0, int64_t s0_stride, double r, double q,
                 const double* strike, int64_t strike_stride, const double* maturity, const int32_t* is_call,
                 int32_t M, double* out_price) {
  return run_iv_list(ctx, false, vol, P, S0, s0_stride, r, q, strike, strike_stride, maturity, is_call, M, out_price,
                     nullptr);
}

int dhj_implied_vol_dev(dhj_ctx* ctx, const double* d_price, int64_t P, const double* d_S0, int64_t s0_stride,
                        double r, double q, const double* strike, int32_t scale_by_spot, const double* maturity,
                        const int32_t* is_call, int32_t M, double* d_out_vol, int32_t* d_out_status, void* stream) {
  int rc = check_iv(ctx, d_price, P, d_S0, s0_stride, d_out_vol, M);
  if (rc) return rc;
  bool empty;
  rc = check_list(ctx, P, s0_stride, strike, 0, maturity, is_call, M, &empty);
  if (rc || empty) return rc;
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;   // NULL = the default stream
  iv::IvArgs a{};
  rc = upload_iv_tables(ctx, strike, true, maturity, is_call, M, st, &a);
  if (rc) return rc;
  a.in = d_price; a.S0 = d_S0; a.s0_stride = s0_stride; a.scale_by_spot = scale_by_spot ? 1 : 0;
  a.r = r; a.q = q; a.P = P; a.M = M; a.out = d_out_vol; a.status = d_out_status;
  rc = launch_iv(ctx, a, true, st);
  if (rc) return rc;
  return book_used(ctx, st);
}

// f and the analytic g of B loss evaluations: exp/tanh transform (k_fd_expand without a stencil) -> prices of every
// market option by the pricing kernel (the split loss path's launch: f below has the bits of dhj_loss_batch) and their
// Jacobian (k_price_jac) -> one thread per state (k_loss_grad_reduce).  States are cut into launches of bounded scratch;
// each state's (f, g) is computed by one thread in a fixed order, so it does not depend on the cut or on the other
// states of the call.
static int run_loss_grad(dhj_ctx* ctx, const dhj_market* mk, const double* x, const int32_t* market_index, int64_t B,
                         double* out_f, double* out_g) {
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  const int* d_index = nullptr;
  int rc = stage_x(ctx, mk, x, market_index, B, &d_index);
  if (rc) return rc;
  if (!out_f || !out_g) return fail(ctx, DHJ_ERR_ARG, "null output");
  if (B == 0) return DHJ_OK;
  const int M = mk->M;
  const bool iv_objective = mk->objective == DHJ_OBJECTIVE_IV;
  const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(B, (int64_t)(((size_t)1 << 27) / ((size_t)M * kJacChannels))));
  DHJ_CUDA(ctx, ctx->d_fg.reserve((size_t)B * kFdPoints * sizeof(double)));
  DHJ_CUDA(ctx, ctx->d_prices.reserve((size_t)2 * chunk * M * sizeof(double)));   // pricing kernel | k_price_jac
  DHJ_CUDA(ctx, ctx->d_jac.reserve((size_t)chunk * M * kNumParams * sizeof(double)));
  if (iv_objective) DHJ_CUDA(ctx, ctx->d_ivres.reserve((size_t)2 * chunk * M * sizeof(double)));   // vol | 1/vega
  PriceArgs all;
  rc = expand_x(ctx, mk, d_index, B, 0, 0.0, &all);
  if (rc) return rc;
  double* fg = (double*)ctx->d_fg.p;
  for (int64_t lo = 0; lo < B; lo += chunk) {
    const int64_t n = std::min(chunk, B - lo);
    double* prices = (double*)ctx->d_prices.p;
    PriceArgs pa = all;
    pa.params += lo * kNumParams; pa.row_index += lo; pa.P = n; pa.out = prices;
    rc = launch_price(ctx, mk->view, pa, mk->book.max_slice, ctx->stream);
    if (rc) return rc;
    JacArgs a;
    a.params = pa.params; a.S0 = pa.S0; a.s0_stride = 1; a.row_index = pa.row_index;
    a.P = n; a.out_price = prices + n * (int64_t)M; a.out_jac = (double*)ctx->d_jac.p;
    rc = launch_jac(ctx, mk->view, a, ctx->stream);
    if (rc) return rc;
    if (iv_objective) {
      double* vol = (double*)ctx->d_ivres.p;
      double* inv_vega = vol + n * (int64_t)M;
      rc = launch_iv_residual(ctx, mk, prices, a.row_index, n, vol, inv_vega, nullptr);
      if (rc) return rc;
      k_loss_iv_grad_reduce<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(
          vol, inv_vega, a.out_jac, a.params, a.row_index, (const double*)mk->d_mvol.p, mk->view.pos, M, n,
          fg + lo * kFdPoints);
    } else {
      k_loss_grad_reduce<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(
          prices, a.out_jac, a.params, a.row_index, (const double*)mk->d_price.p, mk->view.pos, M, n,
          fg + lo * kFdPoints);
    }
    DHJ_LAUNCHED(ctx);
  }
  return download_fg(ctx, B, out_f, out_g, nullptr);
}

int dhj_loss_grad(dhj_ctx* ctx, const dhj_market* market, const double* x, const int32_t* market_index, int64_t C,
                  double* out_f, double* out_g) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  return run_loss_grad(ctx, market, x, market_index, C, out_f, out_g);
}

int dhj_lbfgs_minimize_grad(dhj_lbfgs* opt, dhj_ctx* ctx, const dhj_market* market, const int32_t* state_market,
                            int64_t n_states, int64_t* rounds, int64_t* state_rounds, double* seconds) {
  return run_lockstep(opt, ctx, market, state_market, n_states, rounds, state_rounds, seconds,
                      [&](const double* x, const int32_t* mi, int64_t na, double* f, double* g) {
                        return run_loss_grad(ctx, market, x, mi, na, f, g);
                      });
}

int dhj_market_prices(dhj_ctx* ctx, const dhj_market* mk, const double* x, const int32_t* market_index,
                      int64_t B, double* out_prices) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  const int* d_index = nullptr;
  int rc = stage_x(ctx, mk, x, market_index, B, &d_index);
  if (rc) return rc;
  if (!out_prices) return fail(ctx, DHJ_ERR_ARG, "null output");
  if (B == 0) return DHJ_OK;
  const size_t ob = (size_t)B * mk->M * sizeof(double);
  DHJ_CUDA(ctx, ctx->d_prices.reserve(ob));
  DHJ_CUDA(ctx, ctx->h_res.reserve(ob));
  // without an index every x uses market 0: a zero table does that
  if (!d_index) {
    DHJ_CUDA(ctx, ctx->d_idx.reserve((size_t)B * sizeof(int)));
    DHJ_CUDA(ctx, cudaMemsetAsync(ctx->d_idx.p, 0, (size_t)B * sizeof(int), ctx->stream));
    d_index = (const int*)ctx->d_idx.p;
  }
  PriceArgs a;
  a.params = (const double*)ctx->d_x.p; a.S0 = (const double*)mk->d_S0.p; a.s0_stride = 1;
  a.row_index = d_index; a.P = B; a.transform = 1; a.out = (double*)ctx->d_prices.p;
  rc = launch_price(ctx, mk->view, a, mk->book.max_slice, ctx->stream);
  if (rc) return rc;
  DHJ_CUDA(ctx, cudaMemcpyAsync(ctx->h_res.p, ctx->d_prices.p, ob, cudaMemcpyDeviceToHost, ctx->stream));
  DHJ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  memcpy(out_prices, ctx->h_res.p, ob);
  return DHJ_OK;
}

// ---- implied-volatility objective (dhj_ivloss.cuh) ---------------------------------------------------
// maturity[M] | is_call[M] of the market in the caller's option order, rebuilt from the slice book
static int ensure_iv_tables(dhj_ctx* ctx, dhj_market* mk) {
  if (mk->d_ivtab.p) return DHJ_OK;
  const int M = mk->M;
  const BookHost& b = mk->book;
  std::vector<unsigned char> image((size_t)M * (sizeof(double) + sizeof(int32_t)));
  double* T = (double*)image.data();
  int32_t* call = (int32_t*)(image.data() + (size_t)M * sizeof(double));
  for (int s = 0; s < b.n_slices; ++s)
    for (int d = b.slice_off[s]; d < b.slice_off[s + 1]; ++d) {
      T[b.pos[d]] = b.slice_T[s];
      call[b.pos[d]] = b.call[d];
    }
  DHJ_CUDA(ctx, ctx->pool_take(&mk->d_ivtab, image.size()));
  DHJ_CUDA(ctx, cudaMemcpyAsync(mk->d_ivtab.p, image.data(), image.size(), cudaMemcpyHostToDevice, ctx->stream));
  DHJ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return DHJ_OK;
}

// k_iv_residual over n_units x M (grid-stride, as launch_iv); status non-null: reporting mode
static int launch_iv_residual(dhj_ctx* ctx, const dhj_market* mk, const double* prices, const int* row_index,
                              long long n_units, double* vol, double* inv_vega, int32_t* status) {
  IvResidualArgs a;
  a.prices = prices; a.row_index = row_index; a.S0 = (const double*)mk->d_S0.p;
  a.strike = (const double*)mk->d_strike.p; a.strike_stride = mk->strike_stride;
  a.maturity = (const double*)mk->d_ivtab.p;
  a.is_call = (const int32_t*)((const unsigned char*)mk->d_ivtab.p + (size_t)mk->M * sizeof(double));
  a.mvol = (const double*)mk->d_mvol.p; a.r = mk->r; a.n_units = n_units; a.M = mk->M; a.n_markets = mk->n_markets;
  a.vol = vol; a.inv_vega = inv_vega; a.status = status;
  k_iv_residual<<<grid_stride_blocks(ctx, n_units * (long long)mk->M), 256, 0, ctx->stream>>>(a);
  DHJ_LAUNCHED(ctx);
  return DHJ_OK;
}

int dhj_market_set_objective(dhj_ctx* ctx, dhj_market* mk, int32_t objective, double* out_market_vol,
                             int32_t* out_status) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (!mk) return fail(ctx, DHJ_ERR_ARG, "null market");
  if (mk->ctx != ctx) return fail(ctx, DHJ_ERR_ARG, "market belongs to another context");
  if (objective != DHJ_OBJECTIVE_PRICE && objective != DHJ_OBJECTIVE_IV)
    return fail(ctx, DHJ_ERR_ARG, "unknown objective %d", objective);
  if (objective == DHJ_OBJECTIVE_PRICE) { mk->objective = objective; return DHJ_OK; }
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  int rc = ensure_iv_tables(ctx, mk);
  if (rc) return rc;
  const int M = mk->M;
  const size_t n_opt = (size_t)mk->n_markets * M;
  // the quotes are inverted into scratch: the market's vols and objective change only when the call succeeds
  DHJ_CUDA(ctx, ctx->d_ivres.reserve(n_opt * (sizeof(double) + sizeof(int32_t))));
  // the market's quotes through dhj_implied_vol's solver (q = 0, as the market assumes)
  iv::IvArgs a{};
  a.in = (const double*)mk->d_price.p; a.S0 = (const double*)mk->d_S0.p; a.s0_stride = 1;
  a.strike = (const double*)mk->d_strike.p; a.strike_stride = mk->strike_stride; a.scale_by_spot = 0;
  a.maturity = (const double*)mk->d_ivtab.p;
  a.is_call = (const int32_t*)((const unsigned char*)mk->d_ivtab.p + (size_t)M * sizeof(double));
  a.r = mk->r; a.q = 0.0; a.P = mk->n_markets; a.M = M;
  a.out = (double*)ctx->d_ivres.p; a.status = (int32_t*)((double*)ctx->d_ivres.p + n_opt);
  rc = launch_iv(ctx, a, true, ctx->stream);
  if (rc) return rc;
  std::vector<double> vol(n_opt);
  std::vector<int32_t> st(n_opt);
  DHJ_CUDA(ctx, cudaMemcpyAsync(vol.data(), a.out, n_opt * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DHJ_CUDA(ctx, cudaMemcpyAsync(st.data(), a.status, n_opt * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DHJ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  // a quote without an implied vol (status != 0; "not converged" returns its last iterate) is left out: NaN
  int empty = -1;
  for (int m = 0; m < mk->n_markets; ++m) {
    int valid = 0;
    for (int o = 0; o < M; ++o) {
      const size_t i = (size_t)m * M + o;
      if (st[i] != iv::kOk) vol[i] = NAN;
      else ++valid;
    }
    if (!valid && empty < 0) empty = m;
  }
  if (out_market_vol) memcpy(out_market_vol, vol.data(), n_opt * sizeof(double));
  if (out_status) memcpy(out_status, st.data(), n_opt * sizeof(int32_t));
  if (empty >= 0)
    return fail(ctx, DHJ_ERR_ARG, "market %d has no option with an implied vol (every quote's status is != 0)", empty);
  if (!mk->d_mvol.p) DHJ_CUDA(ctx, ctx->pool_take(&mk->d_mvol, n_opt * sizeof(double)));
  DHJ_CUDA(ctx, cudaMemcpyAsync(mk->d_mvol.p, vol.data(), n_opt * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  DHJ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  mk->objective = DHJ_OBJECTIVE_IV;
  return DHJ_OK;
}

int dhj_market_implied_vols(dhj_ctx* ctx, const dhj_market* market, const double* x, const int32_t* market_index,
                            int64_t B, double* out_vol, int32_t* out_status) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  const int* d_index = nullptr;
  int rc = stage_x(ctx, market, x, market_index, B, &d_index);
  if (rc) return rc;
  if (!out_vol) return fail(ctx, DHJ_ERR_ARG, "null output");
  if (B == 0) return DHJ_OK;
  dhj_market* mk = const_cast<dhj_market*>(market);   // the option tables are a cache of the market's own book
  rc = ensure_iv_tables(ctx, mk);
  if (rc) return rc;
  const int M = mk->M;
  const size_t nb = (size_t)B * M;
  DHJ_CUDA(ctx, ctx->d_prices.reserve(nb * sizeof(double)));
  DHJ_CUDA(ctx, ctx->d_ivres.reserve(nb * (sizeof(double) + sizeof(int32_t))));
  DHJ_CUDA(ctx, ctx->h_res.reserve(nb * (sizeof(double) + sizeof(int32_t))));
  PriceArgs pa;
  rc = expand_x(ctx, mk, d_index, B, 0, 0.0, &pa);
  if (rc) return rc;
  pa.out = (double*)ctx->d_prices.p;
  rc = launch_price(ctx, mk->view, pa, mk->book.max_slice, ctx->stream);
  if (rc) return rc;
  double* vol = (double*)ctx->d_ivres.p;
  int32_t* st = (int32_t*)(vol + nb);
  rc = launch_iv_residual(ctx, mk, pa.out, pa.row_index, B, vol, nullptr, st);
  if (rc) return rc;
  DHJ_CUDA(ctx, cudaMemcpyAsync(ctx->h_res.p, vol, nb * (sizeof(double) + sizeof(int32_t)), cudaMemcpyDeviceToHost,
                                ctx->stream));
  DHJ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  host_copy(out_vol, ctx->h_res.p, nb * sizeof(double));
  if (out_status) host_copy(out_status, (const double*)ctx->h_res.p + nb, nb * sizeof(int32_t));
  return DHJ_OK;
}

// ---- the remaining public methods of DoubleHeston --------------------------------------------
// one synchronous staged launch each (stage_sync, one chunk)
int dhj_cf(dhj_ctx* ctx, const double* params, double r, double q, double tau, const double* u, int32_t n,
           double* out_re, double* out_im) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (!params || !u || !out_re || !out_im || n < 0) return fail(ctx, DHJ_ERR_ARG, "bad arguments");
  if (n == 0) return DHJ_OK;
  return stage_sync(ctx, n, kOneChunk,
                    {table_in(params, kNumParams * sizeof(double)), rows_in(u, sizeof(double)),
                     rows_out(out_re, sizeof(double)), rows_out(out_im, sizeof(double))},
                    [&](int64_t, void* const* d) {
                      k_cf<<<(n + 127) / 128, 128, 0, ctx->stream>>>((const double*)d[0], r, q, tau,
                                                                      (const double*)d[1], n, (double*)d[2],
                                                                      (double*)d[3]);
                      DHJ_LAUNCHED(ctx);
                      return DHJ_OK;
                    });
}

int dhj_cf_complex(dhj_ctx* ctx, const double* params, double r, double q, double tau, const double* u_re,
                   const double* u_im, int32_t n, double* out_re, double* out_im) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (!params || !u_re || !u_im || !out_re || !out_im || n < 0) return fail(ctx, DHJ_ERR_ARG, "bad arguments");
  if (n == 0) return DHJ_OK;
  return stage_sync(ctx, n, kOneChunk,
                    {table_in(params, kNumParams * sizeof(double)), rows_in(u_re, sizeof(double)),
                     rows_in(u_im, sizeof(double)), rows_out(out_re, sizeof(double)),
                     rows_out(out_im, sizeof(double))},
                    [&](int64_t, void* const* d) {
                      k_cf_complex<<<(n + 127) / 128, 128, 0, ctx->stream>>>(
                          (const double*)d[0], r, q, tau, (const double*)d[1], (const double*)d[2], n, (double*)d[3],
                          (double*)d[4]);
                      DHJ_LAUNCHED(ctx);
                      return DHJ_OK;
                    });
}

int dhj_truncation_range(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride,
                         double r, const double* strike, const double* maturity, int32_t M, double L,
                         double* out_ab) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (!params || !S0 || !strike || !maturity || !out_ab || P < 0 || M < 0) return fail(ctx, DHJ_ERR_ARG, "bad arguments");
  if (s0_stride != 0 && s0_stride != 1) return fail(ctx, DHJ_ERR_ARG, "s0_stride must be 0 or 1");
  if (P == 0 || M == 0) return DHJ_OK;
  if (P * (int64_t)M > (int64_t)1 << 28) return fail(ctx, DHJ_ERR_ARG, "P*M too large for this helper");
  const size_t mb = (size_t)M * sizeof(double);
  return stage_sync(ctx, P, kOneChunk,
                    {rows_in(params, kNumParams * sizeof(double)), s0_in(S0, s0_stride), table_in(strike, mb),
                     table_in(maturity, mb), rows_out(out_ab, 2 * mb)},
                    [&](int64_t, void* const* d) {
                      const long long n = P * (long long)M;
                      k_truncation_range<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(
                          (const double*)d[0], P, (const double*)d[1], s0_stride, (const double*)d[2],
                          (const double*)d[3], M, r, L, (double*)d[4]);
                      DHJ_LAUNCHED(ctx);
                      return DHJ_OK;
                    });
}

int dhj_chi_psi(dhj_ctx* ctx, const int32_t* k, int32_t n, double c, double d, double a, double b,
                double* out_chi, double* out_psi) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (!k || !out_chi || !out_psi || n < 0) return fail(ctx, DHJ_ERR_ARG, "bad arguments");
  if (n == 0) return DHJ_OK;
  return stage_sync(ctx, n, kOneChunk,
                    {rows_in(k, sizeof(int32_t)), rows_out(out_chi, sizeof(double)), rows_out(out_psi, sizeof(double))},
                    [&](int64_t, void* const* dev) {
                      k_chi_psi<<<(n + 127) / 128, 128, 0, ctx->stream>>>((const int*)dev[0], n, c, d, a, b,
                                                                           (double*)dev[1], (double*)dev[2]);
                      DHJ_LAUNCHED(ctx);
                      return DHJ_OK;
                    });
}

}  // extern "C"

// ---- synthetic dataset sweep (counter stream; dhj_generate.cuh) ------------------------------------
namespace {

struct GenConfig {
  GenArgs g;
  int nK, nT, N;
  double r, L;
  const double* strikes_rel;
  const double* maturities;
};

int check_generate(dhj_ctx* ctx, int64_t first, int64_t n, int32_t path_len, const double* lo, const double* hi,
                   const double* strikes_rel, int32_t nK, const double* maturities, int32_t nT, int32_t N) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (first < 0 || n < 0) return fail(ctx, DHJ_ERR_ARG, "first and n must be >= 0");
  if (path_len < 1) return fail(ctx, DHJ_ERR_ARG, "path_len must be >= 1 (got %d)", path_len);
  if (!lo || !hi || !strikes_rel || !maturities) return fail(ctx, DHJ_ERR_ARG, "null table");
  if (nK < 1 || nT < 1 || (int64_t)nK * nT > kGenMaxOptions)
    return fail(ctx, DHJ_ERR_ARG, "the generator grid must have 1..%d options (got %d x %d)", kGenMaxOptions, nT, nK);
  if (N < 1) return fail(ctx, DHJ_ERR_ARG, "N must be >= 1 (got %d)", N);
  return DHJ_OK;
}

// enqueue draws -> prices -> market/loss for samples [first, first + n) on `st`; all pointers are device memory
int enqueue_generate(dhj_ctx* ctx, const GenConfig& c, int64_t first, int64_t n, double* d_params, double* d_spots,
                     double* d_model, double* d_market, double* d_loss, cudaStream_t st) {
  if (n == 0) return DHJ_OK;
  GenArgs g = c.g;
  g.first = first; g.n = n;
  const long long q_first = first / g.path_len, q_last = (first + n - 1) / g.path_len;
  const long long paths = q_last - q_first + 1;
  k_gen_draws<<<(unsigned)((paths + kGenWarps - 1) / kGenWarps), 32 * kGenWarps, 0, st>>>(g, d_params, d_spots);
  DHJ_LAUNCHED(ctx);
  SliceView v;
  int rc = grid_view(ctx, c.strikes_rel, c.nK, c.maturities, c.nT, /*scale_by_spot=*/1, /*is_call=*/1, c.N, c.r, 0.0,
                     c.L, st, &v);
  if (rc) return rc;
  PriceArgs a;
  a.params = d_params; a.S0 = d_spots; a.s0_stride = 1; a.row_index = nullptr; a.P = n; a.transform = 0;
  a.out = d_model;
  rc = launch_price(ctx, v, a, c.nK, st);
  if (rc) return rc;
  rc = book_used(ctx, st);
  if (rc) return rc;
  if (d_market && d_loss) {
    const int M = c.nK * c.nT;
    const size_t smem = (size_t)kGenMarketSamples * (M | 1) * sizeof(double);
    k_gen_market<<<(unsigned)((n + kGenMarketSamples - 1) / kGenMarketSamples), kGenMarketSamples, smem, st>>>(
        g.seed, first, n, M, g.noise_sd, d_model, d_market, d_loss);
    DHJ_LAUNCHED(ctx);
  }
  return DHJ_OK;
}

void fill_gen_config(GenConfig* c, uint64_t seed, int32_t path_len, const double* lo, const double* hi,
                     double persistence, double spot0, double ret_mean, double ret_sd, double noise_sd,
                     const double* strikes_rel, int32_t nK, const double* maturities, int32_t nT, double r, int32_t N,
                     double L) {
  c->g.seed = seed; c->g.first = 0; c->g.n = 0; c->g.path_len = path_len;
  for (int j = 0; j < kNumParams; ++j) { c->g.lo[j] = lo[j]; c->g.range[j] = hi[j] - lo[j]; }
  c->g.persistence = persistence; c->g.spot0 = spot0; c->g.ret_mean = ret_mean; c->g.ret_sd = ret_sd;
  c->g.noise_sd = noise_sd;
  c->nK = nK; c->nT = nT; c->N = N; c->r = r; c->L = L; c->strikes_rel = strikes_rel; c->maturities = maturities;
}

}  // namespace

extern "C" {

int dhj_generate_dev(dhj_ctx* ctx, uint64_t seed, int64_t first, int64_t n, int32_t path_len, const double* lo,
                     const double* hi, double persistence, double spot0, double ret_mean, double ret_sd,
                     double noise_sd, const double* strikes_rel, int32_t nK, const double* maturities, int32_t nT,
                     double r, int32_t N, double L, double* d_params, double* d_spots, double* d_model,
                     double* d_market, double* d_loss, void* stream) {
  int rc = check_generate(ctx, first, n, path_len, lo, hi, strikes_rel, nK, maturities, nT, N);
  if (rc) return rc;
  if (!d_params || !d_spots || !d_model) return fail(ctx, DHJ_ERR_ARG, "null output (params, spots, model are required)");
  if ((d_market == nullptr) != (d_loss == nullptr))
    return fail(ctx, DHJ_ERR_ARG, "market and loss outputs come together (both or neither)");
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  GenConfig c;
  fill_gen_config(&c, seed, path_len, lo, hi, persistence, spot0, ret_mean, ret_sd, noise_sd, strikes_rel, nK,
                  maturities, nT, r, N, L);
  return enqueue_generate(ctx, c, first, n, d_params, d_spots, d_model, d_market, d_loss, (cudaStream_t)stream);
}

int dhj_generate(dhj_ctx* ctx, uint64_t seed, int64_t first, int64_t n, int32_t path_len, const double* lo,
                 const double* hi, double persistence, double spot0, double ret_mean, double ret_sd, double noise_sd,
                 const double* strikes_rel, int32_t nK, const double* maturities, int32_t nT, double r, int32_t N,
                 double L, double* params, double* spots, double* model, double* market, double* loss) {
  int rc = check_generate(ctx, first, n, path_len, lo, hi, strikes_rel, nK, maturities, nT, N);
  if (rc) return rc;
  if (!params || !spots || !model || !market || !loss) return fail(ctx, DHJ_ERR_ARG, "null output array");
  if (n == 0) return DHJ_OK;
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  GenConfig c;
  fill_gen_config(&c, seed, path_len, lo, hi, persistence, spot0, ret_mean, ret_sd, noise_sd, strikes_rel, nK,
                  maturities, nT, r, N, L);
  const int M = nK * nT;
  const bool pinned = is_pinned_host(params) && is_pinned_host(spots) && is_pinned_host(model) &&
                      is_pinned_host(market) && is_pinned_host(loss);
  // chunks of whole paths where possible (a chunk that starts inside a path re-draws the path's head)
  int64_t chunk = 131072;
  if (path_len < chunk) chunk -= chunk % path_len;
  for (int i = 0; i < kSlots; ++i) {
    Slot& sl = ctx->slots[i];
    DHJ_CUDA(ctx, cudaEventSynchronize(sl.done));
    sl.pending = false; sl.user_out = nullptr; sl.out_bytes = 0; sl.pieces.clear();
  }
  int slot_i = 0;
  for (int64_t lo_i = 0; lo_i < n; lo_i += chunk, slot_i = (slot_i + 1) % kSlots) {
    const int64_t cnt = std::min(chunk, n - lo_i);
    Slot& sl = ctx->slots[slot_i];
    DHJ_CUDA(ctx, cudaEventSynchronize(sl.done));
    sl.drain_pieces(host_copy);
    // device layout of a chunk: params | spots | model | market | loss
    const size_t pb = (size_t)cnt * kNumParams * sizeof(double), sb = (size_t)cnt * sizeof(double);
    const size_t mb = (size_t)cnt * M * sizeof(double);
    const size_t total = pb + sb + 2 * mb + sb;
    DHJ_CUDA(ctx, sl.d_out.reserve(total));
    unsigned char* d = (unsigned char*)sl.d_out.p;
    double* d_params = (double*)d; double* d_spots = (double*)(d + pb); double* d_model = (double*)(d + pb + sb);
    double* d_market = (double*)(d + pb + sb + mb); double* d_loss = (double*)(d + pb + sb + 2 * mb);
    rc = enqueue_generate(ctx, c, first + lo_i, cnt, d_params, d_spots, d_model, d_market, d_loss, sl.stream);
    if (rc) return rc;
    void* dst[5] = {params + lo_i * kNumParams, spots + lo_i, model + lo_i * M, market + lo_i * M, loss + lo_i};
    const size_t off[5] = {0, pb, pb + sb, pb + sb + mb, pb + sb + 2 * mb};
    const size_t len[5] = {pb, sb, mb, mb, sb};
    if (pinned) {
      for (int k = 0; k < 5; ++k)
        DHJ_CUDA(ctx, cudaMemcpyAsync(dst[k], d + off[k], len[k], cudaMemcpyDeviceToHost, sl.stream));
    } else {
      DHJ_CUDA(ctx, sl.h_out.reserve(total));
      DHJ_CUDA(ctx, cudaMemcpyAsync(sl.h_out.p, d, total, cudaMemcpyDeviceToHost, sl.stream));
      for (int k = 0; k < 5; ++k) sl.pieces.push_back({dst[k], off[k], len[k]});
    }
    DHJ_CUDA(ctx, cudaEventRecord(sl.done, sl.stream));
  }
  for (int i = 0; i < kSlots; ++i) {
    Slot& sl = ctx->slots[i];
    DHJ_CUDA(ctx, cudaEventSynchronize(sl.done));
    sl.drain_pieces(host_copy);
  }
  return DHJ_OK;
}

}  // extern "C"

// ---- Monte Carlo pricing of path-dependent options (dhj_mc.cuh) ------------------------------------
namespace {

int check_mc(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride, double T,
             int32_t n_steps, int32_t n_obs, int32_t M, const int32_t* kind, const int32_t* is_call,
             const double* strike, const double* barrier, int64_t n_paths, const double* out_price) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (!params || !S0 || !kind || !is_call || !strike || !out_price) return fail(ctx, DHJ_ERR_ARG, "null array");
  if (P < 1 || M < 1 || n_paths < 1)
    return fail(ctx, DHJ_ERR_ARG, "P, M and n_paths must be >= 1 (got %lld, %d, %lld)", (long long)P, M,
                (long long)n_paths);
  if (M > mc::kMcMaxOptions) return fail(ctx, DHJ_ERR_ARG, "M must be <= %d (got %d)", mc::kMcMaxOptions, M);
  if (s0_stride != 0 && s0_stride != 1) return fail(ctx, DHJ_ERR_ARG, "s0_stride must be 0 or 1");
  if (n_steps < 1 || n_obs < 1 || n_steps > mc::kMcMaxSteps || n_steps % n_obs != 0)
    return fail(ctx, DHJ_ERR_ARG, "need 1 <= n_obs, n_obs | n_steps, n_steps <= %d (got n_steps %d, n_obs %d)",
                mc::kMcMaxSteps, n_steps, n_obs);
  if (!(std::isfinite(T) && T > 0.0)) return fail(ctx, DHJ_ERR_ARG, "T must be finite and > 0 (got %g)", T);
  for (int m = 0; m < M; ++m) {
    if (kind[m] < 0 || kind[m] >= mc::kMcKinds) return fail(ctx, DHJ_ERR_ARG, "option %d: unknown kind %d", m, kind[m]);
    if (!(std::isfinite(strike[m]) && strike[m] >= 0.0))
      return fail(ctx, DHJ_ERR_ARG, "option %d: strike must be finite and >= 0 (got %g)", m, strike[m]);
    if (kind[m] >= mc::kUpOut && !(barrier && std::isfinite(barrier[m]) && barrier[m] > 0.0))
      return fail(ctx, DHJ_ERR_ARG, "option %d: a barrier option needs a finite barrier > 0", m);
  }
  return DHJ_OK;
}

// (chunk, option) partials the scratch holds at once; DHJ_MC_SCRATCH_ENTRIES (developer knob) lowers it so that the
// split paths of the host loop can be exercised at small sizes
int64_t mc_scratch_entries() {
  const char* e = getenv("DHJ_MC_SCRATCH_ENTRIES");
  const long long v = e ? atoll(e) : 0;
  return v > 0 ? (int64_t)v : ((int64_t)1 << 22);
}

}  // namespace

extern "C" {

int dhj_mc_price(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride, double r,
                 double q, double T, int32_t n_steps, int32_t n_obs, int32_t M, const int32_t* kind,
                 const int32_t* is_call, const double* strike, const double* barrier, uint64_t seed, int64_t n_paths,
                 double* out_price, double* out_stderr) {
  int rc = check_mc(ctx, params, P, S0, s0_stride, T, n_steps, n_obs, M, kind, is_call, strike, barrier, n_paths,
                    out_price);
  if (rc) return rc;
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  // inputs: params[P][13] | S0 | options (kind, is_call)[M] | (strike, barrier)[M]
  const size_t pb = (size_t)P * kNumParams * sizeof(double), sb = (size_t)(s0_stride ? P : 1) * sizeof(double);
  const size_t ob = (size_t)M * 2 * sizeof(int32_t), kb = (size_t)M * 2 * sizeof(double);
  std::vector<int32_t> opt((size_t)2 * M);
  std::vector<double> kbar((size_t)2 * M);
  for (int m = 0; m < M; ++m) {
    opt[2 * m] = kind[m]; opt[2 * m + 1] = is_call[m] ? 1 : 0;
    kbar[2 * m] = strike[m]; kbar[2 * m + 1] = (kind[m] >= mc::kUpOut) ? barrier[m] : 0.0;
  }
  DHJ_CUDA(ctx, ctx->d_mc_in.reserve(pb + sb + ob + kb));
  unsigned char* din = (unsigned char*)ctx->d_mc_in.p;
  DHJ_CUDA(ctx, cudaMemcpyAsync(din, params, pb, cudaMemcpyHostToDevice, st));
  DHJ_CUDA(ctx, cudaMemcpyAsync(din + pb, S0, sb, cudaMemcpyHostToDevice, st));
  DHJ_CUDA(ctx, cudaMemcpyAsync(din + pb + sb, opt.data(), ob, cudaMemcpyHostToDevice, st));
  DHJ_CUDA(ctx, cudaMemcpyAsync(din + pb + sb + ob, kbar.data(), kb, cudaMemcpyHostToDevice, st));
  // pieces: groups of whole sets while a set's partials fit the scratch, else one set at a time in runs of chunks
  const int64_t n_chunks = (n_paths + mc::kMcChunk - 1) / mc::kMcChunk;
  const int64_t cap = std::max<int64_t>(mc::kMcChunk, mc_scratch_entries());
  const int64_t per_set = n_chunks * M;
  const int64_t group = per_set <= cap ? std::min<int64_t>(P, cap / per_set) : 1;
  const int64_t run = per_set <= cap ? n_chunks : std::max<int64_t>(1, cap / M);
  const size_t part_bytes = (size_t)group * run * M * sizeof(double2);
  const size_t acc_bytes = (size_t)group * M * 3 * sizeof(double);
  DHJ_CUDA(ctx, ctx->d_mc_part.reserve(part_bytes + acc_bytes));
  DHJ_CUDA(ctx, ctx->d_mc_out.reserve((size_t)P * M * 2 * sizeof(double)));
  double2* d_part = (double2*)ctx->d_mc_part.p;
  double* d_acc = (double*)((unsigned char*)ctx->d_mc_part.p + part_bytes);
  double* d_price = (double*)ctx->d_mc_out.p;
  double* d_stderr = d_price + (size_t)P * M;
  mc::McArgs a{};
  a.s0_stride = s0_stride; a.opt = (const int*)(din + pb + sb); a.opt_kb = (const double*)(din + pb + sb + ob);
  a.r = r; a.q = q; a.dt = T / (double)n_steps; a.n_steps = n_steps; a.n_obs = n_obs; a.M = M; a.seed = seed;
  a.n_paths = n_paths; a.partial = d_part;
  mc::McFinalArgs f{};
  f.partial = d_part; f.acc = d_acc; f.n_paths = n_paths; f.M = M; f.disc = exp(-r * T);
  for (int64_t p0 = 0; p0 < P; p0 += group) {
    const int64_t g = std::min(group, P - p0);
    a.params = (const double*)din + p0 * kNumParams;
    a.S0 = (const double*)(din + pb) + p0 * s0_stride;
    a.sets = (int)g;
    f.sets = (int)g; f.price = d_price + p0 * M; f.stderr_ = d_stderr + p0 * M;
    for (int64_t c0 = 0; c0 < n_chunks; c0 += run) {
      const int64_t cn = std::min(run, n_chunks - c0);
      a.chunk0 = c0; a.chunks = cn;
      mc::k_mc_paths<<<grid_1d(g * cn), mc::kMcChunk, 0, st>>>(a);
      DHJ_LAUNCHED(ctx);
      f.chunk0 = c0; f.chunks = cn; f.first = c0 == 0; f.last = c0 + cn == n_chunks;
      mc::k_mc_finalize<<<grid_1d((g * M + 127) / 128), 128, 0, st>>>(f);
      DHJ_LAUNCHED(ctx);
    }
  }
  DHJ_CUDA(ctx, cudaMemcpyAsync(out_price, d_price, (size_t)P * M * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (out_stderr)
    DHJ_CUDA(ctx, cudaMemcpyAsync(out_stderr, d_stderr, (size_t)P * M * sizeof(double), cudaMemcpyDeviceToHost, st));
  DHJ_CUDA(ctx, cudaStreamSynchronize(st));
  return DHJ_OK;
}

}  // extern "C"

extern "C" {

// ---- checked build ---------------------------------------------------------------------------------
int dhj_debug_checks(dhj_ctx* ctx, int32_t* enabled, uint64_t* counts) {
  if (!ctx || !enabled || !counts) return fail(ctx, DHJ_ERR_ARG, "null argument");
  for (int i = 0; i < kChkCodes; ++i) counts[i] = 0;
#if defined(DHJ_CHECKED)
  *enabled = 1;
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  DHJ_CUDA(ctx, cudaDeviceSynchronize());
  unsigned long long host[kChkCodes];
  DHJ_CUDA(ctx, cudaMemcpyFromSymbol(host, g_check_fail, sizeof(host)));
  for (int i = 0; i < kChkCodes; ++i) counts[i] = host[i];
#else
  *enabled = 0;
#endif
  return DHJ_OK;
}

// ---- measurement -----------------------------------------------------------------------------
int dhj_fp64_peak(dhj_ctx* ctx, int32_t iters, double* tflops, double* milliseconds) {
  if (!ctx) return fail(nullptr, DHJ_ERR_ARG, "null context");
  if (iters < 1 || !tflops) return fail(ctx, DHJ_ERR_ARG, "bad arguments");
  DHJ_CUDA(ctx, cudaSetDevice(ctx->device));
  const int threads = 256, blocks = ctx->sm_count * 8;
  DHJ_CUDA(ctx, ctx->d_peak.reserve((size_t)threads * blocks * sizeof(double)));
  cudaEvent_t e0, e1;
  DHJ_CUDA(ctx, cudaEventCreate(&e0));
  DHJ_CUDA(ctx, cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 8; ++rep) {           // two operand forms (dhj_kernels.cuh), 4 repetitions each, the first a warm-up
    DHJ_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
    if (rep < 4) k_fp64_peak<false><<<blocks, threads, 0, ctx->stream>>>((double*)ctx->d_peak.p, iters, 0.999999, 1e-7);
    else k_fp64_peak<true><<<blocks, threads, 0, ctx->stream>>>((double*)ctx->d_peak.p, iters, 0.999999, 1e-7);
    DHJ_LAUNCHED(ctx);
    DHJ_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    DHJ_CUDA(ctx, cudaEventSynchronize(e1));
    float ms = 0.f;
    DHJ_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
    if (rep % 4 > 0) best = std::min(best, ms);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  const double flop = 2.0 * (double)threads * blocks * (double)iters * kPeakChains * kPeakUnroll;
  *tflops = flop / ((double)best * 1e-3) / 1e12;
  if (milliseconds) *milliseconds = best;
  return DHJ_OK;
}

}  // extern "C"
