// C ABI of the B200-native fast WordPiece encoder (include/wordpiece_b200.h).
// Host logic only: handle lifetime, device buffers, streams, error reporting.
// All tokenisation work happens in the CUDA kernels of wp_encode.cu; there is no
// CPU fallback — without a usable CUDA device every call fails loudly.
#include <cuda_runtime.h>
#include <emmintrin.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <functional>
#include <mutex>
#include <new>
#include <optional>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/wordpiece_b200.h"
#include "wp_encode.h"
#include "wp_vocab.h"

namespace {

thread_local std::string g_error;
const char *const kHostOnly = "host-only vocabulary handle (device -1): encoding needs a CUDA device; there is no CPU path";
std::atomic<uint64_t> g_launches{0};

// WORDPIECE_B200_TRACE=1: wall-clock milestones of a process on stderr (where does a short job's time go?)
void trace(const char *what) {
  static const bool on = std::getenv("WORDPIECE_B200_TRACE") != nullptr;
  if (!on) return;
  static const auto t0 = std::chrono::steady_clock::now();
  std::fprintf(stderr, "[wordpiece_b200 %8.2f ms] %s\n",
               std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(), what);
}
// WORDPIECE_B200_TRACE=2 additionally waits for the stream at every stage of a pipeline part, so that the
// differences between milestones are the stages' own durations (a diagnosis mode: it serialises the pipeline)
cudaError_t trace_stage(cudaStream_t stream, const char *what) {
  static const bool on = std::getenv("WORDPIECE_B200_TRACE") != nullptr && std::atoi(std::getenv("WORDPIECE_B200_TRACE")) >= 2;
  if (!on) return cudaSuccess;
  const cudaError_t e = cudaStreamSynchronize(stream);
  trace(what);
  return e;
}

wp_status fail(wp_status st, const std::string &msg) {
  g_error = msg;
  return st;
}

#define WP_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      return fail(WP_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorName(_e) + ": " + cudaGetErrorString(_e)); \
  } while (0)

// WORDPIECE_B200_POISON=1 (tests): every device allocation of the library is filled with 0xCD bytes, so that a
// kernel that reads scratch it has not written shows up in a fresh process as it would on recycled memory.
// (value = bit mask of allocation classes: 1 scratch, 2 ids / text staging, 4 pipeline slot input, 8 batch output,
// 16 tables, 32 call counters, 64 pipeline slot ids, 128 device batch (packed column, its text index, check flag);
// "1" alone therefore poisons the scratch only, 255 everything)
template <class T>
cudaError_t dev_alloc(T **p, size_t bytes, int cls = 127) {
  cudaError_t e = cudaMalloc(reinterpret_cast<void **>(p), bytes);
  static const int poison = std::getenv("WORDPIECE_B200_POISON") ? std::atoi(std::getenv("WORDPIECE_B200_POISON")) : 0;
  if (e == cudaSuccess && (poison & cls)) {
    e = cudaMemset(*p, 0xCD, bytes);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();  // (the library's streams do not wait for the null stream)
  }
  return e;
}

struct DeviceGuard {
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    ok = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// An array that frees itself: device memory (dev_alloc, poison class `cls`) or pinned host memory.  grow(n) makes
// room for at least n elements and reallocates only when n exceeds the capacity: exactly n the first time, an
// eighth and 256 bytes more when it has to grow again, so that a handle's memory follows its largest call and is
// never reallocated per call.  An empty array makes no CUDA call (host-only handles run on machines without one).
template <class T, bool kPinned>
class Buffer {
 public:
  T *p = nullptr;
  size_t cap = 0;  // elements
  explicit Buffer(int cls = 127) : cls_(cls) {}
  Buffer(Buffer &&o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)), cls_(o.cls_) {}
  Buffer &operator=(Buffer &&) = delete;
  ~Buffer() { release(); }
  cudaError_t grow(size_t n) {
    if (n <= cap) return cudaSuccess;
    const size_t want = cap ? n + n / 8 + 256 / sizeof(T) : n;
    release();
    const cudaError_t e = kPinned ? cudaMallocHost(reinterpret_cast<void **>(&p), want * sizeof(T))
                                  : dev_alloc(&p, want * sizeof(T), cls_);
    if (e == cudaSuccess) cap = want;
    return e;
  }

 private:
  void release() {
    if (p) kPinned ? cudaFreeHost(p) : cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  int cls_;
};
template <class T>
using DeviceBuffer = Buffer<T, false>;
template <class T>
using PinnedBuffer = Buffer<T, true>;

// A CUDA event or stream that destroys itself
template <class H, cudaError_t (*Destroy)(H)>
struct Owned {
  H h = nullptr;
  Owned() = default;
  Owned(Owned &&o) noexcept : h(std::exchange(o.h, nullptr)) {}
  Owned &operator=(Owned &&) = delete;
  ~Owned() {
    if (h) Destroy(h);
  }
  operator H() const { return h; }
};
using Event = Owned<cudaEvent_t, cudaEventDestroy>;
using Stream = Owned<cudaStream_t, cudaStreamDestroy>;


constexpr size_t kRangeBytesMax = size_t(64) << 20;  // text bytes encoded per K1/K2/K3 round (bounds the scratch)
constexpr uint32_t kWorkWordSlotsLog2 = 20;          // working word table of a large call: 2^20 slots of 64 bytes = 64 MiB
constexpr size_t kMemoMinBytes = size_t(4) << 20;    // texts below this use the static word table as it is: recording
                                                     // words into a working copy would only cost the copy
static_assert(kRangeBytesMax / 2 + 1024 <= (size_t(1) << wp::SEG_SLOW_INDEX_BITS), "slow indices must fit seg_result");

}  // namespace

struct wp_vocab {
  wp::HostVocab host;
  int device = 0;
  Stream stream;
  // device tables
  DeviceBuffer<wp::Edge> d_edges{16};
  DeviceBuffer<wp::WordSlot> d_words_static{16};  // image built from the vocabulary, never written by a kernel
  DeviceBuffer<wp::WordSlot> d_words_work{16};    // per-call working table K2 records into (allocated on the first large call)
  uint32_t work_words_log2 = 0;
  size_t device_bytes = 0;
  DeviceBuffer<uint8_t> d_work{1};  // scratch (layout: see Workspace below)
  DeviceBuffer<wp::CallCounters> d_call{32};
  int sm_count = 0;
  size_t persist_words_bytes = 0, persist_edges_bytes = 0, persist_work_bytes = 0;  // L2 access-policy windows
  float persist_words_ratio = 0.f, persist_edges_ratio = 0.f, persist_work_ratio = 0.f;
  size_t set_aside = 0, max_window = 0;
  DeviceBuffer<uint8_t> d_text{2};  // staging of the single-shot host-buffer path
  DeviceBuffer<int32_t> d_ids{2};
  DeviceBuffer<char> d_fmt;  // wp_encode_text: the ids as decimal text
  PinnedBuffer<wp::CallCounters> h_call;
  // The host pipeline (run_pipeline): input block in pinned host memory and on the device, ids, a batch part's
  // per-text outputs (first segment, first id) and id offsets, counters, pinned id staging for pageable callers
  struct Slot {
    PinnedBuffer<uint8_t> h_in;
    DeviceBuffer<uint8_t> d_in{4};
    DeviceBuffer<int32_t> d_ids{64};
    DeviceBuffer<uint8_t> d_out{8};
    PinnedBuffer<unsigned long long> h_offsets;
    PinnedBuffer<wp::CallCounters> h_call;
    PinnedBuffer<int32_t> h_ids;
    Event h2d_done, cmp_done, d2h_done;
  } slot[3];
  Stream s_h2d, s_d2h;
  // The device batch (wp_encode_batch_device): the column packed into whole tiles (16-byte aligned for K1's vector
  // loads), the text starts, the tile index, K1's first segments, and the column check's flag (a word of its own:
  // enqueue_encode clears the call counters after the check has run).  Never shared with the pipeline's slots,
  // whose input the host pipeline writes without waiting for the handle's previous call.
  DeviceBuffer<uint8_t> d_col_text{128};
  DeviceBuffer<unsigned long long> d_col_bounds{128};
  DeviceBuffer<uint32_t> d_col_tile_bound{128};
  DeviceBuffer<uint32_t> d_col_bound_seg{128};
  DeviceBuffer<unsigned int> d_col_bad{128};
  PinnedBuffer<unsigned int> h_col_bad;
  // every call on a handle shares its scratch, counters and word table: the kernels of one call must have
  // finished before those of the next begin, on whatever streams the caller enqueues them
  Event last_done;
  bool use_ticket = false;  // K1 hands its tiles out by ticket (set for good once a look-back has stalled, see wp_encode.cu)
  bool dense_tiles = false; // K1 with full-capacity segment lists (set for good once a tile overflowed the regular ones)
  // optional per-kernel timing (wp_set_kernel_timing): events around K1/K2/K3 of every range
  bool timing = false;
  std::vector<Event> timing_events;  // 4 per range of the last call
  size_t timing_used = 0;
  wp_stats stats{};
};

namespace {

uint32_t log2_of(size_t pow2) {
  uint32_t l = 0;
  while ((size_t(1) << l) < pow2) l++;
  return l;
}

wp::DeviceVocab device_view(const wp_vocab *v) {
  wp::DeviceVocab d{};
  d.edges = v->d_edges.p;
  d.edge_mask = static_cast<uint32_t>(v->host.edges.size() - 1);
  d.edge_shift = 32 - log2_of(v->host.edges.size());
  d.unk_id = v->host.unk_id;
  d.han_swallow = v->host.max_len >= 2 ? 1u : 0u;
  return d;
}

wp_status upload(wp_vocab *v) {
  const wp::HostVocab &h = v->host;
  const size_t b_edges = h.edges.size() * sizeof(wp::Edge);
  const size_t b_words = h.words.size() * sizeof(wp::WordSlot);
  WP_CUDA(v->d_edges.grow(h.edges.size()));
  WP_CUDA(v->d_words_static.grow(h.words.size()));
  WP_CUDA(cudaMemcpy(v->d_edges.p, h.edges.data(), b_edges, cudaMemcpyHostToDevice));
  WP_CUDA(cudaMemcpy(v->d_words_static.p, h.words.data(), b_words, cudaMemcpyHostToDevice));
  v->device_bytes = b_edges + b_words;
  for (Stream *s : {&v->stream, &v->s_h2d, &v->s_d2h}) WP_CUDA(cudaStreamCreateWithFlags(&s->h, cudaStreamNonBlocking));
  WP_CUDA(v->h_call.grow(1));
  WP_CUDA(v->d_call.grow(1));
  WP_CUDA(cudaDeviceGetAttribute(&v->sm_count, cudaDevAttrMultiProcessorCount, v->device));
  {
    // keep the table a kernel reads at random resident in L2 (best effort: an unsupported attribute only
    // costs the hint).  The set-aside is sized for the word table; the hit ratio scales a window down to it.
    int max_persist = 0, max_window = 0;
    if (cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, v->device) == cudaSuccess &&
        cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, v->device) == cudaSuccess &&
        max_persist > 0 && max_window > 0) {
      size_t want = b_words > b_edges ? b_words : b_edges;
      if (want < (size_t(1) << kWorkWordSlotsLog2) * sizeof(wp::WordSlot)) want = (size_t(1) << kWorkWordSlotsLog2) * sizeof(wp::WordSlot);
      size_t set_aside = want < static_cast<size_t>(max_persist) ? want : static_cast<size_t>(max_persist);
      size_t current = 0;
      cudaDeviceGetLimit(&current, cudaLimitPersistingL2CacheSize);
      if (current >= set_aside || cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, set_aside) == cudaSuccess) {
        if (current > set_aside) set_aside = current;
        auto fit = [&](size_t bytes, size_t *win, float *ratio) {
          *win = bytes < static_cast<size_t>(max_window) ? bytes : static_cast<size_t>(max_window);
          *ratio = static_cast<float>(set_aside) / static_cast<float>(*win);
          if (*ratio > 1.f) *ratio = 1.f;
        };
        fit(b_words, &v->persist_words_bytes, &v->persist_words_ratio);
        fit(b_edges, &v->persist_edges_bytes, &v->persist_edges_ratio);
        v->set_aside = set_aside;
        v->max_window = static_cast<size_t>(max_window);
      }
    }
    cudaGetLastError();
  }
  return WP_OK;
}

// Scratch of one range of `range_bytes` text bytes.  Capacities are the exact worst cases, so the only
// overflow that can happen is the id spill of segments walked from global memory (words longer than a
// tile's window may be arbitrarily long); `spill_ids` bounds that part and the caller retries with more.
struct Workspace {
  size_t zero_bytes;     // counters + look-back words, zeroed before every range
  size_t off_tile_state, off_block_state, off_seg, off_slow, off_long, off_arena, total;
  uint32_t n_tiles, n_scatter_blocks, seg_cap, slow_cap, long_cap, arena_cap;
};

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

Workspace plan_workspace(size_t range_bytes, size_t spill_ids) {
  Workspace w{};
  const size_t tile = wp::encode_tile_bytes();
  w.n_tiles = static_cast<uint32_t>((range_bytes + tile - 1) / tile);
  const size_t padded = static_cast<size_t>(w.n_tiles) * tile;
  w.seg_cap = static_cast<uint32_t>(padded);                  // a segment has at least one byte
  w.slow_cap = static_cast<uint32_t>(padded / 2 + 1024);      // an unsettled segment has at least two
  // arena words per tile: its slow segments lie inside the window (tile + 256 bytes) and each takes
  // len + ceil(len / 4) words => at most 1.25 x window + 0.75 x (tile / 2 + 8) < 7000; + the spill of LONG segments
  size_t arena = static_cast<size_t>(w.n_tiles) * 7000 + 4096 + spill_ids;
  if (arena > 0xFFFFFFF0ull) arena = 0xFFFFFFF0ull;
  w.arena_cap = static_cast<uint32_t>(arena);
  w.n_scatter_blocks = static_cast<uint32_t>((w.seg_cap + wp::scatter_block_segments() - 1) / wp::scatter_block_segments());
  size_t off = align_up(sizeof(wp::RangeCounters), 256);
  w.off_tile_state = off;
  off += static_cast<size_t>(w.n_tiles) * 8;
  w.off_block_state = off;
  off += static_cast<size_t>(w.n_scatter_blocks) * 8;
  w.zero_bytes = off;
  off = align_up(off, 256);
  w.off_seg = off;
  off = align_up(off + static_cast<size_t>(w.seg_cap) * 4, 256);
  w.off_slow = off;
  off = align_up(off + static_cast<size_t>(w.slow_cap) * sizeof(wp::SlowEntry), 256);
  w.off_long = off;
  w.long_cap = w.n_tiles * 18 + 16;  // per tile: segments of more than 256 bytes (<= 17) and one that leaves the window
  off = align_up(off + static_cast<size_t>(w.long_cap) * 4, 256);
  w.off_arena = off;
  off = align_up(off + static_cast<size_t>(w.arena_cap) * 4, 256);
  w.total = off;
  return w;
}

// A batch of texts packed into one buffer (wp_encode_batch, wp_encode_batch_device): see EncodeParams::bounds.
struct BatchArgs {
  const unsigned long long *h_bounds = nullptr;  // host copy of the text starts (ascending), n_texts entries; null:
                                                 // K5 reads the texts of a range from d_tile_bound on the device
  size_t n_texts = 0;
  const unsigned long long *d_bounds = nullptr;
  const uint32_t *d_tile_bound = nullptr;
  uint32_t *d_bound_seg = nullptr;
  unsigned long long *d_offsets = nullptr;
};

struct EnqueueInfo {
  uint32_t n_tiles = 0;
  uint32_t n_ranges = 0;
  uint64_t launches = 0;
};

// Enqueue the kernels for a whole text on `stream`: K1/K2/K3 per range of at most kRangeBytesMax bytes.
// No synchronisation.  The running id count ends up in d_call->ids_total[n_ranges & 1].
// `warm` = a later chunk of one pipelined call: the memo is neither cleared nor warmed up again.
wp_status enqueue_encode(wp_vocab *v, const void *d_text, size_t n_bytes, int32_t *d_ids, size_t capacity,
                         cudaStream_t stream, size_t spill_ids, EnqueueInfo *info, bool warm = false,
                         size_t call_bytes = 0, const BatchArgs *batch = nullptr) {
  const size_t tile = wp::encode_tile_bytes();
  const size_t n_tiles = (n_bytes + tile - 1) / tile;
  if (n_tiles > 0x7FFFFFFFull) return fail(WP_ERR_INVALID_ARG, "text too large for one call (> 2^31 tiles)");
  size_t range_max = kRangeBytesMax;
  if (const char *e = std::getenv("WORDPIECE_B200_RANGE_BYTES")) {  // test hook: force several ranges on small texts
    const long long x = std::atoll(e);
    if (x > 0 && static_cast<size_t>(x) < range_max) range_max = (static_cast<size_t>(x) + tile - 1) / tile * tile;
  }
  const size_t range_bytes = n_bytes < range_max ? n_bytes : range_max;
  const Workspace w = plan_workspace(range_bytes, spill_ids ? spill_ids : range_bytes + tile);
  if (!v->last_done) WP_CUDA(cudaEventCreateWithFlags(&v->last_done.h, cudaEventDisableTiming));
  WP_CUDA(cudaStreamWaitEvent(stream, v->last_done, 0));  // (a never-recorded event does not block)
  WP_CUDA(cudaMemsetAsync(v->d_call.p, 0, sizeof(wp::CallCounters), stream));
  v->timing_used = 0;
  bool use_memo = (call_bytes ? call_bytes : n_bytes) >= kMemoMinBytes;  // judged on the whole user call
  if (const char *e = std::getenv("WORDPIECE_B200_MEMO")) use_memo = std::atoi(e) != 0;  // 0 = off, 1 = on (tests)
  uint64_t launches = 0;
  if (use_memo) {
    if (!v->d_words_work.p) {
      uint32_t lg = kWorkWordSlotsLog2;
      if (const char *e = std::getenv("WORDPIECE_B200_WORD_SLOTS_LOG2")) {  // test hook: a small, crowded table
        const int x = std::atoi(e);
        if (x >= 6 && x <= 26) lg = static_cast<uint32_t>(x);
      }
      const uint32_t static_lg = log2_of(v->host.words.size());
      if (lg < static_lg) lg = static_lg;  // the static words must fit with room to spare
      WP_CUDA(v->d_words_work.grow(size_t(1) << lg));
      v->work_words_log2 = lg;
      if (v->persist_words_bytes) {
        const size_t b = (size_t(1) << lg) * sizeof(wp::WordSlot);
        v->persist_work_bytes = b < v->max_window ? b : v->max_window;
        v->persist_work_ratio = static_cast<float>(v->set_aside) / static_cast<float>(v->persist_work_bytes);
        if (v->persist_work_ratio > 1.f) v->persist_work_ratio = 1.f;
      }
    }
    // every user call starts from the static words only: what K2 records never outlives the call (the chunks
    // of one pipelined host-buffer call share it), so neither ids nor timing depend on earlier calls
    if (!warm)
      WP_CUDA(wp::launch_seed_words(v->d_words_static.p, static_cast<uint32_t>(v->host.words.size()), v->d_words_work.p,
                                    v->work_words_log2, stream, &launches));
  }
  wp::EncodeParams P{};
  P.vocab = device_view(v);
  P.text = static_cast<const uint8_t *>(d_text);
  P.n_bytes = n_bytes;
  P.ids = d_ids;
  P.capacity = capacity;
  P.call = v->d_call.p;
  P.seg_capacity = w.seg_cap;
  P.slow_capacity = w.slow_cap;
  P.long_capacity = w.long_cap;
  P.arena_capacity = w.arena_cap;
  P.n_scatter_blocks = w.n_scatter_blocks;
  P.words = use_memo ? v->d_words_work.p : v->d_words_static.p;
  const uint32_t words_log2 = use_memo ? v->work_words_log2 : log2_of(v->host.words.size());
  P.word_mask = (1u << words_log2) - 1u;
  P.word_shift = 32 - words_log2;
  P.record_words = use_memo ? 1u : 0u;
  P.use_ticket = v->use_ticket ? 1u : 0u;
  P.dense_tiles = v->dense_tiles ? 1u : 0u;
  if (const char *e = std::getenv("WORDPIECE_B200_TICKET")) P.use_ticket = std::atoi(e) != 0 ? 1u : 0u;  // test hook
  P.persist_words_bytes = use_memo ? v->persist_work_bytes : v->persist_words_bytes;
  P.persist_words_ratio = use_memo ? v->persist_work_ratio : v->persist_words_ratio;
  P.persist_edges_bytes = v->persist_edges_bytes;
  P.persist_edges_ratio = v->persist_edges_ratio;
  if (batch) {
    P.bounds = batch->d_bounds;
    P.tile_bound = batch->d_tile_bound;
    P.bound_seg = batch->d_bound_seg;
    P.id_offsets = batch->d_offsets;
  }
  // batch calls: the texts [i0, i1) that start in the range whose K3 was just enqueued get their id offsets
  auto text_offsets = [&]() -> cudaError_t {
    if (!batch) return cudaSuccess;
    if (!batch->h_bounds) return wp::launch_text_offsets_device(P, v->sm_count, stream, &launches);
    const unsigned long long lo = static_cast<unsigned long long>(P.first_tile) * tile;
    const unsigned long long hi = lo + static_cast<unsigned long long>(P.n_tiles) * tile;
    const unsigned long long *b = batch->h_bounds, *e = b + batch->n_texts;
    const uint32_t i0 = static_cast<uint32_t>(std::lower_bound(b, e, lo) - b);
    const uint32_t i1 = static_cast<uint32_t>(std::lower_bound(b, e, hi) - b);
    return wp::launch_text_offsets(P, i0, i1, stream, &launches);
  };
  // Two small ranges first (2 MiB, 8 MiB): the first fills the word memo — its own unsettled words all go
  // through K2 — the second shows whether the text repeats its words (memo_worthwhile), so that the bulk of
  // the text, in full ranges, either finds the frequent repeats in the memo or does not pay for it.
  std::vector<std::pair<size_t, size_t>> ranges;  // first tile, tile count
  {
    size_t next_tiles = w.n_tiles;
    if (use_memo && !warm) {
      const size_t first_tiles = (size_t(2) << 20) / tile;
      if (first_tiles < next_tiles) next_tiles = first_tiles;
    }
    for (size_t first = 0; first < n_tiles;) {
      const size_t count = n_tiles - first < next_tiles ? n_tiles - first : next_tiles;
      ranges.emplace_back(first, count);
      first += count;
      // 2 MiB, then 8 MiB (enough lookups to judge whether the memo pays on this text), then full ranges
      next_tiles = (use_memo && !warm && ranges.size() == 1 && ((size_t(8) << 20) / tile) < w.n_tiles) ? (size_t(8) << 20) / tile
                                                                                                       : w.n_tiles;
    }
  }
  const uint32_t n_ranges = static_cast<uint32_t>(ranges.size());

  WP_CUDA(v->d_work.grow(w.total));
  uint8_t *const scratch = v->d_work.p;
  P.counters = reinterpret_cast<wp::RangeCounters *>(scratch);
  P.tile_state = reinterpret_cast<unsigned long long *>(scratch + w.off_tile_state);
  P.block_state = reinterpret_cast<unsigned long long *>(scratch + w.off_block_state);
  P.seg_result = reinterpret_cast<uint32_t *>(scratch + w.off_seg);
  P.slow = reinterpret_cast<wp::SlowEntry *>(scratch + w.off_slow);
  P.long_list = reinterpret_cast<uint32_t *>(scratch + w.off_long);
  P.arena = reinterpret_cast<uint32_t *>(scratch + w.off_arena);
  for (uint32_t range = 0; range < n_ranges; range++) {
    P.first_tile = static_cast<uint32_t>(ranges[range].first);
    P.n_tiles = static_cast<uint32_t>(ranges[range].second);
    P.range_parity = range & 1u;
    P.range_index = warm ? range + 2 : range;
    static const bool poison_scratch = std::getenv("WORDPIECE_B200_POISON_SCRATCH") != nullptr;
    if (poison_scratch)  // (tests) everything a range must write before it reads, filled with 0xCD on the launching stream
      WP_CUDA(cudaMemsetAsync(scratch + w.off_seg, 0xCD, w.total - w.off_seg, stream));
    WP_CUDA(cudaMemsetAsync(scratch, 0, w.zero_bytes, stream));
    cudaEvent_t tev[4];
    if (v->timing) {
      while (v->timing_events.size() < v->timing_used + 4) {
        Event e;
        WP_CUDA(cudaEventCreate(&e.h));
        v->timing_events.push_back(std::move(e));
      }
      for (int k = 0; k < 4; k++) tev[k] = v->timing_events[v->timing_used + k];
      v->timing_used += 4;
    }
    WP_CUDA(wp::launch_encode_range(P, v->sm_count, stream, &launches, v->timing ? tev : nullptr));
    WP_CUDA(text_offsets());
  }
  WP_CUDA(cudaEventRecord(v->last_done, stream));
  g_launches.fetch_add(launches, std::memory_order_relaxed);
  info->n_tiles = static_cast<uint32_t>(n_tiles);
  info->n_ranges = n_ranges;
  info->launches = launches;
  return WP_OK;
}

// The outcome of a finished call of n_bytes text bytes, from its counters (as copied to the host) and its
// EnqueueInfo.  The K1 modes the call asked for are switched on for the handle for good, and its statistics are
// added to *acc.  Returns true if the call's ids are void (a scratch capacity was exceeded): the call is then
// repeated with the id spill left in *spill — unchanged if the overflow switched a K1 mode on, which is cure
// enough, else one as large as the text.  Every repeat so turns on one of three one-way switches (ticket, dense
// tiles, large spill), and kMaxAttempts bounds the repeats of every entry point.
constexpr int kMaxAttempts = 1 + 3;
bool absorb_call(wp_vocab *v, const wp::CallCounters &c, const EnqueueInfo &info, size_t n_bytes, wp_stats *acc,
                 size_t *spill) {
  const bool switched = (c.stalled && !v->use_ticket) || (c.dense && !v->dense_tiles);
  if (c.stalled) v->use_ticket = true;  // a K1 look-back gave up: from now on tiles go by ticket
  if (c.dense) v->dense_tiles = true;   // a tile with more segments than the regular K1's lists hold
  acc->n_tiles += info.n_tiles;
  acc->dirty_tiles += c.dirty_tiles;
  acc->long_segments += c.long_segments;
  acc->memo_hits += c.memo_hits;
  acc->kernel_launches += info.launches;
  if (!c.overflow) return false;
  if (!switched) *spill = n_bytes + 4096;
  return true;
}

// One call of n_bytes text bytes, repeated while its ids are void (absorb_call), the first time with id spill
// `spill`.  attempt(spill, &info) enqueues the call on `stream` and a copy of its counters to `counters` (pinned).
template <class Attempt>
wp_status repeat_call(wp_vocab *v, cudaStream_t stream, size_t n_bytes, size_t spill,
                      const wp::CallCounters &counters, Attempt &&attempt) {
  for (int i = 0; i < kMaxAttempts; i++) {
    EnqueueInfo info;
    const wp_status st = attempt(spill, &info);
    if (st != WP_OK) return st;
    WP_CUDA(cudaStreamSynchronize(stream));
    wp_stats acc{};
    if (absorb_call(v, counters, info, n_bytes, &acc, &spill)) continue;
    v->stats = acc;
    v->stats.n_bytes = n_bytes;
    v->stats.n_ids = counters.ids_total[info.n_ranges & 1u];
    return WP_OK;
  }
  return fail(WP_ERR_CUDA, "internal scratch overflow");
}

// A device-resident text, encoded and waited for
wp_status run_encode(wp_vocab *v, const void *d_text, size_t n_bytes, int32_t *d_ids, size_t capacity,
                     cudaStream_t stream, size_t spill = 0) {
  return repeat_call(v, stream, n_bytes, spill, *v->h_call.p, [&](size_t sp, EnqueueInfo *info) -> wp_status {
    const wp_status st = enqueue_encode(v, d_text, n_bytes, d_ids, capacity, stream, sp, info);
    if (st != WP_OK) return st;
    WP_CUDA(cudaMemcpyAsync(v->h_call.p, v->d_call.p, sizeof(wp::CallCounters), cudaMemcpyDeviceToHost, stream));
    return WP_OK;
  });
}

// ---- the device batch (wp_encode_batch_device): a string column in device memory, packed on the device as
// wp_encode_batch packs host texts (pack_part), encoded in one call of the kernels

// Check and pack the column into the handle's device batch buffers, on `stream` behind the handle's previous call
// (which may still read them).  `packed` = n_chars + n_texts bytes, whole tiles of which are written.
wp_status enqueue_column(wp_vocab *v, const void *d_chars, size_t n_chars, const uint64_t *d_offsets, size_t n_texts,
                         size_t packed, cudaStream_t stream, uint64_t *launches) {
  const size_t tile = wp::encode_tile_bytes();
  const size_t n_tiles = (packed + tile - 1) / tile;
  WP_CUDA(v->d_col_text.grow(n_tiles * tile));
  WP_CUDA(v->d_col_bounds.grow(n_texts));
  WP_CUDA(v->d_col_tile_bound.grow(n_tiles + 1));
  WP_CUDA(v->d_col_bound_seg.grow(n_texts));
  WP_CUDA(v->d_col_bad.grow(1));
  if (!v->last_done) WP_CUDA(cudaEventCreateWithFlags(&v->last_done.h, cudaEventDisableTiming));
  WP_CUDA(cudaStreamWaitEvent(stream, v->last_done, 0));
  WP_CUDA(cudaMemsetAsync(v->d_col_bad.p, 0, sizeof(unsigned int), stream));
  wp::ColumnArgs A{};
  A.chars = static_cast<const uint8_t *>(d_chars);
  A.n_chars = n_chars;
  A.offsets = reinterpret_cast<const unsigned long long *>(d_offsets);
  A.n_texts = static_cast<uint32_t>(n_texts);
  A.n_tiles = static_cast<uint32_t>(n_tiles);
  A.bad = v->d_col_bad.p;
  A.text = v->d_col_text.p;
  A.bounds = v->d_col_bounds.p;
  A.tile_bound = v->d_col_tile_bound.p;
  uint64_t n = 0;
  WP_CUDA(wp::launch_column_pack(A, stream, &n));
  g_launches.fetch_add(n, std::memory_order_relaxed);
  *launches += n;
  return WP_OK;
}

// The kernels over the packed column (enqueue_column) into d_ids, K5 writing d_id_offsets[0, n_texts), then
// d_id_offsets[n_texts] <- the id count, or UINT64_MAX if the call's ids are void or the column is malformed.
wp_status enqueue_column_encode(wp_vocab *v, size_t packed, size_t n_texts, int32_t *d_ids, size_t capacity,
                                uint64_t *d_id_offsets, cudaStream_t stream, size_t spill, EnqueueInfo *info) {
  BatchArgs batch;  // (no h_bounds: K5 takes the texts of every range from the tile index)
  batch.n_texts = n_texts;
  batch.d_bounds = v->d_col_bounds.p;
  batch.d_tile_bound = v->d_col_tile_bound.p;
  batch.d_bound_seg = v->d_col_bound_seg.p;
  batch.d_offsets = reinterpret_cast<unsigned long long *>(d_id_offsets);
  const wp_status st = enqueue_encode(v, v->d_col_text.p, packed, d_ids, capacity, stream, spill, info, false, 0, &batch);
  if (st != WP_OK) return st;
  uint64_t launches = 0;
  WP_CUDA(wp::launch_publish_count(v->d_call.p, info->n_ranges & 1u, batch.d_offsets + n_texts, stream, &launches,
                                   v->d_col_bad.p));
  WP_CUDA(cudaEventRecord(v->last_done, stream));  // (the count reads the counters and the flag the next call clears)
  g_launches.fetch_add(launches, std::memory_order_relaxed);
  info->launches += launches;
  return WP_OK;
}

// Host text -> ids in the handle's device buffer v->d_ids (count in v->stats.n_ids), through the staging buffer
// v->d_text.  The id buffer holds at least ids_want ids; `retry_short`: if that was too few, once more with the
// exact count (the launches of both attempts are counted).
wp_status encode_staged(wp_vocab *v, const char *text, size_t n_bytes, size_t ids_want, bool retry_short,
                        size_t spill = 0) {
  WP_CUDA(v->d_text.grow(n_bytes));
  WP_CUDA(cudaMemcpyAsync(v->d_text.p, text, n_bytes, cudaMemcpyHostToDevice, v->stream));
  for (int attempt = 0;; attempt++) {
    WP_CUDA(v->d_ids.grow(ids_want));
    const uint64_t before = v->stats.kernel_launches;
    const wp_status st = run_encode(v, v->d_text.p, n_bytes, v->d_ids.p, v->d_ids.cap, v->stream, spill);
    if (st != WP_OK) return st;
    if (attempt) v->stats.kernel_launches += before;
    if (!retry_short || attempt || v->stats.n_ids <= v->d_ids.cap) return WP_OK;
    ids_want = static_cast<size_t>(v->stats.n_ids);
  }
}

// ---- copies into pinned staging memory with STREAMING (non-temporal) stores
// Measured on the B200 box (profiles/r2r_batch_stages.txt): the H2D copy of an 8 MiB pinned block that the CPU
// has just written with ordinary stores runs at 6 GB/s, a D2H of the same size at 50 GB/s — the DMA engine has to
// pull every line out of the writing cores' caches.  Streaming stores go to memory through the write-combining
// buffers and leave nothing behind in the caches, so the copy engine reads plain DRAM.  (glibc's memcpy does this
// on its own only above a threshold of several MB per call.)  WORDPIECE_B200_STREAM_STORES=0 switches back.
bool stream_stores() {
  static const bool on = [] {
    const char *e = std::getenv("WORDPIECE_B200_STREAM_STORES");
    return e == nullptr || std::atoi(e) != 0;
  }();
  return on;
}

// dst 64-byte aligned, n a multiple of 64
inline void stream_lines(char *dst, const char *src, size_t n) {
  for (size_t i = 0; i < n; i += 64) {
    const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i));
    const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i + 16));
    const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i + 32));
    const __m128i d = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i + 48));
    _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i), a);
    _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 16), b);
    _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 32), c);
    _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 48), d);
  }
}

// memcpy whose whole cache lines are written with streaming stores (the ragged head and tail with ordinary ones).
// The caller issues stream_fence() once it has written its share, before anybody is told that the data is there.
inline void stream_copy(void *dst, const void *src, size_t n) {
  char *d = static_cast<char *>(dst);
  const char *s = static_cast<const char *>(src);
  if (n < 256) {
    std::memcpy(d, s, n);
    return;
  }
  const size_t head = (64 - (reinterpret_cast<uintptr_t>(d) & 63u)) & 63u;
  std::memcpy(d, s, head);
  const size_t body = (n - head) & ~size_t(63);
  stream_lines(d + head, s + head, body);
  std::memcpy(d + head + body, s + head + body, n - head - body);
}
inline void stream_fence() { _mm_sfence(); }

// Many small pieces -> one contiguous destination, streamed: the pieces are gathered in a small buffer that
// stays in the core's L1 and leave it as whole cache lines, so that a line shared by two texts is still written
// once, by one streaming store.
class StreamWriter {
 public:
  explicit StreamWriter(char *dst) : dst_(dst) {}
  void put(const char *p, size_t n) {
    while (n) {
      if (fill_ == 0 && (reinterpret_cast<uintptr_t>(dst_) & 63u)) {  // (only at the start: up to the first line border)
        size_t k = 64 - (reinterpret_cast<uintptr_t>(dst_) & 63u);
        if (k > n) k = n;
        std::memcpy(dst_, p, k);
        dst_ += k;
        p += k;
        n -= k;
        continue;
      }
      if (fill_ == 0 && n >= sizeof(buf_)) {  // a long piece: straight from the source
        const size_t k = n & ~size_t(63);
        stream_lines(dst_, p, k);
        dst_ += k;
        p += k;
        n -= k;
        continue;
      }
      size_t k = sizeof(buf_) - fill_;
      if (k > n) k = n;
      std::memcpy(buf_ + fill_, p, k);
      fill_ += k;
      p += k;
      n -= k;
      if (fill_ == sizeof(buf_)) {
        stream_lines(dst_, buf_, fill_);
        dst_ += fill_;
        fill_ = 0;
      }
    }
  }
  void put(char c) { put(&c, 1); }
  void finish() {
    const size_t k = fill_ & ~size_t(63);
    stream_lines(dst_, buf_, k);
    std::memcpy(dst_ + k, buf_ + k, fill_ - k);
    dst_ += fill_;
    fill_ = 0;
    stream_fence();
  }

 private:
  char *dst_;
  size_t fill_ = 0;
  alignas(64) char buf_[8192];
};

// Host threads that copy between a caller's pageable memory and the pinned staging buffers of the pipeline.
// One memcpy stream moves 5-10 GB/s (less into pages that are touched for the first time, e.g. the storage of
// a fresh std::vector), a quarter of what PCIe 5 x16 takes: the copy is cut into one slice per thread.
// Process-wide, started on first use, never joined (the threads sleep on a condition variable).
class CopyPool {
 public:
  static CopyPool &get() {
    static CopyPool *pool = new CopyPool();  // leaked on purpose: no static-destruction order to get wrong
    return *pool;
  }
  // job(part, parts) on every thread of the pool and on the caller (part 0); returns when all parts are done
  template <class F>
  void run(F &&job) {
    if (n_workers_ == 0) {
      job(size_t(0), size_t(1));
      return;
    }
    std::unique_lock<std::mutex> call(call_mu_);  // one job at a time
    std::function<void(size_t, size_t)> f = std::ref(job);
    {
      std::lock_guard<std::mutex> lk(mu_);
      job_ = &f;
      pending_ = n_workers_;
      gen_++;
    }
    cv_work_.notify_all();
    job(size_t(0), n_workers_ + 1);
    std::unique_lock<std::mutex> lk(mu_);
    cv_done_.wait(lk, [&] { return pending_ == 0; });
    job_ = nullptr;
  }
  // memcpy(dst, src, n) in one slice per thread.  `streamed`: the destination is pinned memory that a copy engine
  // reads next (see stream_copy).
  void copy(void *dst, const void *src, size_t n, bool streamed = false) {
    streamed = streamed && stream_stores();
    if (n < (size_t(1) << 20) || n_workers_ == 0) {
      if (streamed) {
        stream_copy(dst, src, n);
        stream_fence();
      } else {
        std::memcpy(dst, src, n);
      }
      return;
    }
    run([&](size_t part, size_t parts) {
      const size_t slice = ((n + parts - 1) / parts + 4095) & ~size_t(4095);
      const size_t lo = part * slice;
      if (lo >= n) return;
      const size_t len = n - lo < slice ? n - lo : slice;
      if (streamed) {
        stream_copy(static_cast<char *>(dst) + lo, static_cast<const char *>(src) + lo, len);
        stream_fence();
      } else {
        std::memcpy(static_cast<char *>(dst) + lo, static_cast<const char *>(src) + lo, len);
      }
    });
  }

 private:
  CopyPool() {
    // all cores, at most 16: the copies are bound by what one core can move (measured on the 16-core B200 host, 1 GiB
    // through fast::encode(std::string): 4 threads 0.187 s, 8 0.10-0.14 s, 12 0.093 s, 16 0.078 s); the threads
    // sleep between copies
    size_t n = std::thread::hardware_concurrency();
    if (n > 16) n = 16;
    if (const char *e = std::getenv("WORDPIECE_B200_COPY_THREADS")) {
      const int x = std::atoi(e);
      if (x >= 1 && x <= 64) n = static_cast<size_t>(x);
    }
    n_workers_ = n > 1 ? n - 1 : 0;
    for (size_t i = 0; i < n_workers_; i++) std::thread([this, i] { work(i + 1); }).detach();
  }
  void work(size_t index) {
    uint64_t seen = 0;
    for (;;) {
      std::function<void(size_t, size_t)> *f;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_work_.wait(lk, [&] { return gen_ != seen; });
        seen = gen_;
        f = job_;
      }
      (*f)(index, n_workers_ + 1);
      {
        std::lock_guard<std::mutex> lk(mu_);
        pending_--;
      }
      cv_done_.notify_one();
    }
  }
  std::mutex call_mu_, mu_;
  std::condition_variable cv_work_, cv_done_;
  size_t n_workers_ = 0;
  uint64_t gen_ = 0;
  size_t pending_ = 0;
  std::function<void(size_t, size_t)> *job_ = nullptr;
};

// Is this host pointer pageable memory (neither cudaMallocHost nor cudaHostRegister memory)?  Copies from and
// to it are staged by the driver through one thread; the pipeline stages them itself, with several.
bool is_pageable(const void *p) {
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return a.type == cudaMemoryTypeUnregistered;
}

constexpr size_t kPipeChunk = size_t(16) << 20;  // host-buffer pipeline: text bytes per chunk (16 MiB measured best: 8/16/32 MiB -> 41.6/43.6/40.5 GB/s e2e on one box)
inline bool is_ascii_space(unsigned char c) { return (c >= 0x09 && c <= 0x0D) || c == 0x20; }
inline bool is_ascii_punct(unsigned char c) {
  return (c >= 0x21 && c <= 0x2F) || (c >= 0x3A && c <= 0x40) || (c >= 0x5B && c <= 0x60) || (c >= 0x7B && c <= 0x7E);
}
inline bool is_cont(unsigned char c) { return (c & 0xC0) == 0x80; }

// Is byte offset c a SAFE CUT of the text: do [0, c) and [c, n) encode independently, so that their ids
// concatenate to the ids of the whole?  The reference's serial state is reset at every is_space code point
// (fast.cpp:89-91) and its own chunking cuts there (fast.cpp:113-115); SURVEY A.2 lists the other safe
// starts, which matter for space-free CJK text: a punctuation position, the position right after a
// punctuation char (a punctuation window is one char, fast.cpp:55), and a Han position.  Only byte patterns
// that are certain whatever surrounds them are accepted: ASCII bytes are always whole chars, E2 96 81 is
// always U+2581, and a lead E4 B8..BF / E5..E9 followed by two continuation bytes is always a Han char
// U+4E00..U+9FFF (lead bytes are always decode starts, utf8.cpp:130-147).
bool safe_cut(const unsigned char *t, size_t n, size_t c) {
  if (c == 0 || c >= n) return true;
  const unsigned char prev = t[c - 1], cur = t[c];
  if (is_ascii_space(prev) || is_ascii_punct(prev) || is_ascii_punct(cur)) return true;
  if (c >= 3 && t[c - 3] == 0xE2 && t[c - 2] == 0x96 && prev == 0x81) return true;  // after U+2581
  if (c + 2 < n && is_cont(t[c + 1]) && is_cont(t[c + 2])) {
    if (cur >= 0xE5 && cur <= 0xE9) return true;
    if (cur == 0xE4 && t[c + 1] >= 0xB8) return true;
  }
  return false;
}

// Cuts of [0, n) into k contiguous shards of near-equal size (BASELINE configs[3]): cut i is the first safe
// cut at or after n * i / k.  cuts[0] = 0, cuts[k] = n; shards may be empty when the text is tiny or has no
// safe cut for a long stretch.
void plan_shards(const unsigned char *t, size_t n, size_t k, size_t *cuts) {
  cuts[0] = 0;
  for (size_t i = 1; i < k; i++) {
    size_t c = static_cast<size_t>((static_cast<unsigned __int128>(n) * i) / k);
    if (c < cuts[i - 1]) c = cuts[i - 1];
    while (c < n && !safe_cut(t, n, c)) c++;
    cuts[i] = c;
  }
  cuts[k] = n;
}

// Cut [0, n) into chunks of at most kPipeChunk bytes, each ending at a safe cut (see safe_cut): the chunks
// encode independently and their ids concatenate.  Returns false if some stretch has no safe cut.
size_t pipe_chunk_bytes() {
  if (const char *e = std::getenv("WORDPIECE_B200_PIPE_CHUNK")) {  // test hook: pipeline small texts
    const long long x = std::atoll(e);
    if (x >= 64 && static_cast<size_t>(x) <= kPipeChunk) return static_cast<size_t>(x);
  }
  return kPipeChunk;
}

// The first chunks grow (chunk/8, /4, /2, then full) and the last ones shrink the same way: the pipeline's
// fill (copy-in + encode of the first chunk) and drain (encode + copy-out of the last) are the only parts
// of the call that do not overlap with a PCIe copy in the other direction.
bool plan_chunks(const char *text, size_t n, size_t chunk, std::vector<size_t> *cuts) {
  cuts->clear();
  cuts->push_back(0);
  size_t start = 0;
  const size_t small = chunk / 8 >= 64 ? chunk / 8 : chunk;
  for (size_t j = 0;; j++) {
    const size_t remaining = n - start;
    size_t want = j < 3 ? small << j : chunk;
    if (want > chunk) want = chunk;
    const size_t tail = remaining / 2 > small ? remaining / 2 : small;
    if (want > tail) want = tail;
    if (remaining <= want) break;
    size_t end = start + want;
    size_t cut = end;
    const size_t floor = start + want / 2;
    while (cut > floor && !safe_cut(reinterpret_cast<const unsigned char *>(text), n, cut)) cut--;
    if (cut <= floor) return false;
    cuts->push_back(cut);
    start = cut;
  }
  cuts->push_back(n);
  return true;
}

/* ------------------------------------------------------------------ the host pipeline (run_pipeline)
 * A batch is packed into one buffer, each text followed by one space: a space ends every word and resets the
 * matcher's state (fast.cpp:89-91), a byte sequence cut short at the end of a text stays invalid in front of
 * it, so the ids of the packed buffer are the ids of the texts one after the other.  K1 numbers the first
 * segment of every text, K5 turns the numbers into id offsets (wp_encode.h). */

constexpr size_t kBatchPart = size_t(8) << 20;  // packed bytes per part of a large batch

size_t batch_part_bytes() {
  if (const char *e = std::getenv("WORDPIECE_B200_BATCH_PART")) {  // test hook: pipeline small batches
    const long long x = std::atoll(e);
    if (x >= 256 && static_cast<size_t>(x) <= kBatchPart) return static_cast<size_t>(x);
  }
  return kBatchPart;
}

// One part of a pipelined call: a chunk of one text (wp_encode_into: no texts; only `packed` and `in_bytes`, the
// chunk's length, are set), or whole texts of a batch, whose input block is laid out as
// tile index | text starts | packed texts (16-byte aligned for K1's vector loads)
struct PartPlan {
  size_t first = 0, last = 0;  // texts [first, last)
  size_t packed = 0;           // bytes incl. one separator per text
  size_t n_tiles = 0, off_bounds = 0, off_text = 0, in_bytes = 0, off_offsets = 0, out_bytes = 0;
};

PartPlan plan_part(const size_t *lens, size_t first, size_t last) {
  PartPlan p;
  p.first = first;
  p.last = last;
  const size_t n = last - first;
  p.packed = n;
  for (size_t i = first; i < last; i++) p.packed += lens[i];
  const size_t tile = wp::encode_tile_bytes();
  p.n_tiles = (p.packed + tile - 1) / tile;
  p.off_bounds = align_up((p.n_tiles + 1) * sizeof(uint32_t), 256);
  p.off_text = align_up(p.off_bounds + n * sizeof(unsigned long long), 256);
  p.in_bytes = p.off_text + p.packed;
  p.off_offsets = align_up(n * sizeof(uint32_t), 256);
  p.out_bytes = p.off_offsets + (n + 1) * sizeof(unsigned long long);
  return p;
}

// texts -> the part's input block (text starts, tile index, the texts with their separators)
void pack_part(uint8_t *block, const PartPlan &p, const char *const *texts, const size_t *lens,
               bool streamed = stream_stores()) {
  const size_t n = p.last - p.first;
  uint32_t *tile_bound = reinterpret_cast<uint32_t *>(block);
  unsigned long long *bounds = reinterpret_cast<unsigned long long *>(block + p.off_bounds);
  char *text = reinterpret_cast<char *>(block + p.off_text);
  unsigned long long at = 0;
  for (size_t i = 0; i < n; i++) {
    bounds[i] = at;
    at += lens[p.first + i] + 1;
  }
  auto pack = [&](size_t part, size_t parts) {  // equal byte shares, whole texts
    const unsigned long long lo = static_cast<unsigned long long>(p.packed) * part / parts;
    const unsigned long long hi = static_cast<unsigned long long>(p.packed) * (part + 1) / parts;
    size_t i = static_cast<size_t>(std::lower_bound(bounds, bounds + n, lo) - bounds);
    const size_t end = part + 1 == parts ? n : static_cast<size_t>(std::lower_bound(bounds, bounds + n, hi) - bounds);
    if (streamed) {  // (the texts of a share are contiguous in the packed buffer)
      if (i >= end) return;
      StreamWriter w(text + bounds[i]);
      for (; i < end; i++) {
        w.put(texts[p.first + i], lens[p.first + i]);
        w.put(' ');
      }
      w.finish();
      return;
    }
    for (; i < end; i++) {
      char *dst = text + bounds[i];
      const size_t len = lens[p.first + i];
      if (len) std::memcpy(dst, texts[p.first + i], len);
      dst[len] = ' ';
    }
  };
  if (p.packed >= (size_t(1) << 20)) {
    CopyPool::get().run(pack);
  } else {
    pack(0, 1);
  }
  const size_t tile = wp::encode_tile_bytes();
  size_t i = 0;
  for (size_t t = 0; t <= p.n_tiles; t++) {  // tile_bound[t] = first text that starts at or after byte t * tile
    const unsigned long long lo = static_cast<unsigned long long>(t) * tile;
    while (i < n && bounds[i] < lo) i++;
    tile_bound[t] = static_cast<uint32_t>(i);
  }
}

constexpr int kSlots = 3;

// Room in slot sl for part p (`fill_pinned`: its input is staged in the slot's pinned memory; `stage_ids`: pinned
// id staging).  Before a buffer of a slot in use grows, the host waits until the slot's previous part has left it.
wp_status fit_slot(wp_vocab::Slot &sl, const PartPlan &p, bool fill_pinned, size_t stage_ids, bool in_use) {
  bool waited = !in_use;
  auto grow = [&](auto &buf, size_t want) -> cudaError_t {
    if (want > buf.cap && !waited) {
      waited = true;
      const cudaError_t e = cudaEventSynchronize(sl.d2h_done);
      if (e != cudaSuccess) return e;
    }
    return buf.grow(want);
  };
  WP_CUDA(grow(sl.h_in, fill_pinned ? p.in_bytes : 0));
  WP_CUDA(grow(sl.d_in, p.in_bytes));
  WP_CUDA(grow(sl.d_ids, p.packed));  // one id per byte is the worst case
  WP_CUDA(grow(sl.d_out, p.out_bytes));
  WP_CUDA(grow(sl.h_offsets, p.last > p.first ? p.last - p.first + 1 : 0));  // (a batch part's texts + 1)
  WP_CUDA(grow(sl.h_ids, stage_ids));
  WP_CUDA(grow(sl.h_call, 1));
  for (Event *e : {&sl.h2d_done, &sl.cmp_done, &sl.d2h_done})
    if (!e->h) WP_CUDA(cudaEventCreateWithFlags(&e->h, cudaEventDisableTiming));
  trace("part: buffers ready");
  return WP_OK;
}

// Enqueue part p in slot sl: the H2D copy of its input block from host memory `src` on `copy_stream`, then on
// v->stream the kernels, for a batch part its id offsets and their copy to sl.h_offsets, and the copy of the
// counters to sl.h_call.
wp_status enqueue_part(wp_vocab *v, wp_vocab::Slot &sl, const PartPlan &p, const void *src, cudaStream_t copy_stream,
                       size_t spill, bool warm, size_t call_bytes, EnqueueInfo *info) {
  const size_t n = p.last - p.first;  // texts (none: a chunk of one text)
  WP_CUDA(cudaMemcpyAsync(sl.d_in.p, src, p.in_bytes, cudaMemcpyHostToDevice, copy_stream));
  WP_CUDA(trace_stage(copy_stream, "part:   [stage] input block on the device"));
  WP_CUDA(cudaEventRecord(sl.h2d_done, copy_stream));
  WP_CUDA(cudaStreamWaitEvent(v->stream, sl.h2d_done, 0));
  BatchArgs batch;
  batch.h_bounds = reinterpret_cast<const unsigned long long *>(static_cast<const uint8_t *>(src) + p.off_bounds);
  batch.n_texts = n;
  batch.d_tile_bound = reinterpret_cast<const uint32_t *>(sl.d_in.p);
  batch.d_bounds = reinterpret_cast<const unsigned long long *>(sl.d_in.p + p.off_bounds);
  batch.d_bound_seg = reinterpret_cast<uint32_t *>(sl.d_out.p);
  batch.d_offsets = reinterpret_cast<unsigned long long *>(sl.d_out.p + p.off_offsets);
  const wp_status st = enqueue_encode(v, sl.d_in.p + p.off_text, p.packed, sl.d_ids.p, sl.d_ids.cap, v->stream, spill,
                                      info, warm, call_bytes, n ? &batch : nullptr);
  if (st != WP_OK) return st;
  WP_CUDA(trace_stage(v->stream, "part:   [stage] kernels done"));
  if (n) {
    uint64_t launches = 0;
    WP_CUDA(wp::launch_publish_count(v->d_call.p, info->n_ranges & 1u, batch.d_offsets + n, v->stream, &launches));
    WP_CUDA(cudaEventRecord(v->last_done, v->stream));
    g_launches.fetch_add(launches, std::memory_order_relaxed);
    info->launches += launches;
    WP_CUDA(cudaMemcpyAsync(sl.h_offsets.p, batch.d_offsets, (n + 1) * sizeof(unsigned long long),
                            cudaMemcpyDeviceToHost, v->stream));
  }
  WP_CUDA(cudaMemcpyAsync(sl.h_call.p, v->d_call.p, sizeof(wp::CallCounters), cudaMemcpyDeviceToHost, v->stream));
  WP_CUDA(cudaEventRecord(sl.cmp_done, v->stream));
  trace("part: enqueued");
  return WP_OK;
}

// The parts of one call (wp_encode_into: text chunks, wp_encode_batch: whole texts) into ids[0, capacity) through
// three slots: while part k is encoded, part k+1 is filled and copied in and the ids of part k-1 are copied out
// (the PCIe copies, not the kernels, bound these calls).  fill(k, slot) returns the host address of part k's input
// block (`fill_pinned`: it writes it to the slot's pinned input); done(k, slot, first_id) takes what a finished
// part adds besides its ids.  `stage_out`: ids go to the pageable caller through pinned staging and the CopyPool.
// A void part ends the call with *repeat set: the caller repeats the whole call, the first time with *spill.
template <class Fill, class Done>
wp_status run_pipeline(wp_vocab *v, const std::vector<PartPlan> &parts, size_t call_bytes, bool fill_pinned,
                       bool stage_out, int32_t *ids, size_t capacity, Fill &&fill, Done &&done,
                       size_t *n_ids, bool *repeat, size_t *spill) {
  CopyPool &pool = CopyPool::get();
  const size_t n_parts = parts.size();
  // ids per pinned staging slot (32 MiB at the default chunk size; a chunk of ordinary text has a quarter of that)
  const size_t stage_ids = stage_out ? pipe_chunk_bytes() / 2 : 0;
  std::vector<EnqueueInfo> infos(n_parts);
  std::vector<size_t> first_id(n_parts, 0), staged(n_parts, 0);
  size_t total = 0;
  wp_stats acc{};
  *repeat = false;

  // part j's kernels are done: absorb its counters, start the copy of its ids device -> host
  auto finish = [&](size_t j) -> wp_status {
    wp_vocab::Slot &sl = v->slot[j % kSlots];
    WP_CUDA(cudaEventSynchronize(sl.cmp_done));
    *repeat = absorb_call(v, *sl.h_call.p, infos[j], call_bytes, &acc, spill);
    if (*repeat) return WP_OK;
    const size_t cnt = static_cast<size_t>(sl.h_call.p->ids_total[infos[j].n_ranges & 1u]);
    done(j, sl, total);
    first_id[j] = total;
    if (cnt > 0 && total + cnt <= capacity) {
      WP_CUDA(cudaStreamWaitEvent(v->s_d2h, sl.cmp_done, 0));
      if (!stage_out) {
        WP_CUDA(cudaMemcpyAsync(ids + total, sl.d_ids.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost, v->s_d2h));
      } else if (cnt <= sl.h_ids.cap) {
        WP_CUDA(cudaMemcpyAsync(sl.h_ids.p, sl.d_ids.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost, v->s_d2h));
        staged[j] = cnt;
      } else {
        // more ids than the staging slot holds (text of one- and two-byte tokens): piece by piece, synchronously
        for (size_t at = 0; at < cnt; at += sl.h_ids.cap) {
          const size_t piece = std::min(cnt - at, sl.h_ids.cap);
          WP_CUDA(cudaMemcpyAsync(sl.h_ids.p, sl.d_ids.p + at, piece * sizeof(int32_t), cudaMemcpyDeviceToHost,
                                  v->s_d2h));
          WP_CUDA(cudaStreamSynchronize(v->s_d2h));
          pool.copy(ids + total + at, sl.h_ids.p, piece * sizeof(int32_t));
        }
      }
    }
    WP_CUDA(cudaEventRecord(sl.d2h_done, v->s_d2h));
    WP_CUDA(trace_stage(v->s_d2h, "part:   [stage] ids on the host"));
    total += cnt;
    return WP_OK;
  };
  // part j's staged ids have arrived in its slot: hand them to the caller
  auto deliver = [&](size_t j) -> wp_status {
    if (staged[j] == 0) return WP_OK;
    wp_vocab::Slot &sl = v->slot[j % kSlots];
    WP_CUDA(cudaEventSynchronize(sl.d2h_done));
    pool.copy(ids + first_id[j], sl.h_ids.p, staged[j] * sizeof(int32_t));
    return WP_OK;
  };

  // (two more rounds than parts drain the pipeline: the last part is finished, then its staged ids delivered)
  for (size_t k = 0; k < n_parts + 2 && !*repeat; k++) {
    wp_status st;
    if (k < n_parts) {
      wp_vocab::Slot &sl = v->slot[k % kSlots];
      const bool reused = k >= kSlots;  // the slot holds part k-3
      if (reused) {  // its ids must have left before the device reuses its buffers, its input before the host does
        WP_CUDA(cudaStreamWaitEvent(v->s_h2d, sl.d2h_done, 0));
        WP_CUDA(cudaStreamWaitEvent(v->stream, sl.d2h_done, 0));
        if (fill_pinned) WP_CUDA(cudaEventSynchronize(sl.h2d_done));
      }
      st = fit_slot(sl, parts[k], fill_pinned, stage_ids, reused);
      if (st != WP_OK) return st;
      st = enqueue_part(v, sl, parts[k], fill(k, sl), v->s_h2d, 0, /*warm=*/k != 0, call_bytes, &infos[k]);
      if (st != WP_OK) return st;
    }
    if (k >= 2) {  // (before the slot of part k-2 is reused by part k+1; its D2H was started a round ago)
      st = deliver(k - 2);
      if (st != WP_OK) return st;
    }
    if (k >= 1 && k <= n_parts) {
      st = finish(k - 1);
      if (st != WP_OK) return st;
      trace("part: previous part finished (ids on their way out)");
    }
  }
  WP_CUDA(cudaStreamSynchronize(v->s_d2h));
  WP_CUDA(cudaStreamSynchronize(v->stream));  // (idle unless a void part left later parts in flight)
  if (*repeat) return WP_OK;
  v->stats = acc;
  v->stats.n_bytes = call_bytes;
  v->stats.n_ids = total;
  *n_ids = total;
  return WP_OK;
}

wp_status create_common(wp_vocab *v, const char *const *tokens, const size_t *lens, size_t n, int device,
                        wp_vocab **out) {
  std::string err;
  trace("vocabulary: build tables (host)");
  if (!wp::build_host_vocab(tokens, lens, n, &v->host, &err)) {
    delete v;
    return fail(WP_ERR_EMPTY_VOCAB_WORD, err);
  }
  if (device == -1) {  // host-only handle: vocabulary queries and decode work, every encode call fails
    v->device = -1;
    *out = v;
    return WP_OK;
  }
  int count = 0;
  trace("vocabulary: tables built; first CUDA call");
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
    delete v;
    return fail(WP_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU path)");
  }
  if (device < 0 || device >= count) {
    delete v;
    return fail(WP_ERR_INVALID_ARG, "device ordinal out of range");
  }
  v->device = device;
  DeviceGuard g(device);
  if (!g.ok) {
    delete v;
    return fail(WP_ERR_CUDA, "cudaSetDevice failed");
  }
  trace("vocabulary: device selected; upload");
  wp_status st = upload(v);
  trace("vocabulary: on the device");
  if (st != WP_OK) {
    std::string keep = g_error;
    wp_vocab_destroy(v);
    g_error = keep;
    return st;
  }
  *out = v;
  return WP_OK;
}

}  // namespace

extern "C" {

const char *wp_last_error(void) { return g_error.c_str(); }

uint64_t wp_kernel_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

uint32_t wp_tile_bytes(void) { return wp::encode_tile_bytes(); }

void wp_free(void *p) { std::free(p); }

wp_status wp_vocab_create(const char *const *tokens, const size_t *token_lens, size_t n_tokens, int device,
                          wp_vocab **out) {
  if (out == nullptr || (n_tokens > 0 && (tokens == nullptr || token_lens == nullptr)))
    return fail(WP_ERR_INVALID_ARG, "null argument");
  if (n_tokens >= (size_t(1) << 30) - 1) return fail(WP_ERR_INVALID_ARG, "vocabulary too large (ids must fit 30 bits)");
  *out = nullptr;
  wp_vocab *v = new (std::nothrow) wp_vocab();
  if (!v) return fail(WP_ERR_NOMEM, "out of memory");
  return create_common(v, tokens, token_lens, n_tokens, device, out);
}

wp_status wp_vocab_create_from_file(const char *vocab_file, int device, wp_vocab **out) {
  if (out == nullptr || vocab_file == nullptr) return fail(WP_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  std::ifstream fin(vocab_file, std::ios::binary);
  // utils.cpp:123-137 never checks the stream: an unreadable file is an empty vocabulary there.
  // We report it, since silently encoding everything to UNK helps nobody.
  if (!fin) return fail(WP_ERR_IO, std::string("cannot open vocab file: ") + vocab_file);
  std::vector<std::string> lines;
  std::string line;
  while (std::getline(fin, line)) lines.push_back(line);  // '\r' stays, as with the reference's getline
  std::vector<const char *> ptrs(lines.size());
  std::vector<size_t> lens(lines.size());
  for (size_t i = 0; i < lines.size(); i++) {
    ptrs[i] = lines[i].data();
    lens[i] = lines[i].size();
  }
  wp_vocab *v = new (std::nothrow) wp_vocab();
  if (!v) return fail(WP_ERR_NOMEM, "out of memory");
  return create_common(v, ptrs.data(), lens.data(), lines.size(), device, out);
}

void wp_vocab_destroy(wp_vocab *v) {
  std::optional<DeviceGuard> g;  // (a host-only handle owns no CUDA resource: its teardown makes no CUDA call)
  if (v && v->device >= 0) {
    g.emplace(v->device);
    if (v->stream) cudaStreamSynchronize(v->stream);
  }
  delete v;  // (the owners free their memory, events and streams on the handle's device)
}

size_t wp_vocab_size(const wp_vocab *v) { return v ? v->host.tokens.size() : 0; }
int32_t wp_vocab_unk_id(const wp_vocab *v) { return v ? v->host.unk_id : -1; }
size_t wp_vocab_max_len(const wp_vocab *v) { return v ? v->host.max_len : 0; }
int wp_vocab_device(const wp_vocab *v) { return v ? v->device : -1; }
size_t wp_vocab_device_bytes(const wp_vocab *v) { return v ? v->device_bytes : 0; }

int wp_vocab_token_flags(const wp_vocab *v, size_t index) {
  if (!v || index >= v->host.tokens.size()) return -1;
  const wp::HostToken &t = v->host.tokens[index];
  return (t.is_prefix ? 1 : 0) | (t.is_special ? 2 : 0) | (t.is_malformed ? 4 : 0) | (t.had_invalid ? 8 : 0);
}

wp_status wp_encode_device_async(wp_vocab *v, const void *d_text, size_t n_bytes, int32_t *d_ids, size_t capacity,
                                 uint64_t *d_n_ids, void *stream) {
  if (!v || (n_bytes > 0 && d_text == nullptr) || (capacity > 0 && d_ids == nullptr))
    return fail(WP_ERR_INVALID_ARG, "null argument");
  if (v->device < 0) return fail(WP_ERR_NO_DEVICE, kHostOnly);
  DeviceGuard g(v->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);  // NULL = the default stream, as everywhere in CUDA
  if (n_bytes == 0) {  // fast.cpp:145
    if (d_n_ids) WP_CUDA(cudaMemsetAsync(d_n_ids, 0, sizeof(uint64_t), s));
    return WP_OK;
  }
  EnqueueInfo info;
  wp_status st = enqueue_encode(v, d_text, n_bytes, d_ids, capacity, s, 0, &info);
  if (st != WP_OK) return st;
  if (d_n_ids) {
    uint64_t launches = 0;
    WP_CUDA(wp::launch_publish_count(v->d_call.p, info.n_ranges & 1u, reinterpret_cast<unsigned long long *>(d_n_ids), s,
                                     &launches));
    WP_CUDA(cudaEventRecord(v->last_done, s));  // the count reads the counters the next call clears
    g_launches.fetch_add(launches, std::memory_order_relaxed);
  }
  return WP_OK;
}

wp_status wp_encode_device(wp_vocab *v, const void *d_text, size_t n_bytes, int32_t *d_ids, size_t capacity,
                           size_t *n_ids, void *stream) {
  if (!v || n_ids == nullptr || (n_bytes > 0 && d_text == nullptr) || (capacity > 0 && d_ids == nullptr))
    return fail(WP_ERR_INVALID_ARG, "null argument");
  *n_ids = 0;
  if (v->device < 0) return fail(WP_ERR_NO_DEVICE, kHostOnly);
  DeviceGuard g(v->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);  // NULL = the default stream, as everywhere in CUDA
  if (n_bytes == 0) {
    v->stats = wp_stats{};
    return WP_OK;
  }
  wp_status st = run_encode(v, d_text, n_bytes, d_ids, capacity, s);
  if (st != WP_OK) return st;
  *n_ids = static_cast<size_t>(v->stats.n_ids);
  if (v->stats.n_ids > capacity) return fail(WP_ERR_CAPACITY, "id buffer too small");
  return WP_OK;
}

wp_status wp_encode_into(wp_vocab *v, const char *text, size_t n_bytes, int32_t *ids, size_t capacity,
                         size_t *n_ids) {
  if (!v || n_ids == nullptr || (n_bytes > 0 && text == nullptr)) return fail(WP_ERR_INVALID_ARG, "null argument");
  *n_ids = 0;
  if (v->device < 0) return fail(WP_ERR_NO_DEVICE, kHostOnly);
  if (n_bytes == 0) {
    v->stats = wp_stats{};
    return WP_OK;
  }
  DeviceGuard g(v->device);
  trace("wp_encode_into: begin");
  size_t spill = 0;
  bool repeat = true;
  std::vector<size_t> cuts;
  if (n_bytes > 2 * pipe_chunk_bytes() && plan_chunks(text, n_bytes, pipe_chunk_bytes(), &cuts)) {
    // Pageable caller memory (the reference's own signature hands over a std::string and expects a std::vector)
    // is staged through the slots' pinned memory by the CopyPool
    std::vector<PartPlan> chunks(cuts.size() - 1);
    for (size_t k = 0; k < chunks.size(); k++) chunks[k].packed = chunks[k].in_bytes = cuts[k + 1] - cuts[k];
    const bool stage_in = is_pageable(text);
    const wp_status st = run_pipeline(
        v, chunks, n_bytes, stage_in, capacity > 0 && is_pageable(ids), ids, capacity,
        [&](size_t k, wp_vocab::Slot &sl) -> const void * {
          if (!stage_in) return text + cuts[k];
          CopyPool::get().copy(sl.h_in.p, text + cuts[k], chunks[k].packed, /*streamed=*/true);
          return sl.h_in.p;
        },
        [](size_t, wp_vocab::Slot &, size_t) {}, n_ids, &repeat, &spill);
    if (st != WP_OK) return st;
  }
  // Void pipelined ids: the whole text once more in one call (through the pipeline, a single part would need
  // pinned id staging as large as the text).  One id per byte is the worst case (a run of single-byte tokens):
  // the id buffer holds what the caller can take, bounded by that.
  if (repeat) {
    const size_t want = capacity < n_bytes ? capacity : n_bytes;
    const wp_status st = encode_staged(v, text, n_bytes, want ? want : 1, /*retry_short=*/false, spill);
    if (st != WP_OK) return st;
    *n_ids = static_cast<size_t>(v->stats.n_ids);
    trace("wp_encode_into: ids on the device");
    if (*n_ids > 0 && *n_ids <= capacity) {
      WP_CUDA(cudaMemcpyAsync(ids, v->d_ids.p, *n_ids * sizeof(int32_t), cudaMemcpyDeviceToHost, v->stream));
      WP_CUDA(cudaStreamSynchronize(v->stream));
      trace("wp_encode_into: ids on the host");
    }
  }
  return *n_ids > capacity ? fail(WP_ERR_CAPACITY, "id buffer too small") : WP_OK;
}

// Host text -> ids in the handle's device buffer v->d_ids (count in v->stats.n_ids).  First guess: half an id per
// byte (English-like text needs ~0.25); exact retry if short.
static wp_status encode_to_device_buffer(wp_vocab *v, const char *text, size_t n_bytes) {
  return encode_staged(v, text, n_bytes, std::min(n_bytes, n_bytes / 2 + 1024), /*retry_short=*/true);
}

// n bytes of device memory -> a new malloc block of n + extra bytes (at least one), for the caller to free
static wp_status download(wp_vocab *v, const void *d_src, size_t n, size_t extra, const char *what, void **out) {
  void *host = std::malloc(n + extra ? n + extra : 1);
  if (!host) return fail(WP_ERR_NOMEM, "out of memory");
  if (n > 0) {
    cudaError_t e = cudaMemcpyAsync(host, d_src, n, cudaMemcpyDeviceToHost, v->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(v->stream);
    if (e != cudaSuccess) {
      std::free(host);
      return fail(WP_ERR_CUDA, std::string(what) + cudaGetErrorString(e));
    }
  }
  *out = host;
  return WP_OK;
}

wp_status wp_encode(wp_vocab *v, const char *text, size_t n_bytes, int32_t **ids_out, size_t *n_ids) {
  if (!v || ids_out == nullptr || n_ids == nullptr || (n_bytes > 0 && text == nullptr))
    return fail(WP_ERR_INVALID_ARG, "null argument");
  *ids_out = nullptr;
  *n_ids = 0;
  if (v->device < 0) return fail(WP_ERR_NO_DEVICE, kHostOnly);
  if (n_bytes == 0) {
    v->stats = wp_stats{};
    return WP_OK;
  }
  DeviceGuard g(v->device);
  trace("wp_encode: begin");
  const wp_status st = encode_to_device_buffer(v, text, n_bytes);
  if (st != WP_OK) return st;
  trace("wp_encode: ids on the device");
  const size_t cnt = static_cast<size_t>(v->stats.n_ids);
  void *host = nullptr;
  const wp_status dst = download(v, v->d_ids.p, cnt * sizeof(int32_t), 0, "copy ids: ", &host);
  if (dst != WP_OK) return dst;
  *ids_out = static_cast<int32_t *>(host);
  *n_ids = cnt;
  return WP_OK;
}

wp_status wp_encode_batch(wp_vocab *v, const char *const *texts, const size_t *lens, size_t n_texts, int32_t *ids,
                          size_t capacity, size_t *offsets, size_t *n_ids) {
  if (!v || !n_ids || !offsets || (n_texts > 0 && (!texts || !lens)) || (capacity > 0 && !ids))
    return fail(WP_ERR_INVALID_ARG, "null argument");
  *n_ids = 0;
  offsets[0] = 0;
  if (v->device < 0) return fail(WP_ERR_NO_DEVICE, kHostOnly);
  if (n_texts == 0) {
    v->stats = wp_stats{};
    return WP_OK;
  }
  if (n_texts >= (size_t(1) << 31)) return fail(WP_ERR_INVALID_ARG, "too many texts in one batch (>= 2^31)");
  size_t packed = n_texts;  // one separator per text
  for (size_t i = 0; i < n_texts; i++) {
    if (lens[i] > 0 && !texts[i]) return fail(WP_ERR_INVALID_ARG, "null text");
    if (packed + lens[i] < packed) return fail(WP_ERR_INVALID_ARG, "batch too large");
    packed += lens[i];
  }
  DeviceGuard g(v->device);
  trace("wp_encode_batch: begin");
  // a large batch: parts of whole texts, about kBatchPart packed bytes each
  std::vector<PartPlan> parts;
  const size_t part_bytes = batch_part_bytes();
  for (size_t i = 0, first = 0, bytes = 0; packed > 3 * part_bytes / 2 && i < n_texts; i++) {
    bytes += lens[i] + 1;
    if (bytes >= part_bytes || i + 1 == n_texts) {
      parts.push_back(plan_part(lens, first, i + 1));
      first = i + 1;
      bytes = 0;
    }
  }
  static_assert(sizeof(size_t) == sizeof(unsigned long long), "offsets are copied as they are");
  auto fill = [&](size_t k, wp_vocab::Slot &sl) -> const void * {
    pack_part(sl.h_in.p, parts[k], texts, lens);
    trace("wp_encode_batch: part packed");
    return sl.h_in.p;
  };
  auto rebase = [&](size_t k, const wp_vocab::Slot &sl, size_t first_id) {  // part k's offsets
    const PartPlan &p = parts[k];
    for (size_t i = p.first; i < p.last; i++) offsets[i] = first_id + static_cast<size_t>(sl.h_offsets.p[i - p.first]);
  };
  size_t spill = 0;
  bool repeat = true;  // (a small batch goes as one part)
  if (parts.size() > 1) {
    const wp_status st = run_pipeline(v, parts, packed, /*fill_pinned=*/true, /*stage_out=*/false, ids, capacity,
                                      fill, rebase, n_ids, &repeat, &spill);
    if (st != WP_OK) return st;
  }
  if (repeat) {  // the whole batch as one part: a small batch, or a pipelined one whose ids are void
    parts.assign(1, plan_part(lens, 0, n_texts));
    const PartPlan &whole = parts[0];
    wp_vocab::Slot &sl = v->slot[0];
    wp_status st = fit_slot(sl, whole, /*fill_pinned=*/true, 0, /*in_use=*/false);
    if (st != WP_OK) return st;
    const void *src = fill(0, sl);
    st = repeat_call(v, v->stream, packed, spill, *sl.h_call.p, [&](size_t sp, EnqueueInfo *info) {
      return enqueue_part(v, sl, whole, src, v->stream, sp, /*warm=*/false, packed, info);
    });
    if (st != WP_OK) return st;
    *n_ids = static_cast<size_t>(v->stats.n_ids);
    rebase(0, sl, 0);
    if (*n_ids > 0 && *n_ids <= capacity)
      WP_CUDA(cudaMemcpyAsync(ids, sl.d_ids.p, *n_ids * sizeof(int32_t), cudaMemcpyDeviceToHost, v->stream));
    WP_CUDA(cudaStreamSynchronize(v->stream));
  }
  trace("wp_encode_batch: ids on the host");
  offsets[n_texts] = *n_ids;
  return *n_ids > capacity ? fail(WP_ERR_CAPACITY, "id buffer too small") : WP_OK;
}

// Host-side checks shared by both device batch entry points; *packed <- n_chars + n_texts
static wp_status check_batch_device(wp_vocab *v, const void *d_chars, size_t n_chars, const uint64_t *d_offsets,
                                    size_t n_texts, int32_t *d_ids, size_t capacity, uint64_t *d_id_offsets,
                                    size_t *packed) {
  if (!v || !d_offsets || !d_id_offsets || (n_chars > 0 && !d_chars) || (capacity > 0 && !d_ids))
    return fail(WP_ERR_INVALID_ARG, "null argument");
  if (v->device < 0) return fail(WP_ERR_NO_DEVICE, kHostOnly);
  if (n_texts >= (size_t(1) << 31)) return fail(WP_ERR_INVALID_ARG, "too many texts in one batch (>= 2^31)");
  *packed = n_chars + n_texts;
  if (*packed < n_chars || *packed / wp::encode_tile_bytes() >= 0x7FFFFFFFull)
    return fail(WP_ERR_INVALID_ARG, "batch too large for one call (> 2^31 tiles)");
  return WP_OK;
}

wp_status wp_encode_batch_device_async(wp_vocab *v, const void *d_chars, size_t n_chars, const uint64_t *d_offsets,
                                       size_t n_texts, int32_t *d_ids, size_t capacity, uint64_t *d_id_offsets,
                                       void *stream) {
  size_t packed = 0;
  wp_status st = check_batch_device(v, d_chars, n_chars, d_offsets, n_texts, d_ids, capacity, d_id_offsets, &packed);
  if (st != WP_OK) return st;
  DeviceGuard g(v->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);  // NULL = the default stream, as everywhere in CUDA
  if (n_texts == 0) {
    WP_CUDA(cudaMemsetAsync(d_id_offsets, 0, sizeof(uint64_t), s));
    return WP_OK;
  }
  uint64_t launches = 0;
  st = enqueue_column(v, d_chars, n_chars, d_offsets, n_texts, packed, s, &launches);
  if (st != WP_OK) return st;
  EnqueueInfo info;
  return enqueue_column_encode(v, packed, n_texts, d_ids, capacity, d_id_offsets, s, 0, &info);
}

wp_status wp_encode_batch_device(wp_vocab *v, const void *d_chars, size_t n_chars, const uint64_t *d_offsets,
                                 size_t n_texts, int32_t *d_ids, size_t capacity, uint64_t *d_id_offsets, size_t *n_ids,
                                 void *stream) {
  if (!n_ids) return fail(WP_ERR_INVALID_ARG, "null argument");
  *n_ids = 0;
  size_t packed = 0;
  wp_status st = check_batch_device(v, d_chars, n_chars, d_offsets, n_texts, d_ids, capacity, d_id_offsets, &packed);
  if (st != WP_OK) return st;
  DeviceGuard g(v->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (n_texts == 0) {
    v->stats = wp_stats{};
    WP_CUDA(cudaMemsetAsync(d_id_offsets, 0, sizeof(uint64_t), s));
    WP_CUDA(cudaStreamSynchronize(s));
    return WP_OK;
  }
  WP_CUDA(v->h_col_bad.grow(1));
  uint64_t launches = 0;  // (the check and the packer count with the first attempt: a repeat packs nothing again)
  st = enqueue_column(v, d_chars, n_chars, d_offsets, n_texts, packed, s, &launches);
  if (st != WP_OK) return st;
  st = repeat_call(v, s, packed, 0, *v->h_call.p, [&](size_t sp, EnqueueInfo *info) -> wp_status {
    const wp_status est = enqueue_column_encode(v, packed, n_texts, d_ids, capacity, d_id_offsets, s, sp, info);
    if (est != WP_OK) return est;
    info->launches += std::exchange(launches, 0);
    WP_CUDA(cudaMemcpyAsync(v->h_call.p, v->d_call.p, sizeof(wp::CallCounters), cudaMemcpyDeviceToHost, s));
    WP_CUDA(cudaMemcpyAsync(v->h_col_bad.p, v->d_col_bad.p, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
    return WP_OK;
  });
  if (st != WP_OK) return st;
  if (*v->h_col_bad.p)
    return fail(WP_ERR_INVALID_ARG, "malformed column: the offsets must ascend and end at most at n_chars");
  *n_ids = static_cast<size_t>(v->stats.n_ids);
  return *n_ids > capacity ? fail(WP_ERR_CAPACITY, "id buffer too small") : WP_OK;
}

size_t wp_next_safe_cut(const char *text, size_t n_bytes, size_t pos) {
  if (!text) return n_bytes;
  const unsigned char *t = reinterpret_cast<const unsigned char *>(text);
  while (pos < n_bytes && !safe_cut(t, n_bytes, pos)) pos++;
  return pos < n_bytes ? pos : n_bytes;
}

size_t wp_plan_shards(const char *text, size_t n_bytes, size_t n_shards, size_t *cuts) {
  if (!cuts || n_shards == 0 || (n_bytes > 0 && !text)) return 0;
  plan_shards(reinterpret_cast<const unsigned char *>(text), n_bytes, n_shards, cuts);
  return n_shards + 1;
}

// Shared body of wp_encode_sharded / wp_encode_sharded_gather.  Phase 1: one host thread per handle copies
// its shard in and encodes it, ids staying on that device.  Host: exclusive scan of the counts.  Phase 2: one
// host thread per handle copies its ids to their global offset — into the caller's host array, or peer to
// peer into device memory of the gathering handle.
static wp_status encode_sharded(wp_vocab *const *handles, size_t n, const char *text, size_t n_bytes, int32_t *h_ids,
                                int32_t *d_gather, int gather_device, size_t capacity, size_t *n_ids, wp_shard *shards,
                                float *copy_ms) {
  if (!handles || n == 0 || !n_ids || (n_bytes > 0 && !text)) return fail(WP_ERR_INVALID_ARG, "null argument");
  for (size_t i = 0; i < n; i++) {
    if (!handles[i]) return fail(WP_ERR_INVALID_ARG, "null handle");
    if (handles[i]->device < 0) return fail(WP_ERR_NO_DEVICE, kHostOnly);
    for (size_t j = 0; j < i; j++)
      if (handles[j] == handles[i]) return fail(WP_ERR_INVALID_ARG, "the same handle appears twice");
  }
  *n_ids = 0;
  std::vector<size_t> cuts(n + 1);
  plan_shards(reinterpret_cast<const unsigned char *>(text), n_bytes, n, cuts.data());
  std::vector<wp_shard> info(n);
  std::vector<wp_status> status(n, WP_OK);
  std::vector<std::string> errors(n);
  auto run = [&](auto &&body) {
    std::vector<std::thread> threads;
    for (size_t i = 1; i < n; i++) threads.emplace_back([&, i] {
      status[i] = body(i);
      if (status[i] != WP_OK) errors[i] = g_error;
    });
    status[0] = body(0);
    if (status[0] != WP_OK) errors[0] = g_error;
    for (auto &t : threads) t.join();
    for (size_t i = 0; i < n; i++)
      if (status[i] != WP_OK) return fail(status[i], "shard " + std::to_string(i) + ": " + errors[i]);
    return WP_OK;
  };
  wp_status st = run([&](size_t i) -> wp_status {
    wp_vocab *v = handles[i];
    info[i] = wp_shard{};
    info[i].begin = cuts[i];
    info[i].end = cuts[i + 1];
    info[i].device = v->device;
    const size_t len = cuts[i + 1] - cuts[i];
    if (len == 0) return WP_OK;  // fast.cpp:145
    DeviceGuard g(v->device);
    if (!g.ok) return fail(WP_ERR_CUDA, "cudaSetDevice failed");
    const auto t0 = std::chrono::steady_clock::now();
    const wp_status s1 = encode_to_device_buffer(v, text + cuts[i], len);
    if (s1 != WP_OK) return s1;
    info[i].n_ids = v->stats.n_ids;
    info[i].encode_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return WP_OK;
  });
  if (st != WP_OK) return st;
  uint64_t total = 0;
  for (size_t i = 0; i < n; i++) {  // host-side exclusive scan: the only "exchange" of the sharded path
    info[i].id_offset = total;
    total += info[i].n_ids;
  }
  *n_ids = static_cast<size_t>(total);
  if (shards) std::memcpy(shards, info.data(), n * sizeof(wp_shard));
  if (total > capacity) return fail(WP_ERR_CAPACITY, "id buffer too small");
  const auto t0 = std::chrono::steady_clock::now();
  st = run([&](size_t i) -> wp_status {
    wp_vocab *v = handles[i];
    const size_t cnt = static_cast<size_t>(info[i].n_ids);
    if (cnt == 0) return WP_OK;
    DeviceGuard g(v->device);
    if (!g.ok) return fail(WP_ERR_CUDA, "cudaSetDevice failed");
    if (d_gather) {
      if (v->device != gather_device) {
        cudaDeviceEnablePeerAccess(gather_device, 0);  // best effort: without it the copy is staged through the host
        cudaGetLastError();
        WP_CUDA(cudaMemcpyPeerAsync(d_gather + info[i].id_offset, gather_device, v->d_ids.p, v->device,
                                    cnt * sizeof(int32_t), v->stream));
      } else {
        WP_CUDA(cudaMemcpyAsync(d_gather + info[i].id_offset, v->d_ids.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToDevice,
                                v->stream));
      }
    } else {
      WP_CUDA(cudaMemcpyAsync(h_ids + info[i].id_offset, v->d_ids.p, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost,
                              v->stream));
    }
    WP_CUDA(cudaStreamSynchronize(v->stream));
    return WP_OK;
  });
  if (copy_ms) *copy_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return st;
}

wp_status wp_encode_sharded(wp_vocab *const *handles, size_t n_handles, const char *text, size_t n_bytes, int32_t *ids,
                            size_t capacity, size_t *n_ids, wp_shard *shards) {
  if (capacity > 0 && !ids) return fail(WP_ERR_INVALID_ARG, "null argument");
  return encode_sharded(handles, n_handles, text, n_bytes, ids, nullptr, -1, capacity, n_ids, shards, nullptr);
}

wp_status wp_encode_sharded_gather(wp_vocab *const *handles, size_t n_handles, const char *text, size_t n_bytes,
                                   size_t gather_index, int32_t *d_ids, size_t capacity, size_t *n_ids, wp_shard *shards,
                                   float *gather_ms) {
  if (!handles || gather_index >= n_handles || !handles[gather_index] || (capacity > 0 && !d_ids))
    return fail(WP_ERR_INVALID_ARG, "bad gather target");
  return encode_sharded(handles, n_handles, text, n_bytes, nullptr, d_ids, handles[gather_index]->device, capacity,
                        n_ids, shards, gather_ms);
}

wp_status wp_encode_text(wp_vocab *v, const char *text, size_t n_bytes, char **out, size_t *out_len, size_t *n_ids) {
  if (!v || out == nullptr || out_len == nullptr || n_ids == nullptr || (n_bytes > 0 && text == nullptr))
    return fail(WP_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  *out_len = 0;
  *n_ids = 0;
  if (v->device < 0) return fail(WP_ERR_NO_DEVICE, kHostOnly);
  DeviceGuard g(v->device);
  v->stats = wp_stats{};
  wp_status st = n_bytes ? encode_to_device_buffer(v, text, n_bytes) : WP_OK;  // (no text: "", as fast.cpp:145)
  if (st != WP_OK) return st;
  const size_t cnt = static_cast<size_t>(v->stats.n_ids);
  unsigned long long total = 0;
  if (cnt > 0) {
    // the encode scratch is idle now: [0] total length, [1] ticket, then one look-back word per block
    const size_t n_blocks = (cnt + wp::format_block_ids() - 1) / wp::format_block_ids();
    const size_t need = (2 + n_blocks) * sizeof(unsigned long long);
    WP_CUDA(v->d_work.grow(need));
    unsigned long long *w = reinterpret_cast<unsigned long long *>(v->d_work.p);
    WP_CUDA(cudaMemsetAsync(w, 0, need, v->stream));
    uint64_t launches = 0;
    WP_CUDA(wp::launch_format_total(v->d_ids.p, cnt, w, v->sm_count, v->stream, &launches));
    WP_CUDA(cudaMemcpyAsync(&total, w, sizeof(total), cudaMemcpyDeviceToHost, v->stream));
    WP_CUDA(cudaStreamSynchronize(v->stream));
    WP_CUDA(v->d_fmt.grow(static_cast<size_t>(total)));
    WP_CUDA(wp::launch_format(v->d_ids.p, cnt, v->d_fmt.p, w + 2, reinterpret_cast<unsigned int *>(w + 1), v->sm_count,
                              v->stream, &launches));
    g_launches.fetch_add(launches, std::memory_order_relaxed);
    v->stats.kernel_launches += launches;
  }
  void *block = nullptr;
  st = download(v, v->d_fmt.p, static_cast<size_t>(total), 1, "copy id text: ", &block);
  if (st != WP_OK) return st;
  *out = static_cast<char *>(block);
  (*out)[total] = 0;
  *out_len = static_cast<size_t>(total);
  *n_ids = cnt;
  return WP_OK;
}

wp_status wp_set_kernel_timing(wp_vocab *v, int enabled) {
  if (!v) return fail(WP_ERR_INVALID_ARG, "null argument");
  v->timing = enabled != 0;
  return WP_OK;
}

wp_status wp_last_kernel_ms(wp_vocab *v, float ms[3], uint32_t *n_ranges) {
  if (!v || !ms) return fail(WP_ERR_INVALID_ARG, "null argument");
  if (v->device < 0) return fail(WP_ERR_NO_DEVICE, kHostOnly);
  DeviceGuard g(v->device);
  ms[0] = ms[1] = ms[2] = 0.f;
  for (size_t i = 0; i + 4 <= v->timing_used; i += 4) {
    WP_CUDA(cudaEventSynchronize(v->timing_events[i + 3]));
    for (int k = 0; k < 3; k++) {
      float t = 0.f;
      WP_CUDA(cudaEventElapsedTime(&t, v->timing_events[i + k], v->timing_events[i + k + 1]));
      ms[k] += t;
    }
  }
  if (n_ranges) *n_ranges = static_cast<uint32_t>(v->timing_used / 4);
  return WP_OK;
}

wp_status wp_last_stats(wp_vocab *v, wp_stats *out) {
  if (!v || !out) return fail(WP_ERR_INVALID_ARG, "null argument");
  *out = v->stats;
  return WP_OK;
}

wp_status wp_decode(const wp_vocab *v, const int32_t *ids, size_t n_ids, char **out, size_t **offsets_out,
                    size_t *n_tokens, size_t *n_skipped) {
  if (!v || !out || !offsets_out || !n_tokens || (n_ids > 0 && !ids)) return fail(WP_ERR_INVALID_ARG, "null argument");
  std::string joined;
  std::vector<size_t> offs;
  offs.push_back(0);
  size_t skipped = 0;
  const size_t size = v->host.tokens.size();
  for (size_t i = 0; i < n_ids; i++) {
    const int32_t id = ids[i];
    if (id < 0 || static_cast<size_t>(id) > size) {  // fast.cpp:171-174 (note the reference's `>`)
      skipped++;
      continue;
    }
    if (static_cast<size_t>(id) == size) return fail(WP_ERR_ID_RANGE, "token id equals vocabulary size");  // :175 .at()
    const wp::HostToken &t = v->host.tokens[static_cast<size_t>(id)];
    if (t.is_malformed) {  // fast.cpp:176-177
      skipped++;
      continue;
    }
    if (!t.is_prefix) joined += "##";  // fast.cpp:180-183
    joined += t.word;
    offs.push_back(joined.size());
  }
  char *buf = static_cast<char *>(std::malloc(joined.size() + 1));
  size_t *ob = static_cast<size_t *>(std::malloc(offs.size() * sizeof(size_t)));
  if (!buf || !ob) {
    std::free(buf);
    std::free(ob);
    return fail(WP_ERR_NOMEM, "out of memory");
  }
  std::memcpy(buf, joined.data(), joined.size());
  buf[joined.size()] = 0;
  std::memcpy(ob, offs.data(), offs.size() * sizeof(size_t));
  *out = buf;
  *offsets_out = ob;
  *n_tokens = offs.size() - 1;
  if (n_skipped) *n_skipped = skipped;
  return WP_OK;
}

// Test hook: the host mirror of the device longest-match query (wp_vocab.cpp), so that the table
// image can be unit-tested without a GPU.  Nothing on the encode path calls it.
wp_status wp_debug_longest_match(const wp_vocab *v, const char *text, size_t window_bytes, int kind,
                                 uint32_t *len_out, int32_t *id_out) {
  if (!v || !text || !len_out || !id_out) return fail(WP_ERR_INVALID_ARG, "null argument");
  const wp::MatchResult r =
      wp::host_longest_match(v->host, reinterpret_cast<const uint8_t *>(text), window_bytes, kind ? 1u : 0u);
  *len_out = r.len;
  *id_out = r.id;
  return WP_OK;
}

size_t wp_debug_table_slots(const wp_vocab *v) { return v ? v->host.edges.size() : 0; }
size_t wp_debug_table_nodes(const wp_vocab *v) { return v ? v->host.n_nodes : 0; }
size_t wp_debug_long_tokens(const wp_vocab *v) { return v ? v->host.n_long : 0; }
size_t wp_debug_word_slots(const wp_vocab *v) { return v ? v->host.words.size() : 0; }
size_t wp_debug_static_words(const wp_vocab *v) { return v ? v->host.n_static_words : 0; }

/* Test hook: whole-segment lookup in the STATIC word-table image (host mirror of K1's lookup): returns the
 * id count (0 = absent) and writes the ids (at most 11) and the slot's distance from its home slot. */
uint32_t wp_debug_word_lookup(const wp_vocab *v, const char *text, size_t len, int32_t *ids_out, uint32_t *displacement) {
  if (!v || !text || !ids_out) return 0;
  uint32_t slot = 0;
  const uint32_t cnt = wp::host_word_lookup(v->host, reinterpret_cast<const uint8_t *>(text), len, ids_out, &slot);
  if (cnt && displacement) {
    const wp::WordSlot &s = v->host.words[slot];
    const uint32_t mask = static_cast<uint32_t>(v->host.words.size() - 1);
    const uint32_t home = wp::word_hash(s.key[0], s.key[1], s.key[2], s.key[3], static_cast<uint32_t>(len),
                                        32 - log2_of(v->host.words.size()));
    *displacement = (slot - home) & mask;
  }
  return cnt;
}

size_t wp_debug_kernel_geometry(uint32_t *out, size_t cap) { return wp::kernel_geometry(out, out ? cap : 0); }

/* The chunk plan of the host-buffer pipeline for a text (no device needed): writes up to `cap` cut offsets
 * (first 0, last n) to `cuts`, returns their number, or 0 if some stretch has no ASCII space to cut at. */
size_t wp_debug_plan_chunks(const char *text, size_t n, size_t chunk, size_t *cuts, size_t cap) {
  std::vector<size_t> c;
  if (!text || chunk < 64 || !plan_chunks(text, n, chunk, &c)) return 0;
  for (size_t i = 0; i < c.size() && i < cap; i++) cuts[i] = c[i];
  return c.size();
}

/* Host-only run of the staging code (no device): mode 0/1 = the batch packer with ordinary / streaming stores —
 * out receives the packed texts (every text followed by one space), returns the packed size (0 if out is too
 * small); mode 2/3 = CopyPool::copy of texts[0] (lens[0] bytes) to out, ordinary / streamed. */
size_t wp_debug_stage(const char *const *texts, const size_t *lens, size_t n, char *out, size_t out_cap, int mode) {
  if (!out || (n > 0 && (!texts || !lens))) return 0;
  if (mode >= 2) {
    if (n < 1 || lens[0] > out_cap) return 0;
    CopyPool::get().copy(out, texts[0], lens[0], mode == 3);
    return lens[0];
  }
  const PartPlan p = plan_part(lens, 0, n);
  if (p.packed > out_cap) return 0;
  void *block = nullptr;
  if (posix_memalign(&block, 256, p.in_bytes + 64) != 0) return 0;
  pack_part(static_cast<uint8_t *>(block), p, texts, lens, mode == 1);
  std::memcpy(out, static_cast<uint8_t *>(block) + p.off_text, p.packed);
  std::free(block);
  return p.packed;
}

/* Fills out[0..cap) with the code points of single-char word-initial tokens whose word-table slot is at least
 * `min_displacement` slots away from its home slot; returns how many there are.  Lets a test aim at K1's
 * second-slot lookups (1..3) and its rare probe-sequence walk (>= 4). */
size_t wp_debug_displaced_singles(const wp_vocab *v, uint32_t min_displacement, uint32_t *out, size_t cap) {
  if (!v) return 0;
  size_t n = 0;
  const uint32_t mask = static_cast<uint32_t>(v->host.words.size() - 1);
  const uint32_t shift = 32 - log2_of(v->host.words.size());
  for (size_t i = 0; i < v->host.words.size(); i++) {
    const wp::WordSlot &s = v->host.words[i];
    const uint32_t len = wp::word_meta_len(s.meta);
    if (s.meta == 0 || len > 4 || wp::utf8_lead_len(s.key[0] & 0xFFu) != len) continue;  // empty / more than one char
    const uint32_t home = wp::word_hash(s.key[0], s.key[1], s.key[2], s.key[3], len, shift);
    if (((static_cast<uint32_t>(i) - home) & mask) < (min_displacement ? min_displacement : 1u)) continue;
    uint32_t cp = 0;
    if (len == 1) cp = s.key[0] & 0xFFu;
    else wp::utf8_decode(s.key[0] & 0xFFu, (s.key[0] >> 8) & 0xFFu, (s.key[0] >> 16) & 0xFFu, s.key[0] >> 24, 4u, &cp);
    if (n < cap && out) out[n] = cp;
    n++;
  }
  return n;
}

}  // extern "C"
