// osb_host.cu -- host driver + C-ABI (include/onesweep_b200.h) of the B200 OneSweep sort.
//
// The sorter object plays the role of the reference's OneSweepDispatcher (Sort/OneSweepDispatcher.cuh:17-83):
// it owns the ping-pong buffers and the control state and issues the launch plan of
// OneSweepDispatcher.cuh:311-363 -- GlobalHistogram, Scan, then one DigitBinningPass per digit place,
// ping-ponging keys -> alt -> keys.  Differences, all deliberate (DESIGN.md):
//   * no per-sort memset of the 64-bit inclusive descriptors (epoch-stamped); per sort there are two memsets: the 8.3 KB
//     control block (global histogram + tile tickets) and the compact 16-bit reductions (512 B per tile and place:
//     128 MiB at n = 2^30 u32, ~20 us) -- against the reference's 6 memsets over ~573 MB at n = 2^30;
//   * passes whose digit is the same for every key are skipped, and passes with one dominant bin run in the HOT
//     instantiation of the pass, both decided on the device (osb::SortPlan);
//   * a sort of at most one tile is ONE launch of the single-CTA shared-memory sort (also the segmented sort);
//   * no host synchronisation inside the sort; everything is enqueued on the caller's stream;
//   * the caller owns keys/values.
#include <cstdio>
#include <cstring>
#include <new>

#include "../../include/onesweep_b200.h"
#include "osb_kernels.cuh"
#include "osb_common.cuh"
#include "osb_internal.h"

namespace {

constexpr int kVersion = 1002;  // round 2: device plan, bit ranges, forward-progress fallback, hot passes, segmented sort
constexpr int kMaxPlaces = 8;

inline int cuda_status(cudaError_t e) { return e == cudaSuccess ? OSB200_OK : OSB200_ERR_CUDA - static_cast<int>(e); }

#define OSB_TRY(expr)                                      \
    do {                                                   \
        cudaError_t e__ = (expr);                          \
        if (e__ != cudaSuccess) return cuda_status(e__);   \
    } while (0)

// Control block, zeroed by ONE memset per sort: [ghist: 8*256 u64][tickets: 8 u32 (padded)]
struct ControlLayout {
    static constexpr size_t ghist_bytes = kMaxPlaces * osb::kRadix * sizeof(unsigned long long);
    static constexpr size_t ticket_bytes = 64;  // 8 u32 tickets, padded
    static constexpr size_t zeroed_bytes = ghist_bytes + ticket_bytes;
    static constexpr size_t gbase_bytes = kMaxPlaces * osb::kRadix * sizeof(unsigned long long);
    static constexpr size_t err_bytes = 64;
    static constexpr size_t plan_bytes = 64;  // osb::SortPlan, written by the scan kernel of every sort
    static constexpr size_t total = zeroed_bytes + gbase_bytes + err_bytes + plan_bytes;
};

}  // namespace

struct osb200_sorter {
    int device = 0;
    int sm_count = 148;
    uint64_t max_n = 0;
    int key_bytes = 4;
    int value_bytes = 0;
    osb::BinningConfig cfg;
    bool atomic_order_ok = false;
    bool short_circuit = true;   // skip passes whose digit is the same for all keys (decided on the device, no host sync)
    bool small_path = true;      // n <= one tile: the single-CTA shared-memory sort (one launch)
    bool hot_passes = true;      // low-entropy digit places run in the HOT instantiation of the pass (decided on the device)

    void* alt_keys = nullptr;
    uint32_t* alt_vals = nullptr;
    unsigned char* control = nullptr;  // ControlLayout
    uint64_t* desc = nullptr;          // [tiles][256] 64-bit descriptors (epoch-stamped, never cleared)
    uint16_t* agg16 = nullptr;         // [places][tiles][256] compact reductions (zeroed once per sort)
    uint64_t desc_tiles = 0;
    uint32_t epoch = 0;

    // optional per-kernel timing of the last sort (osb200_set_option "profile"): events on the launching stream
    bool profile = false;
    cudaEvent_t ev[kMaxPlaces + 3] = {};
    int ev_count = 0;

    // lazily created staging for the host-buffer entry points
    void* stage_keys = nullptr;
    uint32_t* stage_vals = nullptr;
    cudaStream_t own_stream = nullptr;

    unsigned long long* ghist() const { return reinterpret_cast<unsigned long long*>(control); }
    uint32_t* tickets() const { return reinterpret_cast<uint32_t*>(control + ControlLayout::ghist_bytes); }
    unsigned long long* gbase() const { return reinterpret_cast<unsigned long long*>(control + ControlLayout::zeroed_bytes); }
    unsigned long long* err() const
    {
        return reinterpret_cast<unsigned long long*>(control + ControlLayout::zeroed_bytes + ControlLayout::gbase_bytes);
    }
    osb::SortPlan* plan() const
    {
        return reinterpret_cast<osb::SortPlan*>(control + ControlLayout::zeroed_bytes + ControlLayout::gbase_bytes + ControlLayout::err_bytes);
    }
};

namespace {

uint64_t tiles_for(uint64_t n, uint32_t tile_keys) { return (n + tile_keys - 1) / tile_keys; }
// the compact reductions are stored in blocks of 8 tiles ([tile/8][digit][tile%8], see osb_kernels.cu agg_index)
uint64_t agg_tiles_for(uint64_t n, uint32_t tile_keys) { return (tiles_for(n, tile_keys) + 7) / 8 * 8; }

uint32_t smallest_tile(int key_bytes, bool pairs)
{
    // descriptors are sized for the smallest tile any variant may use
    osb::BinningConfig c;
    uint32_t t = osb::binning_tile_keys(key_bytes, pairs, c);
    for (int v = 1; v < osb::kNumVariants; ++v) {
        c.variant = v;
        const uint32_t t2 = osb::binning_tile_keys(key_bytes, pairs, c);
        if (t2 < t) t = t2;
    }
    return t;
}

// advance the epoch; on wrap-around clear the descriptors once (every ~16M passes)
int next_epoch(osb200_sorter* s, cudaStream_t stream, uint32_t* out)
{
    if (s->epoch >= osb::kEpochMax) {
        OSB_TRY(cudaMemsetAsync(s->desc, 0, s->desc_tiles * osb::kRadix * sizeof(uint64_t), stream));
        s->epoch = 0;
    }
    *out = ++s->epoch;
    return OSB200_OK;
}

int check_handle(const osb200_sorter* s) { return s ? OSB200_OK : OSB200_ERR_INVALID_ARG; }

// The launch plan (reference: OneSweepDispatcher.cuh:311-363): GlobalHistogram, Scan, one DigitBinningPass per digit
// place of [begin_bit, end_bit), then the (normally empty) copy-back.  Everything is enqueued on `stream`; which passes
// actually move data is decided on the device (osb::SortPlan): the host never waits for the histogram.
int sort_impl(osb200_sorter* s, void* d_keys, uint32_t* d_vals, uint64_t n, cudaStream_t stream,
              const osb::KeyCodec* codec = nullptr, int begin_bit = 0, int end_bit = -1)
{
    const int key_bits = s->key_bytes * 8;
    if (end_bit < 0) end_bit = key_bits;
    if (begin_bit < 0 || end_bit > key_bits || begin_bit > end_bit) return OSB200_ERR_INVALID_ARG;
    if (n <= 1 || begin_bit == end_bit) return OSB200_OK;
    if (n > s->max_n) return OSB200_ERR_SIZE;
    if (!d_keys || (reinterpret_cast<uintptr_t>(d_keys) & 15u)) return OSB200_ERR_INVALID_ARG;
    // d_vals == nullptr is a keys-only sort (also on a pairs-capable handle); the handle is never modified to say so
    if (d_vals && !s->value_bytes) return OSB200_ERR_INVALID_ARG;
    // payloads need the keys' 16-byte alignment: the copy-back after an odd number of executed passes moves them as uint4.
    // Checked for every n, so that whether a call is accepted does not depend on which path its size takes.
    if (reinterpret_cast<uintptr_t>(d_vals) & 15u) return OSB200_ERR_INVALID_ARG;
    const int places = (end_bit - begin_bit + 7) / 8;
    const uint32_t last_bits = static_cast<uint32_t>(end_bit - begin_bit - 8 * (places - 1));
    const bool whole_key = begin_bit == 0 && end_bit == key_bits;
    const bool wide = s->cfg.variant == osb::kVariantWide;
    // the device plan (pass skipping, odd pass counts, bit ranges) is a feature of the default kernel
    if (!wide && !whole_key) return OSB200_ERR_UNSUPPORTED;
    const bool use_plan = wide;

    // small-n path (SURVEY 8f rank 4): up to one tile of keys is sorted by ONE CTA in shared memory, one launch
    if (wide && s->small_path && n <= osb::segment_sort_capacity(s->key_bytes, false)) {
        osb::KeyCodec c;
        if (codec) { c = *codec; c.flags = osb::kCodecEncodeOnLoad | osb::kCodecDecodeOnStore; }
        s->ev_count = 0;
        OSB_TRY(osb::launch_segment_sort(d_keys, d_vals, s->key_bytes, nullptr, 1, n, static_cast<uint32_t>(n),
                                         static_cast<uint32_t>(begin_bit), static_cast<uint32_t>(places), last_bits,
                                         codec ? &c : nullptr, s->cfg.rank_mode, s->sm_count, stream));
        return OSB200_OK;
    }

    OSB_TRY(cudaMemsetAsync(s->control, 0, ControlLayout::zeroed_bytes, stream));
    const bool compact = s->cfg.variant != osb::kVariantTilePerCta;  // every other variant uses the compact reductions
    const uint64_t agg_stride = agg_tiles_for(n, osb::binning_tile_keys(s->key_bytes, d_vals != nullptr, s->cfg)) * osb::kRadix;
    // reductions carry no epoch (16-bit words): they are cleared per sort, 512 B per tile and place (128 MiB at n = 2^30)
    if (compact) OSB_TRY(cudaMemsetAsync(s->agg16, 0, agg_stride * places * sizeof(uint16_t), stream));
    int ne = 0;
    auto mark = [&]() -> cudaError_t {
        if (!s->profile) return cudaSuccess;
        if (!s->ev[ne]) { cudaError_t e = cudaEventCreate(&s->ev[ne]); if (e != cudaSuccess) return e; }
        return cudaEventRecord(s->ev[ne++], stream);
    };
    s->ev_count = 0;
    OSB_TRY(mark());
    osb::KeyCodec enc;  // typed keys: the histogram and the first executed pass see encoded keys, the last one stores them decoded
    if (codec) { enc = *codec; enc.flags = osb::kCodecEncodeOnLoad; }
    if (whole_key)
        OSB_TRY(osb::launch_global_histogram(d_keys, n, s->key_bytes, s->ghist(), s->sm_count, stream, codec ? &enc : nullptr));
    else
        OSB_TRY(osb::launch_global_histogram_bits(d_keys, n, s->key_bytes, s->ghist(), s->sm_count, stream, codec ? &enc : nullptr,
                                                  static_cast<uint32_t>(begin_bit), places, last_bits));
    OSB_TRY(mark());
    // hot passes (low-entropy inputs): the default kernel has a second instantiation for them; both are enqueued per pass
    const bool hot_passes = use_plan && s->hot_passes && !(d_vals && osb::binning_tile_keys(4, true, s->cfg) == 16384);
    OSB_TRY(osb::launch_scan(s->ghist(), s->gbase(), places, stream, use_plan ? s->plan() : nullptr, n, s->short_circuit, hot_passes));
    OSB_TRY(mark());

    void* src = d_keys;
    void* dst = s->alt_keys;
    uint32_t* sv = d_vals;
    uint32_t* dv = d_vals ? s->alt_vals : nullptr;
    for (int p = 0; p < places; ++p) {
        uint32_t epoch = 0;
        int st = next_epoch(s, stream, &epoch);
        if (st != OSB200_OK) return st;
        osb::BinningConfig cfg = s->cfg;
        cfg.digit_bits = p == places - 1 ? last_bits : 8u;
        cfg.place = static_cast<uint32_t>(p);
        if (use_plan) cfg.plan = s->plan();
        cfg.hot_passes = hot_passes;
        if (codec) {
            cfg.codec = *codec;
            cfg.codec.flags = use_plan ? osb::kCodecFromPlan
                                       : (p == 0 ? osb::kCodecEncodeOnLoad : 0u) | (p == places - 1 ? osb::kCodecDecodeOnStore : 0u);
        }
        // with a plan every launch gets (caller buffers, alt buffers) and picks its direction on the device
        OSB_TRY(osb::launch_digit_binning(use_plan ? d_keys : src, use_plan ? s->alt_keys : dst, use_plan ? d_vals : sv,
                                          use_plan ? (d_vals ? s->alt_vals : nullptr) : dv, n, s->key_bytes,
                                          static_cast<uint32_t>(begin_bit + 8 * p), s->gbase() + p * osb::kRadix, s->desc,
                                          s->agg16 + p * agg_stride, s->tickets() + p, epoch, cfg, stream));
        OSB_TRY(mark());
        void* t = src; src = dst; dst = t;
        uint32_t* tv = sv; sv = dv; dv = tv;
    }
    // an odd number of EXECUTED passes leaves the result in the alt buffers.  Without skipping the count is known here
    // (even for whole keys: no launch); with skipping only the device knows, and the kernel exits at once if it is even.
    if (use_plan && (s->short_circuit || (places & 1)))
        OSB_TRY(osb::launch_copy_back(s->plan(), s->alt_keys, d_keys, d_vals ? s->alt_vals : nullptr, d_vals, n, s->key_bytes,
                                      s->sm_count, stream));
    s->ev_count = ne;
    return OSB200_OK;
}

int ensure_staging(osb200_sorter* s)
{
    if (!s->own_stream) OSB_TRY(cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking));
    if (!s->stage_keys) {
        if (cudaMalloc(&s->stage_keys, s->max_n * s->key_bytes) != cudaSuccess) return OSB200_ERR_ALLOC;
    }
    if (s->value_bytes && !s->stage_vals) {
        if (cudaMalloc(&s->stage_vals, s->max_n * sizeof(uint32_t)) != cudaSuccess) return OSB200_ERR_ALLOC;
    }
    return OSB200_OK;
}

int sort_host_impl(osb200_sorter* s, void* h_keys, uint32_t* h_vals, uint64_t n)
{
    if (n <= 1) return OSB200_OK;
    if (n > s->max_n) return OSB200_ERR_SIZE;
    if (!h_keys || (h_vals && !s->value_bytes)) return OSB200_ERR_INVALID_ARG;
    int st = ensure_staging(s);
    if (st != OSB200_OK) return st;
    cudaStream_t q = s->own_stream;
    OSB_TRY(cudaMemcpyAsync(s->stage_keys, h_keys, n * s->key_bytes, cudaMemcpyHostToDevice, q));
    if (h_vals) OSB_TRY(cudaMemcpyAsync(s->stage_vals, h_vals, n * sizeof(uint32_t), cudaMemcpyHostToDevice, q));
    st = sort_impl(s, s->stage_keys, h_vals ? s->stage_vals : nullptr, n, q);
    if (st != OSB200_OK) return st;
    OSB_TRY(cudaMemcpyAsync(h_keys, s->stage_keys, n * s->key_bytes, cudaMemcpyDeviceToHost, q));
    if (h_vals) OSB_TRY(cudaMemcpyAsync(h_vals, s->stage_vals, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, q));
    OSB_TRY(cudaStreamSynchronize(q));
    return OSB200_OK;
}

}  // namespace

// ---- internal interfaces used by the sharded path (osb_internal.h) -----------------------------------------
int osb_internal_digit_histogram(osb200_handle h, const void* d_in, uint64_t n, uint32_t shift,
                                 unsigned long long* d_hist256, cudaStream_t stream)
{
    OSB_TRY(cudaMemsetAsync(d_hist256, 0, osb::kRadix * sizeof(unsigned long long), stream));
    if (n) OSB_TRY(osb::launch_digit_histogram(d_in, n, h->key_bytes, shift, d_hist256, h->sm_count, stream));
    return OSB200_OK;
}

int osb_internal_binning_pass(osb200_handle h, const void* d_in, void* d_out, uint64_t n, uint32_t shift,
                              const unsigned long long* d_hist256, const unsigned long long* out_base,
                              cudaStream_t stream)
{
    if (n == 0) return OSB200_OK;
    if (n > h->max_n) return OSB200_ERR_SIZE;
    const unsigned long long* base = out_base;
    OSB_TRY(cudaMemsetAsync(h->tickets(), 0, ControlLayout::ticket_bytes, stream));
    if (!base) {
        OSB_TRY(osb::launch_scan(d_hist256, h->gbase(), 1, stream));
        base = h->gbase();
    }
    if (h->cfg.variant != osb::kVariantTilePerCta) {
        const uint64_t tiles = agg_tiles_for(n, osb::binning_tile_keys(h->key_bytes, false, h->cfg));
        OSB_TRY(cudaMemsetAsync(h->agg16, 0, tiles * osb::kRadix * sizeof(uint16_t), stream));
    }
    uint32_t epoch = 0;
    int st = next_epoch(h, stream, &epoch);
    if (st != OSB200_OK) return st;
    osb::BinningConfig cfg = h->cfg;
    const uint32_t key_bits = static_cast<uint32_t>(h->key_bytes) * 8u;
    cfg.digit_bits = key_bits - shift < 8u ? key_bits - shift : 8u;  // a shift within 8 bits of the top: fewer than 256 bins
    OSB_TRY(osb::launch_digit_binning(d_in, d_out, nullptr, nullptr, n, h->key_bytes, shift, base, h->desc, h->agg16,
                                      h->tickets(), epoch, cfg, stream));
    return OSB200_OK;
}

extern "C" {

int osb200_version(void) { return kVersion; }

const char* osb200_status_string(int status)
{
    switch (status) {
        case OSB200_OK: return "ok";
        case OSB200_ERR_INVALID_ARG: return "invalid argument";
        case OSB200_ERR_SIZE: return "n exceeds the sorter's max_n";
        case OSB200_ERR_UNSUPPORTED: return "unsupported key/value combination";
        case OSB200_ERR_NO_DEVICE: return "no usable sm_100 CUDA device";
        case OSB200_ERR_ALLOC: return "device allocation failed";
        case OSB200_ERR_NCCL: return "NCCL error";
        default: break;
    }
    if (status <= OSB200_ERR_CUDA) return cudaGetErrorString(static_cast<cudaError_t>(OSB200_ERR_CUDA - status));
    return "unknown status";
}

uint64_t osb200_workspace_bytes(uint64_t max_n, int key_bytes, int value_bytes)
{
    if ((key_bytes != 4 && key_bytes != 8) || (value_bytes != 0 && value_bytes != 4)) return 0;
    const uint64_t tiles = tiles_for(max_n ? max_n : 1, smallest_tile(key_bytes, value_bytes != 0));
    return max_n * key_bytes + max_n * value_bytes + tiles * osb::kRadix * sizeof(uint64_t) +
           (tiles + 8) * osb::kRadix * sizeof(uint16_t) * key_bytes + ControlLayout::total;
}

int osb200_create(osb200_handle* out, uint64_t max_n, int key_bytes, int value_bytes)
{
    if (!out) return OSB200_ERR_INVALID_ARG;
    *out = nullptr;
    if ((key_bytes != 4 && key_bytes != 8) || (value_bytes != 0 && value_bytes != 4)) return OSB200_ERR_INVALID_ARG;
    if (key_bytes == 8 && value_bytes != 0) return OSB200_ERR_UNSUPPORTED;
    if (max_n == 0 || max_n > (1ull << 34)) return OSB200_ERR_INVALID_ARG;

    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return OSB200_ERR_NO_DEVICE; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) { cudaGetLastError(); return OSB200_ERR_NO_DEVICE; }
    if (prop.major != 10) return OSB200_ERR_NO_DEVICE;  // sm_100a binary only: no fallback of any kind

    osb200_sorter* s = new (std::nothrow) osb200_sorter();
    if (!s) return OSB200_ERR_ALLOC;
    s->device = dev;
    s->sm_count = prop.multiProcessorCount;
    s->cfg.sm_count = s->sm_count;
    s->cfg.variant = osb::kVariantWide;
    s->max_n = max_n;
    s->key_bytes = key_bytes;
    s->value_bytes = value_bytes;

    cudaError_t e = osb::configure_kernels();
    if (e != cudaSuccess) { delete s; return cuda_status(e); }

    s->desc_tiles = tiles_for(max_n, smallest_tile(key_bytes, value_bytes != 0));
    bool ok = cudaMalloc(&s->alt_keys, max_n * key_bytes) == cudaSuccess;
    if (ok && value_bytes) ok = cudaMalloc(&s->alt_vals, max_n * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaMalloc(&s->control, ControlLayout::total) == cudaSuccess;
    ok = ok && cudaMalloc(&s->desc, s->desc_tiles * osb::kRadix * sizeof(uint64_t)) == cudaSuccess;
    ok = ok && cudaMalloc(&s->agg16, (s->desc_tiles + 8) * osb::kRadix * sizeof(uint16_t) * key_bytes) == cudaSuccess;
    if (!ok) { cudaGetLastError(); osb200_destroy(s); return OSB200_ERR_ALLOC; }
    e = cudaMemset(s->desc, 0, s->desc_tiles * osb::kRadix * sizeof(uint64_t));  // epoch 0 == never valid
    if (e == cudaSuccess) e = cudaMemset(s->control, 0, ControlLayout::total);

    // Verify on THIS device the hardware property the atomic ranking depends on; otherwise use ballots.
    if (e == cudaSuccess) e = osb::launch_atomic_order_selftest(s->err(), s->sm_count, nullptr);
    unsigned long long mism = 1;
    if (e == cudaSuccess) e = cudaMemcpy(&mism, s->err(), sizeof(mism), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { osb200_destroy(s); return cuda_status(e); }
    s->atomic_order_ok = (mism == 0);
    s->cfg.rank_mode = s->atomic_order_ok ? osb::kRankAtomic : osb::kRankBallot;
    *out = s;
    return OSB200_OK;
}

int osb200_destroy(osb200_handle h)
{
    if (!h) return OSB200_ERR_INVALID_ARG;
    cudaFree(h->alt_keys);
    cudaFree(h->alt_vals);
    cudaFree(h->control);
    cudaFree(h->desc);
    cudaFree(h->agg16);
    cudaFree(h->stage_keys);
    cudaFree(h->stage_vals);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    for (cudaEvent_t e : h->ev) if (e) cudaEventDestroy(e);
    delete h;
    return OSB200_OK;
}

int osb200_sort_keys_u32(osb200_handle h, uint32_t* d_keys, uint64_t n, void* stream)
{
    if (check_handle(h) != OSB200_OK || h->key_bytes != 4) return OSB200_ERR_INVALID_ARG;
    return sort_impl(h, d_keys, nullptr, n, static_cast<cudaStream_t>(stream));  // a pairs-capable sorter may sort keys only
}

int osb200_sort_pairs_u32(osb200_handle h, uint32_t* d_keys, uint32_t* d_values, uint64_t n, void* stream)
{
    if (check_handle(h) != OSB200_OK || h->key_bytes != 4 || h->value_bytes != 4) return OSB200_ERR_INVALID_ARG;
    if (n > 1 && !d_values) return OSB200_ERR_INVALID_ARG;
    return sort_impl(h, d_keys, d_values, n, static_cast<cudaStream_t>(stream));
}

int osb200_sort_keys_u64(osb200_handle h, uint64_t* d_keys, uint64_t n, void* stream)
{
    if (check_handle(h) != OSB200_OK || h->key_bytes != 8) return OSB200_ERR_INVALID_ARG;
    return sort_impl(h, d_keys, nullptr, n, static_cast<cudaStream_t>(stream));
}

// Typed keys (SURVEY 8f rank 1).  key_type must match the handle's key width.
static int make_codec(const osb200_sorter* h, int key_type, int descending, osb::KeyCodec* c)
{
    const bool wide64 = h->key_bytes == 8;
    const unsigned long long all = wide64 ? ~0ull : 0xffffffffull, sign = wide64 ? (1ull << 63) : (1ull << 31);
    switch (key_type) {
        case OSB200_KEY_U32: if (wide64) return OSB200_ERR_INVALID_ARG; c->a = 0; c->b = 0; break;
        case OSB200_KEY_I32: if (wide64) return OSB200_ERR_INVALID_ARG; c->a = 0; c->b = sign; break;
        case OSB200_KEY_F32: if (wide64) return OSB200_ERR_INVALID_ARG; c->a = all; c->b = sign; break;
        case OSB200_KEY_U64: if (!wide64) return OSB200_ERR_INVALID_ARG; c->a = 0; c->b = 0; break;
        case OSB200_KEY_I64: if (!wide64) return OSB200_ERR_INVALID_ARG; c->a = 0; c->b = sign; break;
        case OSB200_KEY_F64: if (!wide64) return OSB200_ERR_INVALID_ARG; c->a = all; c->b = sign; break;
        default: return OSB200_ERR_INVALID_ARG;
    }
    c->d = descending ? all : 0;
    c->flags = 0;
    return OSB200_OK;
}

int osb200_sort_keys_typed(osb200_handle h, void* d_keys, uint64_t n, int key_type, int descending, void* stream)
{
    if (check_handle(h) != OSB200_OK) return OSB200_ERR_INVALID_ARG;
    osb::KeyCodec c;
    int st = make_codec(h, key_type, descending, &c);
    if (st != OSB200_OK) return st;
    if (h->cfg.variant != osb::kVariantWide) return OSB200_ERR_UNSUPPORTED;
    const bool plain = c.a == 0 && c.b == 0 && c.d == 0;
    return sort_impl(h, d_keys, nullptr, n, static_cast<cudaStream_t>(stream), plain ? nullptr : &c);
}

int osb200_segmented_sort_u32(osb200_handle h, uint32_t* d_keys, uint32_t* d_values, const uint64_t* d_segment_offsets,
                              uint64_t num_segments, uint32_t max_segment_len, void* stream)
{
    if (check_handle(h) != OSB200_OK) return OSB200_ERR_INVALID_ARG;
    if (h->key_bytes != 4 || (d_values && h->value_bytes != 4)) return OSB200_ERR_INVALID_ARG;
    if (num_segments == 0 || max_segment_len <= 1) return OSB200_OK;
    if (!d_keys || !d_segment_offsets) return OSB200_ERR_INVALID_ARG;
    if (max_segment_len > osb::segment_sort_capacity(4, false)) return OSB200_ERR_SIZE;  // sort longer segments with osb200_sort_*
    OSB_TRY(osb::launch_segment_sort(d_keys, d_values, 4, reinterpret_cast<const unsigned long long*>(d_segment_offsets), num_segments,
                                     0, max_segment_len, 0, 4, 8, nullptr, h->cfg.rank_mode, h->sm_count,
                                     static_cast<cudaStream_t>(stream)));
    return OSB200_OK;
}

int osb200_sort_bits(osb200_handle h, void* d_keys, uint32_t* d_values, uint64_t n, int begin_bit, int end_bit, void* stream)
{
    if (check_handle(h) != OSB200_OK) return OSB200_ERR_INVALID_ARG;
    if (d_values && (h->key_bytes != 4 || h->value_bytes != 4)) return OSB200_ERR_INVALID_ARG;
    return sort_impl(h, d_keys, d_values, n, static_cast<cudaStream_t>(stream), nullptr, begin_bit, end_bit);
}

int osb200_sort_pairs_typed(osb200_handle h, void* d_keys, uint32_t* d_values, uint64_t n, int key_type, int descending,
                            void* stream)
{
    if (check_handle(h) != OSB200_OK || h->key_bytes != 4 || h->value_bytes != 4) return OSB200_ERR_INVALID_ARG;
    if (n > 1 && !d_values) return OSB200_ERR_INVALID_ARG;
    osb::KeyCodec c;
    int st = make_codec(h, key_type, descending, &c);
    if (st != OSB200_OK) return st;
    if (h->cfg.variant != osb::kVariantWide) return OSB200_ERR_UNSUPPORTED;
    const bool plain = c.a == 0 && c.b == 0 && c.d == 0;
    return sort_impl(h, d_keys, d_values, n, static_cast<cudaStream_t>(stream), plain ? nullptr : &c);
}

int osb200_sort_host_keys_u32(osb200_handle h, uint32_t* h_keys, uint64_t n)
{
    if (check_handle(h) != OSB200_OK || h->key_bytes != 4) return OSB200_ERR_INVALID_ARG;
    return sort_host_impl(h, h_keys, nullptr, n);
}

int osb200_sort_host_pairs_u32(osb200_handle h, uint32_t* h_keys, uint32_t* h_values, uint64_t n)
{
    if (check_handle(h) != OSB200_OK || h->key_bytes != 4 || h->value_bytes != 4) return OSB200_ERR_INVALID_ARG;
    if (n > 1 && !h_values) return OSB200_ERR_INVALID_ARG;
    return sort_host_impl(h, h_keys, h_values, n);
}

int osb200_sort_host_keys_u64(osb200_handle h, uint64_t* h_keys, uint64_t n)
{
    if (check_handle(h) != OSB200_OK || h->key_bytes != 8) return OSB200_ERR_INVALID_ARG;
    return sort_host_impl(h, h_keys, nullptr, n);
}

int osb200_global_histogram(osb200_handle h, const void* d_keys, uint64_t n, uint64_t* d_hist, void* stream)
{
    if (check_handle(h) != OSB200_OK || !d_hist || (n && !d_keys)) return OSB200_ERR_INVALID_ARG;
    if (reinterpret_cast<uintptr_t>(d_keys) & 15u) return OSB200_ERR_INVALID_ARG;
    cudaStream_t q = static_cast<cudaStream_t>(stream);
    OSB_TRY(cudaMemsetAsync(d_hist, 0, static_cast<size_t>(h->key_bytes) * osb::kRadix * sizeof(uint64_t), q));
    if (n == 0) return OSB200_OK;
    OSB_TRY(osb::launch_global_histogram(d_keys, n, h->key_bytes, reinterpret_cast<unsigned long long*>(d_hist),
                                         h->sm_count, q));
    return OSB200_OK;
}

int osb200_digit_binning_pass(osb200_handle h, const void* d_in, void* d_out, const uint32_t* d_in_values,
                              uint32_t* d_out_values, uint64_t n, uint32_t radix_shift, void* stream)
{
    if (check_handle(h) != OSB200_OK) return OSB200_ERR_INVALID_ARG;
    if (n == 0) return OSB200_OK;
    if (!d_in || !d_out || d_in == d_out) return OSB200_ERR_INVALID_ARG;
    if ((reinterpret_cast<uintptr_t>(d_in) & 15u) || (reinterpret_cast<uintptr_t>(d_out) & 15u)) return OSB200_ERR_INVALID_ARG;
    if (n > h->max_n) return OSB200_ERR_SIZE;
    if (radix_shift >= static_cast<uint32_t>(h->key_bytes) * 8u) return OSB200_ERR_INVALID_ARG;
    if ((d_in_values != nullptr) != (d_out_values != nullptr)) return OSB200_ERR_INVALID_ARG;
    if (d_in_values && (h->key_bytes != 4 || h->value_bytes != 4)) return OSB200_ERR_UNSUPPORTED;
    cudaStream_t q = static_cast<cudaStream_t>(stream);
    // histogram of this digit only, then the pass (the reference's multiples of 8 and any other shift alike)
    int st = osb_internal_digit_histogram(h, d_in, n, radix_shift, h->ghist(), q);
    if (st != OSB200_OK) return st;
    OSB_TRY(cudaMemsetAsync(h->tickets(), 0, ControlLayout::ticket_bytes, q));
    OSB_TRY(osb::launch_scan(h->ghist(), h->gbase(), 1, q));
    if (h->cfg.variant != osb::kVariantTilePerCta)
        OSB_TRY(cudaMemsetAsync(h->agg16, 0, (h->desc_tiles + 8) * osb::kRadix * sizeof(uint16_t), q));
    uint32_t epoch = 0;
    st = next_epoch(h, q, &epoch);
    if (st != OSB200_OK) return st;
    osb::BinningConfig cfg = h->cfg;
    const uint32_t key_bits = static_cast<uint32_t>(h->key_bytes) * 8u;
    cfg.digit_bits = key_bits - radix_shift < 8u ? key_bits - radix_shift : 8u;
    OSB_TRY(osb::launch_digit_binning(d_in, d_out, d_in_values, d_out_values, n, h->key_bytes, radix_shift, h->gbase(), h->desc,
                                      h->agg16, h->tickets(), epoch, cfg, q));
    return OSB200_OK;
}

int osb200_validate(osb200_handle h, const void* d_keys, uint64_t n, uint64_t* h_err_count, void* stream)
{
    if (check_handle(h) != OSB200_OK || !h_err_count) return OSB200_ERR_INVALID_ARG;
    *h_err_count = 0;
    if (n < 2) return OSB200_OK;
    if (!d_keys) return OSB200_ERR_INVALID_ARG;
    cudaStream_t q = static_cast<cudaStream_t>(stream);
    OSB_TRY(cudaMemsetAsync(h->err(), 0, sizeof(unsigned long long), q));
    OSB_TRY(osb::launch_validate(d_keys, n, h->key_bytes, h->err(), h->sm_count, q));
    unsigned long long v = 0;
    OSB_TRY(cudaMemcpyAsync(&v, h->err(), sizeof(v), cudaMemcpyDeviceToHost, q));
    OSB_TRY(cudaStreamSynchronize(q));
    *h_err_count = v;
    return OSB200_OK;
}

int osb200_init_random_u32(uint32_t* d_keys, uint32_t* d_payload, uint64_t n, uint32_t and_count, uint32_t seed,
                           int payload_is_index, void* stream)
{
    if (n == 0) return OSB200_OK;
    if (!d_keys) return OSB200_ERR_INVALID_ARG;
    OSB_TRY(osb::launch_init_random(d_keys, d_payload, n, and_count, seed, payload_is_index != 0,
                                    static_cast<cudaStream_t>(stream)));
    return OSB200_OK;
}

int osb200_set_option(osb200_handle h, const char* key, int64_t value)
{
    if (check_handle(h) != OSB200_OK || !key) return OSB200_ERR_INVALID_ARG;
    if (!std::strcmp(key, "rank_mode")) {
        if (value != osb::kRankAtomic && value != osb::kRankBallot) return OSB200_ERR_INVALID_ARG;
        if (value == osb::kRankAtomic && !h->atomic_order_ok) return OSB200_ERR_UNSUPPORTED;
        h->cfg.rank_mode = static_cast<int>(value);
        return OSB200_OK;
    }
    if (!std::strcmp(key, "profile")) { h->profile = value != 0; return OSB200_OK; }
    if (!std::strcmp(key, "short_circuit")) { h->short_circuit = value != 0; return OSB200_OK; }
    if (!std::strcmp(key, "small_path")) { h->small_path = value != 0; return OSB200_OK; }
    if (!std::strcmp(key, "hot_passes")) { h->hot_passes = value != 0; return OSB200_OK; }
    if (!std::strcmp(key, "spin_cap")) {
        if (value < 1 || value > (1ll << 30)) return OSB200_ERR_INVALID_ARG;
        h->cfg.spin_cap = static_cast<uint32_t>(value);
        return OSB200_OK;
    }
    if (!std::strcmp(key, "debug_stall_every")) {  // test hook of the forward-progress fallback (0 = off)
        if (value < 0 || value > (1ll << 30)) return OSB200_ERR_INVALID_ARG;
        h->cfg.debug_stall_every = static_cast<uint32_t>(value);
        return OSB200_OK;
    }
    if (!std::strcmp(key, "variant")) {
        if (value < 0 || value >= osb::kNumVariants) return OSB200_ERR_INVALID_ARG;
        h->cfg.variant = static_cast<int>(value);
        return OSB200_OK;
    }
    return OSB200_ERR_INVALID_ARG;
}

int osb200_get_profile(osb200_handle h, float* out_ms, int capacity)
{
    if (check_handle(h) != OSB200_OK || !out_ms) return OSB200_ERR_INVALID_ARG;
    if (h->ev_count < 2) return 0;
    OSB_TRY(cudaEventSynchronize(h->ev[h->ev_count - 1]));
    int k = 0;
    for (int i = 0; i + 1 < h->ev_count && k < capacity; ++i, ++k) OSB_TRY(cudaEventElapsedTime(&out_ms[k], h->ev[i], h->ev[i + 1]));
    return k;
}

int64_t osb200_get_info(osb200_handle h, const char* key)
{
    if (check_handle(h) != OSB200_OK || !key) return OSB200_ERR_INVALID_ARG;
    if (!std::strcmp(key, "tile_keys")) return osb::binning_tile_keys(h->key_bytes, h->value_bytes != 0, h->cfg);
    if (!std::strcmp(key, "launches_per_sort")) {  // histogram + scan + one pass per place (+ copy-back: keys [+ values])
        const bool wide = h->cfg.variant == osb::kVariantWide;
        const bool cb = wide && h->short_circuit;
        return 2 + h->key_bytes * ((wide && h->hot_passes) ? 2 : 1) + (cb ? (h->value_bytes ? 2 : 1) : 0);
    }
    if (!std::strcmp(key, "memsets_per_sort")) return h->cfg.variant != osb::kVariantTilePerCta ? 2 : 1;
    if (!std::strcmp(key, "short_circuit")) return h->short_circuit ? 1 : 0;
    if (!std::strcmp(key, "small_path")) return h->small_path ? 1 : 0;
    if (!std::strcmp(key, "hot_passes")) return h->hot_passes ? 1 : 0;
    if (!std::strcmp(key, "last_hot_mask")) {
        osb::SortPlan pl;
        if (cudaMemcpy(&pl, h->plan(), sizeof(pl), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        return static_cast<int>((pl.skip_mask >> osb::kPlanHotShift) & 0xffu);
    }
    if (!std::strcmp(key, "small_path_max_n")) return osb::segment_sort_capacity(h->key_bytes, false);
    if (!std::strcmp(key, "spin_cap")) return h->cfg.spin_cap;
    if (!std::strcmp(key, "last_skip_mask") || !std::strcmp(key, "last_executed_passes")) {
        // the plan of the last sort on this handle (synchronises the device: introspection / tests only)
        osb::SortPlan pl;
        if (cudaMemcpy(&pl, h->plan(), sizeof(pl), cudaMemcpyDeviceToHost) != cudaSuccess) return OSB200_ERR_CUDA;
        return key[5] == 's' ? static_cast<int64_t>(pl.skip_mask & 0xffffu) : static_cast<int64_t>(pl.executed);
    }
    if (!std::strcmp(key, "sm_count")) return h->sm_count;
    if (!std::strcmp(key, "rank_mode")) return h->cfg.rank_mode;
    if (!std::strcmp(key, "variant")) return h->cfg.variant;
    if (!std::strcmp(key, "atomic_order_ok")) return h->atomic_order_ok ? 1 : 0;
    if (!std::strcmp(key, "max_n")) return static_cast<int64_t>(h->max_n);
    if (!std::strcmp(key, "epoch")) return h->epoch;
    return OSB200_ERR_INVALID_ARG;
}

}  // extern "C"
