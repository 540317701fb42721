// c_abi.cu -- the extern "C" boundary declared in include/sela_b200.h.
//
// Host-side plumbing only: device selection, a grow-only device workspace, the
// launches.  No algorithm lives here and there is no CPU fallback: without a
// CUDA device every compute entry point returns SELAB200_ERR_NO_DEVICE.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#include "kernels.cuh"

using namespace selab200;

namespace {

thread_local char g_error[512] = "";
std::mutex g_mutex;
std::atomic<uint64_t> g_launches{0};

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof g_error, fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                      \
    do {                                                                                    \
        cudaError_t e_ = (expr);                                                            \
        if (e_ != cudaSuccess)                                                              \
            return fail(SELAB200_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

// A grow-only allocation, on the device or pinned on the host: a request that fits keeps the block, a
// larger one replaces it with an eighth plus 4 KB to spare.
template <bool Pinned>
struct GrowBuffer {
    void *ptr = nullptr;
    size_t bytes = 0;
    int ensure(size_t need)
    {
        if (need <= bytes)
            return 0;
        release();
        const size_t want = need + need / 8 + 4096;
        const cudaError_t e = Pinned ? cudaMallocHost(&ptr, want) : cudaMalloc(&ptr, want);
        if (e != cudaSuccess)
            return Pinned ? fail(SELAB200_ERR_CUDA, "cudaMallocHost(%zu) failed", want)
                          : fail(SELAB200_ERR_CUDA, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        bytes = want;
        return 0;
    }
    void release()
    {
        if (ptr && Pinned)
            cudaFreeHost(ptr);
        else if (ptr)
            cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
    }
};
using DeviceBuffer = GrowBuffer<false>;
using PinnedBuffer = GrowBuffer<true>;

// What a container handle owns besides the walk result: the device image of the bytes, a pinned
// descriptor table and the upload events.  Recycled through a small free list, because a process
// that decodes many files would otherwise pay cudaMalloc/cudaFree (a device-wide sync) and
// cudaMallocHost/cudaFreeHost for every one of them.
struct ContainerBuffers {
    static constexpr int kPieces = 8;
    DeviceBuffer image;
    PinnedBuffer descs; // selab200_subframe_desc, file order
    cudaEvent_t ev_piece[kPieces] = {};
    void destroy()
    {
        for (cudaEvent_t &e : ev_piece)
            if (e) {
                cudaEventDestroy(e);
                e = nullptr;
            }
        image.release();
        descs.release();
    }
};

constexpr size_t kMaxSpareBuffers = 16;
constexpr int kMaxChunks = 72;
constexpr int kLanes = 8; // concurrent compute streams of the pipelined host calls

struct Context {
    bool ready = false;
    int device = -1;
    cudaStream_t stream = nullptr;                 // stage-level calls
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr; // pipelined batch calls: copy engines ...
    cudaStream_t s_compute[kLanes] = {};           // ... and alternating compute lanes
    cudaEvent_t ev_h2d[kMaxChunks], ev_done[kMaxChunks], ev_scan[kMaxChunks], ev_reset;
    bool events = false;
    DeviceBuffer in, descs, words, work, lane_work[kLanes], aux, small;
    int32_t *h_small = nullptr;                    // pinned: [0] status, [2..3] words_used
    unsigned long long *h_totals = nullptr;        // pinned: arena fill level after each chunk
    size_t last_rice_n_sub = 0;                    // selab200_rice_decode_frames_device bookkeeping (flag count query)
    cudaStream_t last_rice_stream = nullptr;
    std::vector<ContainerBuffers> spare;           // recycled container buffers of this device (g_mutex held)
};

// One context per device the library was initialised for (selab200_init / selab200_init_devices), slot 0 the
// primary.  An API call runs on the primary (or, for the *_device forms, on the device that owns the caller's
// pointers) and hands that context down; the multi-device host-buffer calls give every device a worker thread
// of its own, with that device's context.  Contexts share nothing, so the workers never contend.
constexpr int kMaxDevices = 16;
Context g_slots[kMaxDevices];
int g_n_ctx = 0;
int g_last_rice_slot = -1; // the slot selab200_rice_decode_frames_device last ran on (flag count query)

// Makes the context's device the calling thread's current one: the current device is per host thread, and
// callers may arrive on a thread other than init()'s.
int use_device(const Context &c)
{
    cudaError_t e = cudaSetDevice(c.device);
    if (e != cudaSuccess)
        return fail(SELAB200_ERR_CUDA, "cudaSetDevice(%d) failed: %s", c.device, cudaGetErrorString(e));
    return 0;
}

// Returns `rc` after `cleanup`, keeping the message of the error that caused it.
template <typename F>
int fail_after_cleanup(int rc, F cleanup)
{
    char keep[sizeof g_error];
    memcpy(keep, g_error, sizeof keep);
    cleanup();
    memcpy(g_error, keep, sizeof keep);
    return rc;
}

int check_channels(uint32_t channels)
{
    if (channels == 0 || channels > SELAB200_MAX_CHANNELS)
        return fail(SELAB200_ERR_ARGUMENT, "channels must be in [1, %d]", SELAB200_MAX_CHANNELS);
    return 0;
}

// On every exit from a pipelined call -- error paths included -- nothing may still be
// reading or writing the caller's host buffers.
struct PipelineDrain {
    Context &c;
    ~PipelineDrain()
    {
        if (c.s_h2d)
            cudaStreamSynchronize(c.s_h2d);
        for (int i = 0; i < kLanes; i++)
            if (c.s_compute[i])
                cudaStreamSynchronize(c.s_compute[i]);
        if (c.s_d2h)
            cudaStreamSynchronize(c.s_d2h);
    }
};

// Chunk boundaries of the pipelined host-buffer calls (encode and both decode paths).  About eight
// chunks: enough to overlap PCIe with compute, each still several waves of warps, and at most 16 384
// frames, which bounds the workspace for huge batches (tools/e2e_chunk_sweep.py on a B200, BASELINE
// batch of 12 919 stereo frames: encode is best at 8 chunks, 4.2 ms end to end vs 3.8 ms of kernels).
// The first and the last chunk are cut into shrinking pieces: what a pipeline cannot hide is the
// upload of the first chunk before any kernel runs and the download of the last chunk after the last
// kernel, so those two are made small (same batch: encode call 4.06 -> 3.93 ms, decode call 3.80 ->
// 3.67 ms).
struct ChunkPlan {
    std::vector<uint32_t> start; // n_chunks + 1 boundaries
    uint32_t max_frames = 0;     // largest chunk (sizes the per-lane workspace)
    uint32_t chunks() const { return (uint32_t)start.size() - 1; }
};

ChunkPlan plan_chunks(uint32_t n_frames)
{
    // SELAB200_CHUNK_FRAMES (tests and measurement only): frames per chunk, no shrinking pieces; the tests
    // use it to push many tiny chunks through the pipelines on small inputs.
    const char *env = std::getenv("SELAB200_CHUNK_FRAMES");
    const long forced = env ? std::atol(env) : 0;
    uint32_t cf = forced > 0 ? (uint32_t)forced : std::min(std::max((n_frames + 7) / 8, 512u), 16384u);
    while ((n_frames + cf - 1) / cf > (uint32_t)kMaxChunks)
        cf *= 2;
    ChunkPlan p;
    const uint32_t n_base = (n_frames + cf - 1) / cf;
    const bool taper = !env && n_base >= 4 && n_base + 6 <= (uint32_t)kMaxChunks;
    p.start.push_back(0);
    for (uint32_t c = 0; c < n_base; c++) {
        const uint32_t f0 = c * cf, f1 = (f0 + cf <= n_frames) ? f0 + cf : n_frames, len = f1 - f0;
        if (taper && c == 0 && len >= 512) {
            p.start.push_back(f0 + len / 8);
            p.start.push_back(f0 + len / 2);
        } else if (taper && c == n_base - 1 && len >= 512) {
            p.start.push_back(f0 + len / 2);
            p.start.push_back(f0 + len / 2 + len / 4);
            p.start.push_back(f0 + len / 2 + len / 4 + len / 8);
        }
        p.start.push_back(f1);
    }
    for (uint32_t c = 0; c + 1 < p.start.size(); c++)
        p.max_frames = std::max(p.max_frames, p.start[c + 1] - p.start[c]);
    return p;
}

const char *status_text(int s)
{
    switch (s) {
    case SELAB200_ERR_CAPACITY: return "output word arena too small";
    case SELAB200_ERR_RANGE: return "value outside the representable domain (16-bit audio / uint16 word counts)";
    case SELAB200_ERR_BITSTREAM: return "malformed subframe descriptor or Rice stream";
    default: return "device reported an error";
    }
}

// Sets `c` to the primary context and makes its device current (g_mutex held).
int require_ready(Context *&c)
{
    c = &g_slots[0];
    if (g_n_ctx == 0 || !c->ready)
        return fail(SELAB200_ERR_NOT_INIT, "selab200_init() has not been called (or found no CUDA device)");
    return use_device(*c);
}

// The *_device forms run on the device that owns the caller's buffers: sets `c` to that device's context and
// makes it current.  A null pointer selects the primary (the caller reports the null pointer).
int require_ready_for(const void *device_ptr, Context *&c)
{
    if (!device_ptr || g_n_ctx == 0)
        return require_ready(c);
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, device_ptr) != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
        cudaGetLastError();
        return fail(SELAB200_ERR_ARGUMENT, "not a device pointer");
    }
    for (int i = 0; i < g_n_ctx; i++)
        if (g_slots[i].ready && g_slots[i].device == attr.device) {
            c = &g_slots[i];
            return use_device(*c);
        }
    return fail(SELAB200_ERR_ARGUMENT, "the buffers live on device %d, which the library was not initialised for "
                                       "(selab200_init / selab200_init_devices)", attr.device);
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// Raises a kernel's dynamic shared-memory limit; remembered per (kernel, device): the attribute call is a
// host round trip that would otherwise precede every launch.
template <typename K>
int set_smem(K kernel, size_t bytes)
{
    static std::mutex m;
    static std::vector<std::pair<std::pair<const void *, int>, size_t>> done;
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    const std::pair<const void *, int> key(reinterpret_cast<const void *>(kernel), dev);
    std::lock_guard<std::mutex> lock(m);
    for (auto &e : done)
        if (e.first == key) {
            if (e.second >= bytes)
                return 0;
            CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
            e.second = bytes;
            return 0;
        }
    CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    done.emplace_back(key, bytes);
    return 0;
}

int launch_check(const char *what)
{
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
        return fail(SELAB200_ERR_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(e));
    return 0;
}

// ---- device-resident cores (no synchronisation) --------------------------

// `fresh`: reset status and the arena fill level first (a stand-alone batch); the pipelined
// host path resets once and then chains chunks through *d_used.  `before_scan`: optional event
// the scan must wait for (the previous chunk's scan, when chunks alternate between streams).
int encode_device(const int16_t *d_pcm, uint32_t n_frames, uint32_t channels, selab200_subframe_desc *d_descs,
                  uint32_t *d_words, size_t capacity, uint64_t *d_used, int32_t *d_status, void *d_ws,
                  size_t ws_bytes, cudaStream_t stream, bool fresh = true, cudaEvent_t before_scan = nullptr,
                  cudaEvent_t after_scan = nullptr, unsigned long long *h_fill_after = nullptr,
                  uint8_t *d_container = nullptr, unsigned long long sub_base = 0)
{
    if (int rc = check_channels(channels))
        return rc;
    if (ws_bytes < selab200_encode_workspace_bytes(n_frames, channels))
        return fail(SELAB200_ERR_ARGUMENT, "encode workspace too small");
    if (channels == 2 && (reinterpret_cast<uintptr_t>(d_pcm) & 15) != 0) // the stereo kernel reads 16 bytes (4 sample pairs) at a time
        return fail(SELAB200_ERR_ARGUMENT, "stereo PCM must be 16-byte aligned on the device");
    if (fresh) {
        CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int32_t), stream));
        CUDA_TRY(cudaMemsetAsync(d_used, 0, sizeof(uint64_t), stream));
    }
    if (n_frames == 0)
        return 0;
    const bool stereo = channels == 2;
    const size_t n_units = encode_units(n_frames, channels);
    const size_t n_sub = (size_t)n_frames * channels;
    EncodeParams p;
    p.pcm = d_pcm;
    p.n_frames = n_frames;
    p.channels = channels;
    p.descs = d_descs;
    p.words = d_words;
    p.capacity = capacity;
    p.words_used = reinterpret_cast<unsigned long long *>(d_used);
    p.status = d_status;
    p.units = static_cast<UnitRecord *>(d_ws);
    p.slots = reinterpret_cast<uint32_t *>(static_cast<char *>(d_ws) + align256(n_units * sizeof(UnitRecord)));
    p.residues = reinterpret_cast<int32_t *>(reinterpret_cast<char *>(p.slots) + align256(n_units * (size_t)kSlotWords * 4));
    if (stereo) {
        constexpr size_t smem = encode_smem_bytes<true>();
        if (int rc = set_smem(k_encode_units<true>, smem))
            return rc;
        k_encode_units<true><<<(unsigned)n_units, 32, smem, stream>>>(p);
    } else {
        constexpr size_t smem = encode_smem_bytes<false>();
        if (int rc = set_smem(k_encode_units<false>, smem))
            return rc;
        k_encode_units<false><<<(unsigned)n_units, 32, smem, stream>>>(p);
    }
    if (int rc = launch_check("k_encode_units"))
        return rc;
    const unsigned scan_ctas = (unsigned)((n_sub + kScanTile - 1) / kScanTile);
    k_encode_sizes<<<scan_ctas, kScanTile, 0, stream>>>(p);
    if (int rc = launch_check("k_encode_sizes"))
        return rc;
    if (before_scan)
        CUDA_TRY(cudaStreamWaitEvent(stream, before_scan, 0));
    k_encode_scan<<<scan_ctas, kScanTile, 0, stream>>>(p);
    if (int rc = launch_check("k_encode_scan"))
        return rc;
    CUDA_TRY(cudaMemcpyAsync(d_used, p.residues, 8, cudaMemcpyDeviceToDevice, stream)); // the new fill level (see k_encode_scan)
    // The fill level this chunk leaves behind must be captured BEFORE the next chunk's scan (on the
    // other compute lane) may overwrite *d_used: copy it out now and only then release the event.
    if (h_fill_after)
        CUDA_TRY(cudaMemcpyAsync(h_fill_after, d_used, 8, cudaMemcpyDeviceToHost, stream));
    if (after_scan)
        CUDA_TRY(cudaEventRecord(after_scan, stream));
    if (d_container) { // byte-packed .sela stream instead of the word arena
        k_encode_gather_container<<<(unsigned)((n_sub + 7) / 8), 256, 0, stream>>>(p, d_container, sub_base);
        return launch_check("k_encode_gather_container");
    }
    k_encode_gather<<<(unsigned)((n_sub + 7) / 8), 256, 0, stream>>>(p);
    return launch_check("k_encode_gather");
}

// K5 launch: 64-word rings (8.3 KB per warp), eight parser steps per batch.
int launch_rice_decode(const DecodeParams &p, int which, cudaStream_t stream)
{
    const size_t n_sub = (size_t)p.n_frames * p.channels;
    const unsigned blocks = (unsigned)((n_sub + 32 * kRiceWarps - 1) / (32 * kRiceWarps));
    k_rice_decode<kRiceRing, kRiceBatch><<<blocks, 32 * kRiceWarps, 0, stream>>>(p, which);
    return launch_check(which ? "k_rice_decode(res)" : "k_rice_decode(refl)");
}

// Residue streams (K5 proper).  Large batches: one lane per stream through k_rice_decode_vc.  Smaller
// ones: every stream is cut into S parts first (k_rice_split_index), so that a batch of BASELINE's
// size still fills the machine.  aux: n_sub * 64 bytes (split table + per-stream flags).
int rice_split_log2(size_t n_sub)
{
    // SELAB200_RICE_SPLIT = 0 (first-generation kernel only), 1, 2, 4, 8, 16 overrides the choice; it exists for
    // tests and measurement, which reach every S on small inputs.
    if (const char *env = std::getenv("SELAB200_RICE_SPLIT")) {
        const long v = std::atol(env);
        if (v <= 0)
            return -1;
        int l = 0;
        while ((1 << (l + 1)) <= v && l < 4)
            l++;
        return l;
    }
    // Measured on B200 (profiles/r02_rice_decode_roofline.json): from about 12 000 streams up one lane per stream
    // (S = 1) through k_rice_decode_vc is fastest -- the two split passes cost more than the extra warps bring
    // once every SM has a few warps of its own; below that the machine is starved and cutting the streams
    // wins (500 streams: S = 16 is 3.5x the first-generation kernel, 8 000 streams: S = 8 is 1.9x).
    if (n_sub >= 12000)
        return 0;
    int l = 0;
    while (l < 4 && (n_sub << l) < (size_t)40000)
        l++;
    return l;
}

template <int LOG2S>
int launch_split_index(const RiceVsParams &q, size_t n_sub, cudaStream_t stream)
{
    const unsigned blocks = (unsigned)(((n_sub << LOG2S) + 32 * kVsWarps - 1) / (32 * kVsWarps));
    constexpr size_t smem = split_smem_bytes<32>();
    if (int rc = set_smem(k_rice_split_index<LOG2S, 32, 16>, smem))
        return rc;
    k_rice_split_index<LOG2S, 32, 16><<<blocks, 32 * kVsWarps, smem, stream>>>(q);
    return launch_check("k_rice_split_index");
}

int launch_rice_residues(const DecodeParams &p, void *aux, cudaStream_t stream)
{
    const size_t n_sub = (size_t)p.n_frames * p.channels;
    const int log2s = rice_split_log2(n_sub);
    if (log2s < 0 || (reinterpret_cast<uintptr_t>(p.ws_res) & 15) != 0)
        return launch_rice_decode(p, 1, stream);
    RiceVsParams q;
    q.descs = p.descs;
    q.n_sub = (uint32_t)n_sub;
    q.channels = p.channels;
    q.words = p.words;
    q.n_words = p.n_words;
    q.out = p.ws_res;
    q.table = static_cast<uint32_t *>(aux);
    q.flags = q.table + n_sub * 15;
    q.status = p.status;
    int rc = 0;
    switch (log2s) {
    case 0: CUDA_TRY(cudaMemsetAsync(q.flags, 0, n_sub * 4, stream)); break;
    case 1: rc = launch_split_index<1>(q, n_sub, stream); break;
    case 2: rc = launch_split_index<2>(q, n_sub, stream); break;
    case 3: rc = launch_split_index<3>(q, n_sub, stream); break;
    default: rc = launch_split_index<4>(q, n_sub, stream); break;
    }
    if (rc)
        return rc;
    const size_t n_vs = n_sub << log2s;
    const unsigned vs_blocks = (unsigned)((n_vs + 32 * kVsWarps - 1) / (32 * kVsWarps));
    constexpr size_t smem = vc_smem_bytes<32>();
    if (int rc2 = set_smem(k_rice_decode_vc<16, 32>, smem))
        return rc2;
    k_rice_decode_vc<16, 32><<<vs_blocks, 32 * kVsWarps, smem, stream>>>(q, log2s);
    if (int rc2 = launch_check("k_rice_decode_vc"))
        return rc2;
    DecodeParams pf = p; // whatever was flagged: the general lane-per-stream parser decodes it again
    pf.rice_flags = q.flags;
    return launch_rice_decode(pf, 1, stream);
}

// The inputs every decode kernel reads; the workspace and output pointers are left null for the caller.
DecodeParams decode_params(const selab200_subframe_desc *d_descs, uint32_t n_frames, uint32_t channels,
                           const uint32_t *d_words, size_t n_words, int32_t *d_status)
{
    DecodeParams p = {};
    p.descs = d_descs;
    p.n_frames = n_frames;
    p.channels = channels;
    p.words = d_words;
    p.n_words = n_words;
    p.status = d_status;
    return p;
}

int decode_device(const selab200_subframe_desc *d_descs, uint32_t n_frames, uint32_t channels,
                  const uint32_t *d_words, size_t n_words, int16_t *d_pcm, int32_t *d_status, void *d_ws,
                  size_t ws_bytes, cudaStream_t stream, bool fresh = true)
{
    if (int rc = check_channels(channels))
        return rc;
    if (ws_bytes < selab200_decode_workspace_bytes(n_frames, channels))
        return fail(SELAB200_ERR_ARGUMENT, "decode workspace too small");
    if (fresh)
        CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int32_t), stream));
    if (n_frames == 0)
        return 0;
    const size_t n_sub = (size_t)n_frames * channels;
    DecodeParams p = decode_params(d_descs, n_frames, channels, d_words, n_words, d_status);
    p.pcm_out = d_pcm;
    p.ws_q = static_cast<int32_t *>(d_ws);
    p.ws_res = reinterpret_cast<int32_t *>(static_cast<char *>(d_ws) + align256(n_sub * 128 * 4));
    p.order_index = reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(p.ws_res) + align256(n_sub * kFrame * 4));
    void *rice_aux = reinterpret_cast<char *>(p.order_index) + align256((n_sub + 16) * 4);
    const size_t n_slots = (n_sub + 12 + 3) / 4 * 4; // every class segment starts on a warp boundary
    CUDA_TRY(cudaMemsetAsync(p.order_index, 0xff, n_slots * 4, stream));
    const unsigned class_ctas = (unsigned)((n_sub + kScanTile - 1) / kScanTile);
    k_decode_class_counts<<<class_ctas, kScanTile, 0, stream>>>(p, static_cast<ClassCounts *>(rice_aux));
    if (int rc = launch_check("k_decode_class_counts"))
        return rc;
    k_decode_classify<<<class_ctas, kScanTile, 0, stream>>>(p, static_cast<const ClassCounts *>(rice_aux));
    if (int rc = launch_check("k_decode_classify"))
        return rc;
    if (int rc = launch_rice_decode(p, 0, stream))
        return rc;
    if (int rc = launch_rice_residues(p, rice_aux, stream))
        return rc;
    p.fallback_only = 1;
    k_synthesise_quad<<<(unsigned)(n_slots / 4), 32, 0, stream>>>(p);
    if (int rc = launch_check("k_synthesise_quad"))
        return rc;
    if (channels == 2) { // every stereo frame is handled by the batch kernel + the difference fix-up
        k_diff_fixup<<<n_frames, 128, 0, stream>>>(p);
        return launch_check("k_diff_fixup");
    }
    const size_t smem = synthesise_smem_bytes(channels);
    if (int rc = set_smem(k_synthesise, smem))
        return rc;
    k_synthesise<<<n_frames, 32 * ((channels + 1) / 2), smem, stream>>>(p);
    return launch_check("k_synthesise");
}

int read_status(Context &c, cudaStream_t stream, const int32_t *d_status)
{
    CUDA_TRY(cudaMemcpyAsync(c.h_small, d_status, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    if (c.h_small[0] != 0)
        return fail(c.h_small[0], "%s", status_text(c.h_small[0]));
    return 0;
}

} // namespace

extern "C" {

int selab200_abi_version(void) { return SELAB200_ABI_VERSION; }
const char *selab200_last_error(void) { return g_error; }
uint64_t selab200_launch_count(void) { return g_launches.load(); }

// (g_mutex held)
static int init_slot(Context &c, int device)
{
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(SELAB200_ERR_NO_DEVICE, "device %d is sm_%d%d; this build targets sm_100a only", device,
                    prop.major, prop.minor);
    CUDA_TRY(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&c.s_h2d, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&c.s_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < kLanes; i++)
        CUDA_TRY(cudaStreamCreateWithFlags(&c.s_compute[i], cudaStreamNonBlocking));
    for (int i = 0; i < kMaxChunks; i++) {
        CUDA_TRY(cudaEventCreateWithFlags(&c.ev_h2d[i], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&c.ev_done[i], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&c.ev_scan[i], cudaEventDisableTiming));
    }
    CUDA_TRY(cudaEventCreateWithFlags(&c.ev_reset, cudaEventDisableTiming));
    c.events = true;
    CUDA_TRY(cudaMallocHost(reinterpret_cast<void **>(&c.h_small), 64));
    CUDA_TRY(cudaMallocHost(reinterpret_cast<void **>(&c.h_totals), (kMaxChunks + 1) * 8));
    if (int rc = c.small.ensure(256))
        return rc;
    c.device = device;
    c.ready = true;
    return 0;
}

static void shutdown_slot(Context &c)
{
    if (c.device >= 0)
        cudaSetDevice(c.device);
    if (c.stream)
        cudaStreamSynchronize(c.stream);
    for (ContainerBuffers &b : c.spare)
        b.destroy();
    c.spare.clear();
    c.in.release();
    c.descs.release();
    c.words.release();
    c.work.release();
    for (int i = 0; i < kLanes; i++)
        c.lane_work[i].release();
    c.aux.release();
    c.small.release();
    if (c.h_small)
        cudaFreeHost(c.h_small);
    if (c.h_totals)
        cudaFreeHost(c.h_totals);
    for (cudaStream_t st : {c.stream, c.s_h2d, c.s_d2h})
        if (st)
            cudaStreamDestroy(st);
    for (int i = 0; i < kLanes; i++)
        if (c.s_compute[i])
            cudaStreamDestroy(c.s_compute[i]);
    if (c.events) {
        for (int i = 0; i < kMaxChunks; i++) {
            cudaEventDestroy(c.ev_h2d[i]);
            cudaEventDestroy(c.ev_done[i]);
            cudaEventDestroy(c.ev_scan[i]);
        }
        cudaEventDestroy(c.ev_reset);
    }
    c = Context(); // not ready, no device, every handle null
}

static void shutdown_all()
{
    for (int i = 0; i < g_n_ctx; i++)
        shutdown_slot(g_slots[i]);
    g_n_ctx = 0;
    g_last_rice_slot = -1;
}

int selab200_init_devices(int count, const int *devices)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    if (count < 1 || count > kMaxDevices || !devices)
        return fail(SELAB200_ERR_ARGUMENT, "device count must be in [1, %d]", kMaxDevices);
    bool same = count == g_n_ctx;
    for (int i = 0; same && i < count; i++)
        same = g_slots[i].ready && g_slots[i].device == devices[i];
    if (same)
        return 0;
    int have = 0;
    cudaError_t e = cudaGetDeviceCount(&have);
    if (e != cudaSuccess || have == 0)
        return fail(SELAB200_ERR_NO_DEVICE, "no CUDA device available (%s); this library has no CPU path",
                    e == cudaSuccess ? "count == 0" : cudaGetErrorString(e));
    for (int i = 0; i < count; i++) {
        if (devices[i] < 0 || devices[i] >= have)
            return fail(SELAB200_ERR_ARGUMENT, "device %d out of range (have %d)", devices[i], have);
        for (int j = 0; j < i; j++)
            if (devices[j] == devices[i])
                return fail(SELAB200_ERR_ARGUMENT, "device %d listed twice", devices[i]);
    }
    // a different set of devices than before: everything the old contexts own (streams, events, pools) lives on
    // the old devices, so they are torn down completely before the new ones are set up
    shutdown_all();
    for (int i = 0; i < count; i++)
        if (int rc = init_slot(g_slots[i], devices[i])) {
            g_n_ctx = i + 1;
            return fail_after_cleanup(rc, shutdown_all);
        }
    g_n_ctx = count;
    CUDA_TRY(cudaSetDevice(g_slots[0].device));
    return 0;
}

int selab200_init(int device) { return selab200_init_devices(1, &device); }

int selab200_device_count(void)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    return g_n_ctx;
}

void selab200_shutdown(void)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    shutdown_all();
}

void *selab200_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
        fail(SELAB200_ERR_CUDA, "cudaMallocHost(%zu) failed", bytes);
        return nullptr;
    }
    return p;
}

void selab200_host_free(void *p)
{
    if (p)
        cudaFreeHost(p);
}

size_t selab200_encode_words_bound(uint32_t n_frames, uint32_t channels)
{
    // A subframe never exceeds its scratch slot (larger streams are refused with
    // SELAB200_ERR_RANGE): residues <= 1568 words (24.5 bits/sample), coefficients <= 32.
    return (size_t)n_frames * channels * kSlotWords + 64;
}

size_t selab200_encode_workspace_bytes(uint32_t n_frames, uint32_t channels)
{
    const size_t n_units = encode_units(n_frames, channels);
    return align256(n_units * sizeof(UnitRecord)) + align256(n_units * (size_t)kSlotWords * 4) +
           n_units * (size_t)kFrame * 4 + 256;
}

size_t selab200_decode_workspace_bytes(uint32_t n_frames, uint32_t channels)
{
    const size_t n_sub = (size_t)n_frames * channels;
    return align256(n_sub * 128 * 4) + align256(n_sub * kFrame * 4) + align256((n_sub + 16) * 4) + align256(n_sub * 64) + 256;
}

int selab200_encode_frames_device(const int16_t *d_pcm, uint32_t n_frames, uint32_t channels,
                                  selab200_subframe_desc *d_descs, uint32_t *d_words, size_t words_capacity,
                                  uint64_t *d_words_used, int32_t *d_status, void *d_workspace,
                                  size_t workspace_bytes, void *stream)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready_for(d_pcm, c))
        return rc;
    if (!d_pcm || !d_descs || !d_words || !d_words_used || !d_status || !d_workspace)
        return fail(SELAB200_ERR_ARGUMENT, "null device pointer");
    return encode_device(d_pcm, n_frames, channels, d_descs, d_words, words_capacity, d_words_used, d_status,
                         d_workspace, workspace_bytes, (cudaStream_t)stream);
}

int selab200_decode_frames_device(const selab200_subframe_desc *d_descs, uint32_t n_frames, uint32_t channels,
                                  const uint32_t *d_words, size_t n_words, int16_t *d_pcm_out, int32_t *d_status,
                                  void *d_workspace, size_t workspace_bytes, void *stream)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready_for(d_descs, c))
        return rc;
    if (!d_descs || !d_words || !d_pcm_out || !d_status || !d_workspace)
        return fail(SELAB200_ERR_ARGUMENT, "null device pointer");
    return decode_device(d_descs, n_frames, channels, d_words, n_words, d_pcm_out, d_status, d_workspace,
                         workspace_bytes, (cudaStream_t)stream);
}

int selab200_rice_decode_frames_device(const selab200_subframe_desc *d_descs, uint32_t n_frames, uint32_t channels,
                                       const uint32_t *d_words, size_t n_words, int32_t *d_residues,
                                       int32_t *d_status, void *stream)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready_for(d_descs, c))
        return rc;
    if (!d_descs || !d_words || !d_residues || !d_status)
        return fail(SELAB200_ERR_ARGUMENT, "null device pointer");
    if (int rc = check_channels(channels))
        return rc;
    CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int32_t), (cudaStream_t)stream));
    if (n_frames == 0)
        return 0;
    DecodeParams p = decode_params(d_descs, n_frames, channels, d_words, n_words, d_status);
    p.ws_res = d_residues;
    if (int rc = c->aux.ensure((size_t)n_frames * channels * 64 + 256))
        return rc;
    c->last_rice_n_sub = (size_t)n_frames * channels;
    c->last_rice_stream = (cudaStream_t)stream;
    g_last_rice_slot = (int)(c - g_slots);
    return launch_rice_residues(p, c->aux.ptr, (cudaStream_t)stream);
}

int selab200_rice_decode_flagged(uint32_t *n_flagged)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready(c))
        return rc;
    if (!n_flagged)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    *n_flagged = 0;
    if (g_last_rice_slot >= 0 && g_slots[g_last_rice_slot].ready) { // the device the last call ran on, which need not be the primary
        c = &g_slots[g_last_rice_slot];
        if (int rc = use_device(*c))
            return rc;
    }
    const size_t n = c->last_rice_n_sub;
    if (n == 0 || c->aux.bytes < n * 64)
        return 0;
    std::vector<uint32_t> flags(n);
    CUDA_TRY(cudaStreamSynchronize(c->last_rice_stream));
    CUDA_TRY(cudaMemcpy(flags.data(), static_cast<uint32_t *>(c->aux.ptr) + n * 15, n * 4, cudaMemcpyDeviceToHost));
    uint32_t count = 0;
    for (uint32_t f : flags)
        count += f != 0;
    *n_flagged = count;
    return 0;
}

} // extern "C"

// Bytes of container in front of frame f when `words` Rice words precede it.
static unsigned long long container_frame_byte(unsigned long long f, uint32_t channels, unsigned long long words)
{
    return kContainerHeaderBytes + 4 * f + (unsigned long long)kSubframeHeaderBytes * f * channels + 4 * words;
}

// ---- pipelined host-buffer calls ----------------------------------------------------------------
//
// Encode, decode and container decode run in chunks of frames (plan_chunks) over three engines:
//   s_h2d      PCM (encode) / descriptors + words (decode) of chunk c+1 .. go up
//   s_compute  the compute lanes run the kernels of chunk c (tails of one chunk overlap the head of
//              the next); encode alternates two lanes whose scans are chained by events, because each
//              needs the arena fill level its predecessor left in *d_used
//   s_d2h      results of chunk c-1 come down
// With pinned host buffers (selab200_host_alloc) the three overlap; pageable memory works
// but serialises inside the driver.

// Device views of a pipelined call's buffers.
struct PipelineViews {
    int32_t *status;               // Context::small, bytes 0..3
    uint64_t *used;                // Context::small, bytes 8..15: arena fill level (encode)
    int16_t *pcm;                  // Context::in
    selab200_subframe_desc *descs; // Context::descs
    uint32_t *words;               // Context::words
};

// The start every pipelined call shares: grows the context's buffers for the frames of `plan` (`words_bytes` of
// word arena or container image, `ws_bytes` of workspace on each of the first `lanes` lanes the chunks use),
// then clears the status word and the fill level on lane 0 and makes every lane wait for that.  The caller
// holds a PipelineDrain.
static int begin_pipeline(Context &c, const ChunkPlan &plan, uint32_t channels, size_t words_bytes, size_t ws_bytes,
                          uint32_t lanes, PipelineViews &v)
{
    const size_t n_sub = (size_t)plan.start.back() * channels;
    if (int rc = c.in.ensure(n_sub * kFrame * 2)) return rc;
    if (int rc = c.descs.ensure(n_sub * sizeof(selab200_subframe_desc))) return rc;
    if (int rc = c.words.ensure(words_bytes)) return rc;
    for (uint32_t i = 0; i < lanes && i < plan.chunks(); i++)
        if (int rc = c.lane_work[i].ensure(ws_bytes)) return rc;
    v.status = static_cast<int32_t *>(c.small.ptr);
    v.used = reinterpret_cast<uint64_t *>(static_cast<char *>(c.small.ptr) + 8);
    v.pcm = static_cast<int16_t *>(c.in.ptr);
    v.descs = static_cast<selab200_subframe_desc *>(c.descs.ptr);
    v.words = static_cast<uint32_t *>(c.words.ptr);

    CUDA_TRY(cudaMemsetAsync(c.small.ptr, 0, 16, c.s_compute[0]));
    CUDA_TRY(cudaEventRecord(c.ev_reset, c.s_compute[0]));
    for (int i = 1; i < kLanes; i++)
        CUDA_TRY(cudaStreamWaitEvent(c.s_compute[i], c.ev_reset, 0));
    return 0;
}

// The pipelined encoder over host buffers.  Two output forms: descriptors + word arena
// (descs/words), or the byte-packed container (`container`, descs == words == nullptr) whose
// device image lives in c.words.
// `defer`: leave the word arena / container body on the device (c.words) instead of copying it out chunk by
// chunk -- the multi-device driver places every device's block once the sizes of the blocks before it are known.
// With `defer`, `container` is only a flag (any non-null value selects the byte-packed form).
static int encode_host(Context &c, const int16_t *pcm, uint32_t n_frames, uint32_t channels,
                       selab200_subframe_desc *descs, uint32_t *words, size_t words_capacity, size_t *words_used,
                       uint8_t *container, bool defer = false)
{
    *words_used = 0;
    if (n_frames == 0)
        return 0;
    PipelineDrain drain{c};
    const ChunkPlan plan = plan_chunks(n_frames);
    const uint32_t n_chunks = plan.chunks();
    const size_t frame_bytes = (size_t)channels * kFrame * 2;
    constexpr int kEncLanes = 2;
    PipelineViews v;
    if (int rc = begin_pipeline(c, plan, channels, container_frame_byte(n_frames, channels, words_capacity) + 64,
                                selab200_encode_workspace_bytes(plan.max_frames, channels), kEncLanes, v))
        return rc;
    for (uint32_t k = 0; k < n_chunks; k++) {
        const uint32_t f0 = plan.start[k], nf = plan.start[k + 1] - f0;
        CUDA_TRY(cudaMemcpyAsync(v.pcm + (size_t)f0 * channels * kFrame, pcm + (size_t)f0 * channels * kFrame,
                                 nf * frame_bytes, cudaMemcpyHostToDevice, c.s_h2d));
        CUDA_TRY(cudaEventRecord(c.ev_h2d[k], c.s_h2d));
        cudaStream_t cs = c.s_compute[k % kEncLanes];
        DeviceBuffer &ws = c.lane_work[k % kEncLanes];
        CUDA_TRY(cudaStreamWaitEvent(cs, c.ev_h2d[k], 0));
        if (int rc = encode_device(v.pcm + (size_t)f0 * channels * kFrame, nf, channels, v.descs + (size_t)f0 * channels,
                                   v.words, words_capacity, v.used, v.status, ws.ptr, ws.bytes, cs, false,
                                   k ? c.ev_scan[k - 1] : nullptr, c.ev_scan[k], &c.h_totals[k + 1],
                                   container ? static_cast<uint8_t *>(c.words.ptr) : nullptr,
                                   (unsigned long long)f0 * channels))
            return rc;
        CUDA_TRY(cudaEventRecord(c.ev_done[k], cs));
    }
    c.h_totals[0] = 0;
    for (uint32_t k = 0; k < n_chunks; k++) {
        const uint32_t f0 = plan.start[k], nf = plan.start[k + 1] - f0;
        CUDA_TRY(cudaEventSynchronize(c.ev_done[k]));
        const unsigned long long lo = c.h_totals[k], hi = c.h_totals[k + 1];
        if (hi > words_capacity || hi < lo)
            break; // capacity exceeded: reported through the status word below
        if (!container)
            CUDA_TRY(cudaMemcpyAsync(descs + (size_t)f0 * channels, v.descs + (size_t)f0 * channels,
                                     (size_t)nf * channels * sizeof(selab200_subframe_desc), cudaMemcpyDeviceToHost,
                                     c.s_d2h));
        if (defer)
            continue;
        if (container) {
            const unsigned long long b0 = container_frame_byte(f0, channels, lo);
            const unsigned long long b1 = container_frame_byte(f0 + nf, channels, hi);
            CUDA_TRY(cudaMemcpyAsync(container + b0, static_cast<uint8_t *>(c.words.ptr) + b0, b1 - b0,
                                     cudaMemcpyDeviceToHost, c.s_d2h));
        } else {
            CUDA_TRY(cudaMemcpyAsync(words + lo, v.words + lo, (hi - lo) * 4, cudaMemcpyDeviceToHost, c.s_d2h));
        }
    }
    for (int i = 0; i < kEncLanes; i++)
        CUDA_TRY(cudaStreamSynchronize(c.s_compute[i]));
    CUDA_TRY(cudaMemcpyAsync(c.h_small, c.small.ptr, 16, cudaMemcpyDeviceToHost, c.s_d2h));
    CUDA_TRY(cudaStreamSynchronize(c.s_d2h));
    uint64_t used;
    memcpy(&used, c.h_small + 2, 8);
    *words_used = (size_t)used; // for CAPACITY: the size the caller needs
    if (c.h_small[0] != 0)
        return fail(c.h_small[0], "%s", status_text(c.h_small[0]));
    return 0;
}

// The chunk loop of both decode pipelines (decode_host and the container decode).  `stage(k, f0, nf, lane)`
// brings chunk k, frames [f0, f0 + nf) of the call, onto the device: its descriptors to v.descs + f0 * channels
// and the words they reference into the arena, with `lane` made to wait for them.  The loop decodes the chunk
// on that lane and downloads its PCM to pcm_out, which holds the call's frames from its first.
// Every chunk gets its own compute lane (up to kLanes): the Rice kernel is one lane per stream and
// latency-bound (about 0.4 ms however small the chunk), so the chunks' Rice kernels must overlap
// each other and the synthesis kernels of earlier chunks rather than queue up.
template <typename Stage>
static int decode_chunks(Context &c, const ChunkPlan &plan, uint32_t channels, const PipelineViews &v,
                         const uint32_t *d_words, size_t n_words, int16_t *pcm_out, Stage stage)
{
    const size_t frame_bytes = (size_t)channels * kFrame * 2;
    for (uint32_t k = 0; k < plan.chunks(); k++) {
        const uint32_t f0 = plan.start[k], nf = plan.start[k + 1] - f0;
        cudaStream_t cs = c.s_compute[k % kLanes];
        DeviceBuffer &ws = c.lane_work[k % kLanes];
        if (int rc = stage(k, f0, nf, cs))
            return rc;
        if (int rc = decode_device(v.descs + (size_t)f0 * channels, nf, channels, d_words, n_words,
                                   v.pcm + (size_t)f0 * channels * kFrame, v.status, ws.ptr, ws.bytes, cs, false))
            return rc;
        CUDA_TRY(cudaEventRecord(c.ev_done[k], cs));
        CUDA_TRY(cudaStreamWaitEvent(c.s_d2h, c.ev_done[k], 0));
        CUDA_TRY(cudaMemcpyAsync(pcm_out + (size_t)f0 * channels * kFrame, v.pcm + (size_t)f0 * channels * kFrame,
                                 nf * frame_bytes, cudaMemcpyDeviceToHost, c.s_d2h));
    }
    return read_status(c, c.s_d2h, v.status);
}

static int decode_host(Context &c, const selab200_subframe_desc *descs, uint32_t n_frames, uint32_t channels,
                       const uint32_t *words, size_t n_words, int16_t *pcm_out)
{
    if (n_frames == 0)
        return 0;
    PipelineDrain drain{c};
    const ChunkPlan plan = plan_chunks(n_frames);
    PipelineViews v;
    if (int rc = begin_pipeline(c, plan, channels, n_words * 4 + 16,
                                selab200_decode_workspace_bytes(plan.max_frames, channels), kLanes, v))
        return rc;
    return decode_chunks(c, plan, channels, v, v.words, n_words, pcm_out,
                         [&](uint32_t k, uint32_t f0, uint32_t nf, cudaStream_t cs) {
        // the words this chunk's descriptors reference (descriptors need not be in arena order)
        unsigned long long lo = ~0ull, hi = 0;
        const selab200_subframe_desc *dc = descs + (size_t)f0 * channels;
        for (size_t i = 0; i < (size_t)nf * channels; i++) {
            const unsigned long long a0 = dc[i].refl_offset, a1 = a0 + dc[i].refl_words;
            const unsigned long long b0 = dc[i].res_offset, b1 = b0 + dc[i].res_words;
            if (a1 <= n_words && b1 <= n_words) { // out-of-range descriptors are rejected on the device
                lo = a0 < lo ? a0 : lo;
                lo = b0 < lo ? b0 : lo;
                hi = a1 > hi ? a1 : hi;
                hi = b1 > hi ? b1 : hi;
            }
        }
        CUDA_TRY(cudaMemcpyAsync(v.descs + (size_t)f0 * channels, dc, (size_t)nf * channels * sizeof(*dc),
                                 cudaMemcpyHostToDevice, c.s_h2d));
        if (hi > lo)
            CUDA_TRY(cudaMemcpyAsync(v.words + lo, words + lo, (hi - lo) * 4, cudaMemcpyHostToDevice, c.s_h2d));
        CUDA_TRY(cudaEventRecord(c.ev_h2d[k], c.s_h2d));
        CUDA_TRY(cudaStreamWaitEvent(cs, c.ev_h2d[k], 0));
        return 0;
    });
}

// ---- every initialised device at once ----------------------------------------------------------
//
// Frames are independent (src/sela/encoder.cpp:40-92 hands contiguous ranges of them to its threads); with more
// than one device the host-buffer calls do the same with the devices: device d codes the contiguous block
// frame_block(d) on a worker thread of its own, with its own context (streams, pools), straight from / into
// disjoint ranges of the caller's buffers.  Only the encoder needs a second step: where a block's words land
// depends on the sizes of the blocks before it, so the workers leave the words on their devices and the
// calling thread copies them out (all devices at once) when every size is known, re-basing the descriptors'
// offsets on the way.  The byte-packed container works the same way: a block's body is position independent
// (DESIGN.md 6).
struct DevicePart {
    uint32_t f0 = 0, nf = 0;
    int rc = 0;
    size_t used = 0;
    char err[sizeof g_error] = "";
};

static std::vector<DevicePart> device_parts(uint32_t n_frames)
{
    // n/D frames each, the last device takes the rest: the reference's thread split (src/sela/encoder.cpp:58-73)
    std::vector<DevicePart> parts((size_t)g_n_ctx);
    const uint32_t per = n_frames / (uint32_t)g_n_ctx;
    for (int d = 0; d < g_n_ctx; d++) {
        parts[d].f0 = per * d;
        parts[d].nf = d == g_n_ctx - 1 ? n_frames - per * d : per;
    }
    return parts;
}

static bool use_all_devices(uint32_t n_frames)
{
    return g_n_ctx > 1 && n_frames >= 256u * (uint32_t)g_n_ctx;
}

// Runs work(context, part) for every device on a thread of its own, with that device current.
template <typename F>
static int run_on_devices(std::vector<DevicePart> &parts, F work)
{
    std::vector<std::thread> threads;
    for (int d = 0; d < g_n_ctx; d++)
        threads.emplace_back([&, d] {
            Context &c = g_slots[d];
            DevicePart &p = parts[d];
            p.rc = use_device(c);
            if (!p.rc)
                p.rc = work(c, p);
            if (p.rc)
                memcpy(p.err, g_error, sizeof p.err);
        });
    for (std::thread &t : threads)
        t.join();
    cudaSetDevice(g_slots[0].device);
    for (const DevicePart &p : parts)
        if (p.rc) {
            memcpy(g_error, p.err, sizeof g_error);
            return p.rc;
        }
    return 0;
}

static int encode_all_devices(const int16_t *pcm, uint32_t n_frames, uint32_t channels, selab200_subframe_desc *descs,
                              uint32_t *words, size_t words_capacity, size_t *words_used, uint8_t *container)
{
    std::vector<DevicePart> parts = device_parts(n_frames);
    const size_t per_frame = (size_t)channels * kFrame;
    const int rc = run_on_devices(parts, [&](Context &c, DevicePart &p) {
        return encode_host(c, pcm + p.f0 * per_frame, p.nf, channels, descs ? descs + (size_t)p.f0 * channels : nullptr,
                           nullptr, selab200_encode_words_bound(p.nf, channels), &p.used, container, true);
    });
    size_t total = 0;
    for (const DevicePart &p : parts)
        total += p.used;
    *words_used = total;
    if (rc)
        return rc;
    if (total > words_capacity)
        return fail(SELAB200_ERR_CAPACITY, "%s", status_text(SELAB200_ERR_CAPACITY));
    size_t base = 0;
    for (int d = 0; d < g_n_ctx; d++) { // every device's block goes out at once, each over its own link
        Context &c = g_slots[d];
        const DevicePart &p = parts[d];
        if (int rc2 = use_device(c))
            return rc2;
        if (container) {
            const size_t body = (size_t)container_frame_byte(p.nf, channels, p.used) - kContainerHeaderBytes;
            const size_t at = (size_t)container_frame_byte(p.f0, channels, base);
            if (body)
                CUDA_TRY(cudaMemcpyAsync(container + at, static_cast<uint8_t *>(c.words.ptr) + kContainerHeaderBytes, body,
                                         cudaMemcpyDeviceToHost, c.s_d2h));
        } else if (p.used) {
            CUDA_TRY(cudaMemcpyAsync(words + base, c.words.ptr, p.used * 4, cudaMemcpyDeviceToHost, c.s_d2h));
        }
        base += p.used;
    }
    if (!container) { // meanwhile: descriptor offsets from block-local to file order
        size_t b = 0;
        for (const DevicePart &p : parts) {
            if (b)
                for (size_t i = (size_t)p.f0 * channels; i < (size_t)(p.f0 + p.nf) * channels; i++) {
                    descs[i].refl_offset += b;
                    descs[i].res_offset += b;
                }
            b += p.used;
        }
    }
    int rc2 = 0;
    for (int d = 0; d < g_n_ctx; d++) {
        Context &c = g_slots[d];
        cudaSetDevice(c.device);
        cudaError_t e = cudaStreamSynchronize(c.s_d2h);
        if (e != cudaSuccess && !rc2)
            rc2 = fail(SELAB200_ERR_CUDA, "download from device %d failed: %s", c.device, cudaGetErrorString(e));
    }
    cudaSetDevice(g_slots[0].device);
    return rc2;
}

static int decode_all_devices(const selab200_subframe_desc *descs, uint32_t n_frames, uint32_t channels,
                              const uint32_t *words, size_t n_words, int16_t *pcm_out)
{
    std::vector<DevicePart> parts = device_parts(n_frames);
    const size_t per_frame = (size_t)channels * kFrame;
    return run_on_devices(parts, [&](Context &c, DevicePart &p) {
        return decode_host(c, descs + (size_t)p.f0 * channels, p.nf, channels, words, n_words, pcm_out + p.f0 * per_frame);
    });
}

extern "C" {

int selab200_encode_frames(const int16_t *pcm, uint32_t n_frames, uint32_t channels,
                           selab200_subframe_desc *descs, uint32_t *words, size_t words_capacity,
                           size_t *words_used)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready(c))
        return rc;
    if (!pcm || !descs || !words || !words_used)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    if (int rc = check_channels(channels))
        return rc;
    if (use_all_devices(n_frames))
        return encode_all_devices(pcm, n_frames, channels, descs, words, words_capacity, words_used, nullptr);
    return encode_host(*c, pcm, n_frames, channels, descs, words, words_capacity, words_used, nullptr);
}

size_t selab200_container_bound(uint32_t n_frames, uint32_t channels)
{
    return (size_t)container_frame_byte(n_frames, channels, selab200_encode_words_bound(n_frames, channels));
}

int selab200_encode_container(const int16_t *pcm, uint32_t n_frames, uint32_t channels, uint32_t sample_rate,
                              uint16_t bits_per_sample, uint8_t *container, size_t capacity, size_t *bytes_used)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready(c))
        return rc;
    if ((!pcm && n_frames) || !container || !bytes_used)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    if (int rc = check_channels(channels))
        return rc;
    const unsigned long long fixed = container_frame_byte(n_frames, channels, 0);
    *bytes_used = (size_t)fixed;
    if (capacity < fixed)
        return fail(SELAB200_ERR_CAPACITY, "container buffer too small: %zu bytes, need more than %llu", capacity, fixed);
    // file::SelaFile::writeToFile, header part (src/file/sela_file.cpp:107-112)
    const uint8_t header[15] = {'S', 'e', 'L', 'a',
                                (uint8_t)sample_rate, (uint8_t)(sample_rate >> 8), (uint8_t)(sample_rate >> 16), (uint8_t)(sample_rate >> 24),
                                (uint8_t)bits_per_sample, (uint8_t)(bits_per_sample >> 8), (uint8_t)channels,
                                (uint8_t)n_frames, (uint8_t)(n_frames >> 8), (uint8_t)(n_frames >> 16), (uint8_t)(n_frames >> 24)};
    memcpy(container, header, sizeof header);
    size_t words_used = 0;
    const int rc = use_all_devices(n_frames)
                       ? encode_all_devices(pcm, n_frames, channels, nullptr, nullptr, (size_t)((capacity - fixed) / 4), &words_used, container)
                       : encode_host(*c, pcm, n_frames, channels, nullptr, nullptr, (size_t)((capacity - fixed) / 4), &words_used, container);
    *bytes_used = (size_t)container_frame_byte(n_frames, channels, words_used);
    return rc;
}

int selab200_decode_frames(const selab200_subframe_desc *descs, uint32_t n_frames, uint32_t channels,
                           const uint32_t *words, size_t n_words, int16_t *pcm_out)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready(c))
        return rc;
    if (!descs || !pcm_out || (!words && n_words))
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    if (int rc = check_channels(channels))
        return rc;
    if (use_all_devices(n_frames))
        return decode_all_devices(descs, n_frames, channels, words, n_words, pcm_out);
    return decode_host(*c, descs, n_frames, channels, words, n_words, pcm_out);
}

// ---- .sela container, decode side ----------------------------------------------------------

} // extern "C"

struct selab200_container {
    const uint8_t *bytes = nullptr;
    size_t n_bytes = 0;
    selab200_container_info info{};
    ContainerBuffers buf;
    size_t piece_bytes = 0;
    int n_pieces = 0;
};

namespace {

// file::SelaFile::readFromFile (src/file/sela_file.cpp:19-103) without the copies: validates the
// header, then hops from frame to frame.  With `descs` it also emits one descriptor per subframe,
// arena offsets assigned in file order.  Messages match the host mirror's reader.
int walk_container(const uint8_t *b, size_t n, selab200_container_info *info,
                   std::vector<selab200_subframe_desc> *descs, uint64_t *frame_bytes = nullptr,
                   size_t frame_capacity = 0)
{
    memset(info, 0, sizeof *info);
    if (n < 15)
        return fail(SELAB200_ERR_BITSTREAM, "File is too small, probably not a sela file.");
    if (memcmp(b, "SeLa", 4) != 0)
        return fail(SELAB200_ERR_BITSTREAM, "Magic number is incorrect, probably not a sela file.");
    auto u16 = [&](size_t o) { return (uint32_t)b[o] | ((uint32_t)b[o + 1] << 8); };
    auto u32 = [&](size_t o) { return u16(o) | (u16(o + 2) << 16); };
    info->sample_rate = u32(4);
    info->bits_per_sample = (uint16_t)u16(8);
    info->channels = b[10];
    info->header_frames = u32(11);
    const uint32_t channels = info->channels;
    size_t at = 15;
    unsigned long long words = 0;
    uint32_t f = 0;
    for (; f < info->header_frames; f++) {
        if (at + 4 > n || u32(at) != 0xAA55FF00u)
            break;
        if (frame_bytes && f < frame_capacity)
            frame_bytes[f] = at;
        at += 4;
        for (uint32_t c = 0; c < channels; c++) {
            if (at + 7 > n)
                return fail(SELAB200_ERR_BITSTREAM, "sela file is truncated");
            const uint32_t refl_words = u16(at + 4);
            const size_t at2 = at + 7 + 4 * (size_t)refl_words;
            if (at2 + 5 > n)
                return fail(SELAB200_ERR_BITSTREAM, "sela file is truncated");
            const uint32_t res_words = u16(at2 + 1);
            if (at2 + 5 + 4 * (size_t)res_words > n)
                return fail(SELAB200_ERR_BITSTREAM, "sela file is truncated");
            if (descs) {
                selab200_subframe_desc d;
                d.channel = b[at];
                d.subframe_type = b[at + 1];
                d.parent_channel = b[at + 2];
                d.refl_rice_param = b[at + 3];
                d.refl_words = (uint16_t)refl_words;
                d.lpc_order = b[at + 6];
                d.res_rice_param = b[at2];
                d.res_words = (uint16_t)res_words;
                d.samples = (uint16_t)u16(at2 + 3);
                d.reserved = 0;
                d.refl_offset = words;
                d.res_offset = words + refl_words;
                descs->push_back(d);
            }
            words += refl_words + res_words;
            at = at2 + 5 + 4 * (size_t)res_words;
        }
    }
    info->n_frames = f;
    info->n_words = words;
    info->n_bytes_used = at;
    if (frame_bytes && f < frame_capacity)
        frame_bytes[f] = at;
    return 0;
}

} // namespace

extern "C" {

int selab200_container_info_get(const uint8_t *container, size_t n_bytes, selab200_container_info *info)
{
    if (!container || !info)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    return walk_container(container, n_bytes, info, nullptr);
}

int selab200_container_frame_offsets(const uint8_t *container, size_t n_bytes, uint64_t *offsets, size_t capacity,
                                     selab200_container_info *info)
{
    if (!container || !offsets || !info)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    if (int rc = walk_container(container, n_bytes, info, nullptr, offsets, capacity))
        return rc;
    if ((size_t)info->n_frames + 1 > capacity)
        return fail(SELAB200_ERR_CAPACITY, "offset table too small: %zu entries, need %u", capacity, info->n_frames + 1);
    return 0;
}

void selab200_container_close(selab200_container *h)
{
    if (!h)
        return;
    std::lock_guard<std::mutex> lock(g_mutex);
    Context &c = g_slots[0]; // container handles belong to the primary device
    if (c.ready)
        cudaSetDevice(c.device); // the caller may be on a thread that never selected the device
    if (c.s_h2d)
        cudaStreamSynchronize(c.s_h2d); // the upload reads the caller's bytes
    if (c.ready && c.spare.size() < kMaxSpareBuffers)
        c.spare.push_back(h->buf);
    else
        h->buf.destroy();
    delete h;
}

int selab200_container_open(const uint8_t *container, size_t n_bytes, selab200_container **handle,
                            selab200_container_info *info)
{
    if (!container || !handle || !info)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    *handle = nullptr;
    selab200_container_info probe;
    if (int rc = walk_container(container, n_bytes < 15 ? n_bytes : 15, &probe, nullptr)) // header checks only
        return rc;
    selab200_container *h = nullptr;
    int rc = 0;
    {
        std::lock_guard<std::mutex> lock(g_mutex);
        Context *c;
        if ((rc = require_ready(c)) != 0)
            return rc;
        h = new selab200_container;
        h->bytes = container;
        h->n_bytes = n_bytes;
        // recycled buffers: the smallest spare that is large enough, else any spare (it is regrown below)
        std::vector<ContainerBuffers> &spare = c->spare;
        if (!spare.empty()) {
            size_t pick = 0;
            for (size_t i = 0; i < spare.size(); i++)
                if (spare[i].image.bytes >= n_bytes + 64 &&
                    (spare[pick].image.bytes < n_bytes + 64 || spare[i].image.bytes < spare[pick].image.bytes))
                    pick = i;
            h->buf = spare[pick];
            spare.erase(spare.begin() + pick);
        }
        rc = h->buf.image.ensure(n_bytes + 64);
        // start the upload first: the DMA engine streams the bytes while this thread walks them
        cudaError_t e = cudaSuccess;
        h->piece_bytes = ((n_bytes + ContainerBuffers::kPieces - 1) / ContainerBuffers::kPieces + 255) & ~(size_t)255;
        for (int i = 0; rc == 0 && (size_t)i * h->piece_bytes < n_bytes; i++) {
            const size_t lo = (size_t)i * h->piece_bytes;
            const size_t len = lo + h->piece_bytes <= n_bytes ? h->piece_bytes : n_bytes - lo;
            if (!h->buf.ev_piece[i])
                e = cudaEventCreateWithFlags(&h->buf.ev_piece[i], cudaEventDisableTiming);
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(static_cast<uint8_t *>(h->buf.image.ptr) + lo, container + lo, len, cudaMemcpyHostToDevice, c->s_h2d);
            if (e == cudaSuccess)
                e = cudaEventRecord(h->buf.ev_piece[i], c->s_h2d);
            if (e != cudaSuccess)
                rc = fail(SELAB200_ERR_CUDA, "container upload failed: %s", cudaGetErrorString(e));
            h->n_pieces = i + 1;
        }
    }
    if (rc == 0) {
        // One walk, into a growing host vector (numFrames is not trusted for sizing), then a pinned copy
        // the chunked descriptor uploads can stream from.
        std::vector<selab200_subframe_desc> descs;
        descs.reserve(n_bytes / 2048 + 16);
        rc = walk_container(container, n_bytes, &h->info, &descs);
        if (rc == 0 && !descs.empty()) {
            const size_t bytes = descs.size() * sizeof(selab200_subframe_desc);
            rc = h->buf.descs.ensure(bytes);
            if (rc == 0)
                memcpy(h->buf.descs.ptr, descs.data(), bytes);
        }
    }
    if (rc != 0)
        return fail_after_cleanup(rc, [h] { selab200_container_close(h); });
    *info = h->info;
    *handle = h;
    return 0;
}

} // extern "C"

// Frames [F0, F0 + NF) of an open container on the device of context `c`.  The primary device holds the
// whole byte image (uploaded by selab200_container_open, in pieces with events); any other device uploads just
// the bytes of its block.  The word arena keeps the descriptors' file-order offsets: it is addressed through a
// pointer shifted back by the block's first word, so nothing is re-based.
static int container_decode_block(Context &c, selab200_container *h, uint32_t F0, uint32_t NF, int16_t *pcm_out)
{
    if (NF == 0)
        return 0;
    const bool primary = &c == &g_slots[0];
    const uint32_t channels = h->info.channels;
    const selab200_subframe_desc *hd = static_cast<const selab200_subframe_desc *>(h->buf.descs.ptr);
    PipelineDrain drain{c};
    const ChunkPlan plan = plan_chunks(NF);
    const unsigned long long w_lo = hd[(size_t)F0 * channels].refl_offset;
    const selab200_subframe_desc &tail = hd[(size_t)(F0 + NF) * channels - 1];
    const unsigned long long w_hi = tail.res_offset + tail.res_words;
    PipelineViews v;
    if (int rc = begin_pipeline(c, plan, channels, (size_t)(w_hi - w_lo) * 4 + 96,
                                selab200_decode_workspace_bytes(plan.max_frames, channels), kLanes, v))
        return rc;
    // 16 bytes of slack in front (the Rice decoder reads whole 16-byte vectors), the 16-byte phase of file order kept
    uint32_t *d_arena = reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(v.words) + 16 + ((w_lo * 4) & 15)) - w_lo;
    const uint8_t *d_bytes = static_cast<const uint8_t *>(h->buf.image.ptr);
    if (!primary) {
        // the unpack kernel reads aligned 32-bit words of the byte image
        const unsigned long long b0 = container_frame_byte(F0, channels, w_lo) & ~3ull;
        const size_t end = std::min<size_t>(h->n_bytes, (size_t)container_frame_byte(F0 + NF, channels, w_hi) + 4);
        if (int rc = c.aux.ensure(end - (size_t)b0 + 64)) return rc;
        CUDA_TRY(cudaMemcpyAsync(c.aux.ptr, h->bytes + b0, end - (size_t)b0, cudaMemcpyHostToDevice, c.s_h2d));
        CUDA_TRY(cudaEventRecord(c.ev_h2d[0], c.s_h2d));
        d_bytes = static_cast<const uint8_t *>(c.aux.ptr) - b0;
    }
    return decode_chunks(c, plan, channels, v, d_arena, (size_t)h->info.n_words, pcm_out + (size_t)F0 * channels * kFrame,
                         [&](uint32_t, uint32_t f0, uint32_t nf, cudaStream_t cs) {
        const selab200_subframe_desc *dc = hd + (size_t)(F0 + f0) * channels;
        const size_t chunk_sub = (size_t)nf * channels;
        // descriptors go up on the chunk's own lane: s_h2d is still busy with the container bytes
        CUDA_TRY(cudaMemcpyAsync(v.descs + (size_t)f0 * channels, dc, chunk_sub * sizeof(*dc), cudaMemcpyHostToDevice, cs));
        if (primary) {
            // the container bytes this chunk reads end with its last subframe (+3 bytes of slack)
            const selab200_subframe_desc &last = dc[chunk_sub - 1];
            const unsigned long long end_byte =
                container_frame_byte(F0 + f0 + nf, channels, last.res_offset + last.res_words) + 3;
            int piece = (int)(end_byte / h->piece_bytes);
            if (piece >= h->n_pieces)
                piece = h->n_pieces - 1;
            CUDA_TRY(cudaStreamWaitEvent(cs, h->buf.ev_piece[piece], 0));
        } else {
            CUDA_TRY(cudaStreamWaitEvent(cs, c.ev_h2d[0], 0));
        }
        k_container_unpack<<<(unsigned)((chunk_sub + 7) / 8), 256, 0, cs>>>(d_bytes, v.descs + (size_t)f0 * channels,
                                                                           (uint32_t)chunk_sub, channels,
                                                                           (unsigned long long)(F0 + f0) * channels, d_arena);
        return launch_check("k_container_unpack");
    });
}

extern "C" {

int selab200_container_decode(selab200_container *h, int16_t *pcm_out)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready(c))
        return rc;
    if (!h)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    const uint32_t n_frames = h->info.n_frames, channels = h->info.channels;
    if (n_frames == 0)
        return 0;
    if (!pcm_out)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    if (int rc = check_channels(channels))
        return rc;
    if (!use_all_devices(n_frames))
        return container_decode_block(*c, h, 0, n_frames, pcm_out);
    // one block of frames per device; the primary (which holds the whole image) takes the first
    std::vector<DevicePart> parts = device_parts(n_frames);
    return run_on_devices(parts, [&](Context &dc, DevicePart &p) { return container_decode_block(dc, h, p.f0, p.nf, pcm_out); });
}

int selab200_selftest(uint32_t *mismatches)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready(c))
        return rc;
    if (!mismatches)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    uint32_t *d = reinterpret_cast<uint32_t *>(static_cast<char *>(c->small.ptr) + 32);
    CUDA_TRY(cudaMemsetAsync(d, 0, 4, c->stream));
    k_selftest_scaling<<<(131071 + 255) / 256, 256, 0, c->stream>>>(d);
    if (int rc = launch_check("k_selftest_scaling"))
        return rc;
    CUDA_TRY(cudaMemcpyAsync(c->h_small + 8, d, 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    *mismatches = (uint32_t)c->h_small[8];
    return 0;
}

// ---------------------------------------------------------------- stages --

int selab200_lpc_residues(const int32_t *samples, uint32_t n_sub, uint8_t *order, int32_t *q, int32_t *residues)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready(c))
        return rc;
    if (!samples || !order || !q || !residues)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    if (n_sub == 0)
        return 0;
    for (size_t i = 0; i < (size_t)n_sub * kFrame; i++)
        if (samples[i] > 65535 || samples[i] < -65535)
            return fail(SELAB200_ERR_RANGE, "sample %zu = %d outside the 17-bit domain of 16-bit audio", i, samples[i]);
    const size_t sig = (size_t)n_sub * kFrame * 4;
    if (int rc = c->in.ensure(sig)) return rc;
    if (int rc = c->work.ensure(sig)) return rc;
    if (int rc = c->aux.ensure((size_t)n_sub * kMaxOrder * 4 + n_sub + 256)) return rc;
    int32_t *d_q = static_cast<int32_t *>(c->aux.ptr);
    uint8_t *d_order = reinterpret_cast<uint8_t *>(d_q + (size_t)n_sub * kMaxOrder);
    CUDA_TRY(cudaMemcpyAsync(c->in.ptr, samples, sig, cudaMemcpyHostToDevice, c->stream));
    k_lpc_residues<<<n_sub, 32, 0, c->stream>>>(static_cast<const int32_t *>(c->in.ptr), n_sub, d_order, d_q,
                                                static_cast<int32_t *>(c->work.ptr));
    if (int rc = launch_check("k_lpc_residues"))
        return rc;
    CUDA_TRY(cudaMemcpyAsync(residues, c->work.ptr, sig, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(q, d_q, (size_t)n_sub * kMaxOrder * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(order, d_order, n_sub, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int selab200_lpc_samples(const int32_t *residues, uint32_t n_sub, const uint8_t *order, const int32_t *q,
                         int32_t *samples)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready(c))
        return rc;
    if (!residues || !order || !q || !samples)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    if (n_sub == 0)
        return 0;
    for (uint32_t i = 0; i < n_sub; i++)
        if (order[i] > kMaxOrder)
            return fail(SELAB200_ERR_BITSTREAM, "order[%u] = %u exceeds %d", i, order[i], kMaxOrder);
    const size_t sig = (size_t)n_sub * kFrame * 4;
    if (int rc = c->in.ensure(sig)) return rc;
    if (int rc = c->work.ensure(sig)) return rc;
    if (int rc = c->aux.ensure((size_t)n_sub * kMaxOrder * 4 + n_sub + 256)) return rc;
    int32_t *d_q = static_cast<int32_t *>(c->aux.ptr);
    uint8_t *d_order = reinterpret_cast<uint8_t *>(d_q + (size_t)n_sub * kMaxOrder);
    CUDA_TRY(cudaMemcpyAsync(c->in.ptr, residues, sig, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(d_q, q, (size_t)n_sub * kMaxOrder * 4, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(d_order, order, n_sub, cudaMemcpyHostToDevice, c->stream));
    k_lpc_samples<<<n_sub, 32, 0, c->stream>>>(static_cast<const int32_t *>(c->in.ptr), n_sub, d_order, d_q,
                                               static_cast<int32_t *>(c->work.ptr));
    if (int rc = launch_check("k_lpc_samples"))
        return rc;
    CUDA_TRY(cudaMemcpyAsync(samples, c->work.ptr, sig, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

int selab200_rice_encode(const int32_t *values, const uint32_t *counts, uint32_t n_streams, uint32_t stride,
                         uint32_t *rice_param, uint32_t *n_words, uint32_t *words, uint32_t words_stride)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready(c))
        return rc;
    if (!values || !counts || !rice_param || !n_words || !words)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    if (stride > (uint32_t)kFrame)
        return fail(SELAB200_ERR_ARGUMENT, "stride %u exceeds %d values per stream", stride, kFrame);
    for (uint32_t i = 0; i < n_streams; i++)
        if (counts[i] > stride)
            return fail(SELAB200_ERR_ARGUMENT, "counts[%u] exceeds stride", i);
    if (n_streams == 0)
        return 0;
    const size_t vbytes = (size_t)n_streams * stride * 4, wbytes = (size_t)n_streams * words_stride * 4;
    if (int rc = c->in.ensure(vbytes + 16)) return rc;
    if (int rc = c->words.ensure(wbytes + 16)) return rc;
    if (int rc = c->aux.ensure((size_t)n_streams * 12 + 256)) return rc;
    uint32_t *d_counts = static_cast<uint32_t *>(c->aux.ptr);
    uint32_t *d_k = d_counts + n_streams, *d_nw = d_k + n_streams;
    int32_t *d_status = static_cast<int32_t *>(c->small.ptr);
    CUDA_TRY(cudaMemsetAsync(d_status, 0, 4, c->stream));
    CUDA_TRY(cudaMemcpyAsync(c->in.ptr, values, vbytes, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(d_counts, counts, (size_t)n_streams * 4, cudaMemcpyHostToDevice, c->stream));
    k_rice_encode<<<n_streams, 32, 0, c->stream>>>(static_cast<const int32_t *>(c->in.ptr), d_counts, stride, d_k,
                                                   d_nw, static_cast<uint32_t *>(c->words.ptr), words_stride, d_status);
    if (int rc = launch_check("k_rice_encode"))
        return rc;
    CUDA_TRY(cudaMemcpyAsync(rice_param, d_k, (size_t)n_streams * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(n_words, d_nw, (size_t)n_streams * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(words, c->words.ptr, wbytes, cudaMemcpyDeviceToHost, c->stream));
    return read_status(*c, c->stream, d_status);
}

int selab200_rice_decode(const uint32_t *words, const uint32_t *n_words, uint32_t words_stride,
                         const uint32_t *rice_param, const uint32_t *counts, uint32_t n_streams, int32_t *out,
                         uint32_t out_stride)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    Context *c;
    if (int rc = require_ready(c))
        return rc;
    if (!words || !n_words || !rice_param || !counts || !out)
        return fail(SELAB200_ERR_ARGUMENT, "null pointer");
    if (n_streams == 0)
        return 0;
    const size_t wbytes = (size_t)n_streams * words_stride * 4, obytes = (size_t)n_streams * out_stride * 4;
    if (int rc = c->words.ensure(wbytes + 16)) return rc;
    if (int rc = c->work.ensure(obytes + 16)) return rc;
    if (int rc = c->aux.ensure((size_t)n_streams * 12 + 256)) return rc;
    uint32_t *d_nw = static_cast<uint32_t *>(c->aux.ptr);
    uint32_t *d_k = d_nw + n_streams, *d_counts = d_k + n_streams;
    int32_t *d_status = static_cast<int32_t *>(c->small.ptr);
    CUDA_TRY(cudaMemsetAsync(d_status, 0, 4, c->stream));
    CUDA_TRY(cudaMemsetAsync(c->work.ptr, 0, obytes, c->stream));
    CUDA_TRY(cudaMemcpyAsync(c->words.ptr, words, wbytes, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(d_nw, n_words, (size_t)n_streams * 4, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(d_k, rice_param, (size_t)n_streams * 4, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(d_counts, counts, (size_t)n_streams * 4, cudaMemcpyHostToDevice, c->stream));
    k_rice_decode_streams<<<(n_streams + 32 * kRiceWarps - 1) / (32 * kRiceWarps), 32 * kRiceWarps, 0, c->stream>>>(
        static_cast<const uint32_t *>(c->words.ptr), d_nw, words_stride, d_k, d_counts, n_streams,
        static_cast<int32_t *>(c->work.ptr), out_stride, d_status);
    if (int rc = launch_check("k_rice_decode_streams"))
        return rc;
    CUDA_TRY(cudaMemcpyAsync(out, c->work.ptr, obytes, cudaMemcpyDeviceToHost, c->stream));
    return read_status(*c, c->stream, d_status);
}

} // extern "C"
